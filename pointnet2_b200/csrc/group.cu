// group.cu — gather_point, group_point, their gradients, the fused sample_and_group tail and
// selection_sort, for sm_100a.
//
// Replaces (reference, tf_ops/):
//   gatherpointKernel / scatteraddpointKernel   sampling/tf_sampling_g.cu:172-192
//   group_point_gpu / group_point_grad_gpu      grouping/tf_grouping_g.cu:40-78
//   selection_sort_gpu                          grouping/tf_grouping_g.cu:83-123
// and fuses the glue of utils/pointnet_util.py:45-54 / :179-186 (pn2_group_concat).
//
// These are the HBM-bound kernels of the path.  The reference gives one thread a whole
// (nsample x c) row block, so neighbouring lanes write nsample*c*4 bytes apart.  Here the output
// is treated as one flat array: consecutive lanes write consecutive 16-byte vectors (streaming
// stores, the output is write-once), and read the matching 16 bytes of the source row (rows are
// served from L2: the source tensor is at most tens of MB).
#include <stdlib.h>

#include "pn2_common.cuh"

namespace pn2 {

constexpr int kCopyThreads = 256;

static bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

// ---- gather_point: out[b,j,:] = inp[b,idx[b,j],:] (3 floats) -----------------------------------
__global__ void __launch_bounds__(kCopyThreads)
gather_point_kernel(int n, int m, long long total, const float* __restrict__ inp, const int* __restrict__ idx,
                    float* __restrict__ out) {
    for (long long r = (long long)blockIdx.x * kCopyThreads + threadIdx.x; r < total;
         r += (long long)gridDim.x * kCopyThreads) {
        const long long cloud = r / m;
        const float* s = inp + (cloud * n + idx[r]) * 3;
        float* d = out + r * 3;
        d[0] = s[0];
        d[1] = s[1];
        d[2] = s[2];
    }
}

__global__ void __launch_bounds__(kCopyThreads)
gather_point_grad_kernel(int n, int m, long long total, const float* __restrict__ out_g,
                         const int* __restrict__ idx, float* __restrict__ inp_g) {
    for (long long r = (long long)blockIdx.x * kCopyThreads + threadIdx.x; r < total;
         r += (long long)gridDim.x * kCopyThreads) {
        const long long cloud = r / m;
        float* d = inp_g + (cloud * n + idx[r]) * 3;
        const float* s = out_g + r * 3;
        atomicAdd(d + 0, s[0]);
        atomicAdd(d + 1, s[1]);
        atomicAdd(d + 2, s[2]);
    }
}

// ---- group_point, vector path: c % 4 == 0, 16-byte aligned bases -------------------------------
// One thread per output float4.  rows = b*m*nsample flat rows, rows_per_cloud = m*nsample.
template <typename IndexT, int U>
__global__ void __launch_bounds__(kCopyThreads)
group_point_vec4_kernel(int n, int c4, IndexT rows_per_cloud, IndexT total_vec, const float4* __restrict__ points,
                        const int* __restrict__ idx, float4* __restrict__ out) {
    // U independent 16-byte gathers in flight per thread (all loads first, then the streaming stores)
    const IndexT stride = (IndexT)gridDim.x * kCopyThreads;
    for (IndexT v0 = (IndexT)blockIdx.x * kCopyThreads + threadIdx.x; v0 < total_vec; v0 += stride * U) {
        float4 val[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const IndexT v = v0 + (IndexT)u * stride;
            if (v < total_vec) {
                const IndexT row = v / (IndexT)c4;
                const int l = (int)(v - row * (IndexT)c4);
                const IndexT cloud = row / rows_per_cloud;
                const int a = __ldg(idx + row);
                val[u] = __ldg(points + ((size_t)cloud * n + a) * c4 + l);
            }
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const IndexT v = v0 + (IndexT)u * stride;
            if (v < total_vec) st_stream_f4(out + v, val[u]);
        }
    }
}

// ---- group_point, vector path, row-batched: LPR lanes per row, R rows in flight per lane-group ----
// No per-vector integer division and no load->load dependency per vector: the R row indices of a
// batch are fetched first (one broadcast load each), then every lane issues R independent 16-byte
// gathers per channel step and streams them out.  cfg3 layer 2 (C=320): see profiles/.
template <int LPR, int R>
__global__ void __launch_bounds__(kCopyThreads)
group_rows_vec4_kernel(int n, int c4, unsigned rows_per_cloud, const float4* __restrict__ points,
                       const int* __restrict__ idx, float4* __restrict__ out) {
    constexpr int RPW = 32 / LPR;  // row slots per warp
    const int lane = threadIdx.x & 31, g = lane % LPR, sub = lane / LPR;
    const unsigned cloud = blockIdx.y;
    const unsigned warps = (gridDim.x * kCopyThreads) >> 5;
    const unsigned warp = (blockIdx.x * kCopyThreads + threadIdx.x) >> 5;
    const size_t cloud_row0 = (size_t)cloud * rows_per_cloud;
    const int* __restrict__ cidx = idx + cloud_row0;
    const float4* __restrict__ cpts = points + (size_t)cloud * n * c4;
    // this lane-group walks rows r = (warp*RPW + sub)*R + rr, stride warps*RPW*R
    for (unsigned r0 = (warp * RPW + sub) * R; r0 < rows_per_cloud; r0 += warps * RPW * R) {
        const float4* __restrict__ src[R];
        float4* __restrict__ dst[R];
        bool ok[R];
#pragma unroll
        for (int rr = 0; rr < R; ++rr) {
            const unsigned r = r0 + rr;
            ok[rr] = r < rows_per_cloud;
            const int a = ok[rr] ? __ldg(cidx + r) : 0;
            src[rr] = cpts + (size_t)a * c4;
            dst[rr] = out + (cloud_row0 + r) * c4;
        }
        for (int l = g; l < c4; l += LPR) {
            float4 v[R];
#pragma unroll
            for (int rr = 0; rr < R; ++rr)
                if (ok[rr]) v[rr] = __ldg(src[rr] + l);
#pragma unroll
            for (int rr = 0; rr < R; ++rr)
                if (ok[rr]) st_stream_f4(dst[rr] + l, v[rr]);
        }
    }
}

// ---- group_point general path and the fused sample_and_group tail: LPR lanes per output row ----
// Row r of cloud `blockIdx.y` is the (3+c)- or c-wide output row of one (centroid, sample) pair:
//   HAS_XYZ: out[r, xyz_lo..xyz_lo+3) = xyz[a] - new_xyz[r / nsample]   (also to grouped_xyz if given)
//            out[r, feat_lo..feat_lo+c) = points[a]                      a = idx[r]
//   else   : out[r, 0..c) = points[a]
// LPR consecutive lanes own one row and walk its channels with stride LPR, so a warp's loads and
// stores are runs of consecutive 4-byte words (full sectors) whatever the row width; the per-row
// index/centroid loads are broadcasts.  No per-element division or branching.
template <int LPR, bool HAS_XYZ>
__global__ void __launch_bounds__(kCopyThreads)
group_rows_kernel(int n, int c, int nsample, unsigned rows_per_cloud, const float* __restrict__ xyz,
                  const float* __restrict__ new_xyz, const float* __restrict__ points,
                  const int* __restrict__ idx, int xyz_lo, int feat_lo, float* __restrict__ out,
                  float* __restrict__ grouped_xyz) {
    constexpr int RPW = 32 / LPR;  // rows per warp per pass
    const int lane = threadIdx.x & 31, g = lane % LPR, sub = lane / LPR;
    const unsigned cloud = blockIdx.y;
    const int w = c + (HAS_XYZ ? 3 : 0);
    const unsigned warps = (gridDim.x * kCopyThreads) >> 5;
    const unsigned warp = (blockIdx.x * kCopyThreads + threadIdx.x) >> 5;
    const size_t cloud_row0 = (size_t)cloud * rows_per_cloud;
    const int* __restrict__ cidx = idx + cloud_row0;
    const float* __restrict__ cpts = points ? points + (size_t)cloud * n * c : nullptr;
    const float* __restrict__ cxyz = HAS_XYZ ? xyz + (size_t)cloud * n * 3 : nullptr;
    // R rows per lane group and trip, U words per row and lane in flight: what limits these copies is bytes in
    // flight per SM (measured: 32 KB/SM -> 3.5 TB/s, 64 KB/SM -> 5.5 TB/s for the same gather), so all R*U loads of a
    // trip are issued before the first store
    constexpr int R = 2, U = 4;  // measured at C = 320 + 3: R = 2: 58 / 94 / 172 us (38 registers); R = 4: 66 / 103 / 180 us (58 registers)
    for (unsigned r0 = (warp * RPW + sub) * R; r0 < rows_per_cloud; r0 += warps * RPW * R) {
        const float* __restrict__ src[R];
        float* __restrict__ d[R];
        bool ok[R];
#pragma unroll
        for (int rr = 0; rr < R; ++rr) {
            const unsigned r = r0 + rr;
            ok[rr] = r < rows_per_cloud;
            const int a = ok[rr] ? __ldg(cidx + r) : 0;
            float* __restrict__ dst = out + (cloud_row0 + r) * w;
            src[rr] = cpts ? cpts + (size_t)a * c : nullptr;
            d[rr] = dst + feat_lo;
            if (HAS_XYZ && ok[rr] && g < 3) {
                const size_t ctr = (size_t)cloud * (rows_per_cloud / (unsigned)nsample) + r / (unsigned)nsample;  // global centroid index
                const float v = __fsub_rn(__ldg(cxyz + (size_t)a * 3 + g), __ldg(new_xyz + ctr * 3 + g));
                __stcs(dst + xyz_lo + g, v);
                if (grouped_xyz) __stcs(grouped_xyz + (cloud_row0 + r) * 3 + g, v);
            }
        }
        for (int l0 = g; l0 < c; l0 += LPR * U) {
            float v[R][U];
#pragma unroll
            for (int rr = 0; rr < R; ++rr)
#pragma unroll
                for (int u = 0; u < U; ++u)
                    if (ok[rr] && l0 + u * LPR < c) v[rr][u] = __ldg(src[rr] + l0 + u * LPR);
#pragma unroll
            for (int rr = 0; rr < R; ++rr)
#pragma unroll
                for (int u = 0; u < U; ++u)
                    if (ok[rr] && l0 + u * LPR < c) __stcs(d[rr] + l0 + u * LPR, v[rr][u]);
        }
    }
}

// ---- the fused sample_and_group tail with features, c % 4 == 0: 16-byte gathers AND 16-byte stores ----
// Output rows are w = 3 + c floats wide (67, 131, 259, 323 in the reference's networks), so a row's feature
// segment starts 0..3 floats past a 16-byte boundary — differently for every row.  The source rows ARE
// aligned (c % 4 == 0): lane k of the row's lane group loads source vector k (LDG.128); the output vector
// that starts `head` floats into the segment is the last 4-head floats of source vector k followed by the
// first head floats of vector k+1, which the lane gets from its neighbour by shuffle (the last lane of a
// pass loads it).  So the body of every row goes out as aligned STG.128 with the data re-aligned in
// registers; only the <= 3 head floats, <= 3 tail floats and the 3 xyz floats of a row are scalar stores.
// Round 1's kernel moved every float with a 4-byte load and a 4-byte store: 4x the LSU instructions, 42-54 %
// of the HBM peak at C = 320 where the aligned C % 4 == 0 gather (same bytes) reaches 84 %.
// R rows are in flight per lane group (all their gathers are issued before the first store).
template <int LPR, int R>
__global__ void __launch_bounds__(kCopyThreads, 4)  // <= 64 registers: at 114 (R = 4, unbounded) occupancy fell to 25 % and the kernel with it
group_concat_vec_kernel(int n, int c4, int nsample, unsigned rows_per_cloud, const float* __restrict__ xyz,
                        const float* __restrict__ new_xyz, const float4* __restrict__ points, const int* __restrict__ idx,
                        int xyz_lo, int feat_lo, float* __restrict__ out, float* __restrict__ grouped_xyz) {
    constexpr int RPW = 32 / LPR;
    const int lane = threadIdx.x & 31, g = lane % LPR, sub = lane / LPR;
    const unsigned cloud = blockIdx.y;
    const unsigned warps = (gridDim.x * kCopyThreads) >> 5;
    const unsigned warp = (blockIdx.x * kCopyThreads + threadIdx.x) >> 5;
    const size_t cloud_row0 = (size_t)cloud * rows_per_cloud;
    const unsigned m = rows_per_cloud / (unsigned)nsample;
    const int c = 4 * c4;
    const size_t w = (size_t)c + 3;
    const int* __restrict__ cidx = idx + cloud_row0;
    const float4* __restrict__ cpts = points + (size_t)cloud * n * c4;
    const float* __restrict__ cxyz = xyz + (size_t)cloud * n * 3;
    const float* __restrict__ cctr = new_xyz + (size_t)cloud * m * 3;
    for (unsigned r0 = (warp * RPW + sub) * R; r0 < rows_per_cloud; r0 += warps * RPW * R) {
        const float4* __restrict__ src[R];
        float* __restrict__ fdst[R];  // start of the row's feature segment
        int head[R];
        bool ok[R];
#pragma unroll
        for (int rr = 0; rr < R; ++rr) {
            const unsigned r = r0 + rr;
            ok[rr] = r < rows_per_cloud;
            const int a = ok[rr] ? __ldg(cidx + r) : 0;
            src[rr] = cpts + (size_t)a * c4;
            const size_t obase = (cloud_row0 + r) * w;
            fdst[rr] = out + obase + feat_lo;
            head[rr] = (int)((4u - (unsigned)((obase + (size_t)feat_lo) & 3u)) & 3u);
            // The row's scalar words — 3 centred xyz, `head` floats in front of the first aligned vector and 4-head
            // behind the last one — go out as ONE predicated store instruction: lane t < 3 takes xyz[t], the next
            // `head` lanes the head floats, the next 4-head lanes the tail floats (7 lanes at most).  (One store
            // instruction per word, as a first version did, is 9 store instructions per row against the 2.5 that
            // move the row's 80 vectors: the LSU queue, not the bytes, set the pace.)
            if (ok[rr] && g < 7) {
                const int h = head[rr];
                float* dst = nullptr;
                float val = 0.f;
                if (g < 3) {
                    val = __fsub_rn(__ldg(cxyz + (size_t)a * 3 + g), __ldg(cctr + (size_t)(r / (unsigned)nsample) * 3 + g));
                    dst = out + obase + xyz_lo + g;
                    if (grouped_xyz) __stcs(grouped_xyz + (cloud_row0 + r) * 3 + g, val);
                } else if (h != 0) {
                    const int t = g - 3;                  // 0..3
                    const int e = t < h ? t : c - 4 + t;  // head float t, or the tail float (c - 4) + t for t >= h
                    val = __ldg(reinterpret_cast<const float*>(src[rr]) + e);
                    dst = fdst[rr] + e;
                }
                if (dst) __stcs(dst, val);
            }
        }
        for (int k0 = 0; k0 < c4; k0 += LPR) {
            const int k = k0 + g;
            float4 v[R];
            float3 nx[R];
#pragma unroll
            for (int rr = 0; rr < R; ++rr) {
                v[rr] = make_float4(0.f, 0.f, 0.f, 0.f);
                if (ok[rr] && k < c4) v[rr] = __ldg(src[rr] + k);
            }
#pragma unroll
            for (int rr = 0; rr < R; ++rr) {
                nx[rr].x = __shfl_down_sync(kFullMask, v[rr].x, 1, LPR);
                nx[rr].y = __shfl_down_sync(kFullMask, v[rr].y, 1, LPR);
                nx[rr].z = __shfl_down_sync(kFullMask, v[rr].z, 1, LPR);
                if (g == LPR - 1 && ok[rr] && k + 1 < c4 && head[rr] != 0) {  // next pass's first vector
                    const float4 t = __ldg(src[rr] + k + 1);
                    nx[rr] = make_float3(t.x, t.y, t.z);
                }
            }
#pragma unroll
            for (int rr = 0; rr < R; ++rr) {
                if (!ok[rr] || k >= c4) continue;
                const int h = head[rr];
                float* __restrict__ d = fdst[rr];
                if (h == 0) {
                    st_stream_f4(reinterpret_cast<float4*>(d) + k, v[rr]);
                    continue;
                }
                if (k + 1 < c4) {  // aligned body vector: floats [h + 4k, h + 4k + 4) of the segment
                    float4 o;
                    o.x = h == 1 ? v[rr].y : (h == 2 ? v[rr].z : v[rr].w);
                    o.y = h == 1 ? v[rr].z : (h == 2 ? v[rr].w : nx[rr].x);
                    o.z = h == 1 ? v[rr].w : (h == 2 ? nx[rr].x : nx[rr].y);
                    o.w = h == 1 ? nx[rr].x : (h == 2 ? nx[rr].y : nx[rr].z);
                    st_stream_f4(reinterpret_cast<float4*>(d + h + 4 * k), o);
                }  // (the head floats [0, h) and the tail floats behind the last aligned vector were written above)
            }
        }
    }
}

// Narrow rows (w <= 4 floats, e.g. group_point(xyz) and the C=0 sample_and_group tail): one thread
// per output row — the per-row index/centroid work is the cost, not the copy.
template <bool HAS_XYZ>
__global__ void __launch_bounds__(kCopyThreads)
group_narrow_kernel(int n, int c, int nsample, unsigned rows_per_cloud, const float* __restrict__ xyz,
                    const float* __restrict__ new_xyz, const float* __restrict__ points,
                    const int* __restrict__ idx, float* __restrict__ out, float* __restrict__ grouped_xyz) {
    const unsigned cloud = blockIdx.y;
    const size_t cloud_row0 = (size_t)cloud * rows_per_cloud;
    const int* __restrict__ cidx = idx + cloud_row0;
    const unsigned m = rows_per_cloud / (unsigned)nsample;
    for (unsigned r = blockIdx.x * kCopyThreads + threadIdx.x; r < rows_per_cloud; r += gridDim.x * kCopyThreads) {
        const int a = __ldg(cidx + r);
        if (HAS_XYZ) {  // c == 0: the row is the centred xyz
            const float* __restrict__ s = xyz + ((size_t)cloud * n + a) * 3;
            const float* __restrict__ ctr = new_xyz + ((size_t)cloud * m + r / (unsigned)nsample) * 3;
            const float v0 = __fsub_rn(__ldg(s), __ldg(ctr)), v1 = __fsub_rn(__ldg(s + 1), __ldg(ctr + 1)),
                        v2 = __fsub_rn(__ldg(s + 2), __ldg(ctr + 2));
            float* __restrict__ d = out + (cloud_row0 + r) * 3;
            __stcs(d, v0); __stcs(d + 1, v1); __stcs(d + 2, v2);
            if (grouped_xyz) {
                float* __restrict__ gq = grouped_xyz + (cloud_row0 + r) * 3;
                __stcs(gq, v0); __stcs(gq + 1, v1); __stcs(gq + 2, v2);
            }
        } else {
            const float* __restrict__ s = points + ((size_t)cloud * n + a) * c;
            float* __restrict__ d = out + (cloud_row0 + r) * c;
            for (int l = 0; l < c; ++l) __stcs(d + l, __ldg(s + l));
        }
    }
}

template <bool HAS_XYZ>
static int launch_group_rows(int b, int n, int c, int m, int nsample, const float* xyz, const float* new_xyz,
                             const float* points, const int* idx, int xyz_lo, int feat_lo, float* out,
                             float* grouped_xyz, cudaStream_t st) {
    const unsigned rpc = (unsigned)m * (unsigned)nsample;
    const int w = c + (HAS_XYZ ? 3 : 0);
    if (w <= 4 && (!HAS_XYZ || c == 0)) {
        unsigned gx = (rpc + kCopyThreads - 1) / kCopyThreads;
        const unsigned cap = (148u * 16u + b - 1) / b;
        if (gx > cap) gx = cap;
        group_narrow_kernel<HAS_XYZ><<<dim3(gx, b, 1), kCopyThreads, 0, st>>>(n, c, nsample, rpc, xyz, new_xyz, points, idx, out,
                                                                                grouped_xyz);
        return finish_launch();
    }
    if (HAS_XYZ && c >= 8 && c <= 64 && c % 4 == 0 && aligned16(points) && aligned16(out)) {
        // vectorised tail (see group_concat_vec_kernel).  Measured: it wins at C = 64 (30.7 against 35.6 us, cfg4 SA256) and
        // loses to the row kernel below from C = 128 up (C = 320 + 3, S = 64: 125 against 94 us), so only narrow rows take it
        const int c4 = c / 4;
        const int lpr = c4 <= 8 ? 8 : (c4 <= 16 ? 16 : 32);
        constexpr int R = 2;
        const unsigned rows_per_block = (kCopyThreads / 32) * (32 / lpr) * R;
        unsigned gx = (rpc + rows_per_block - 1) / rows_per_block;
        const unsigned cap = (148u * 32u + b - 1) / b;
        if (gx > cap) gx = cap;
        if (gx < 1) gx = 1;
        dim3 grid(gx, b, 1);
        const float4* p4 = reinterpret_cast<const float4*>(points);
        if (lpr == 8) group_concat_vec_kernel<8, R><<<grid, kCopyThreads, 0, st>>>(n, c4, nsample, rpc, xyz, new_xyz, p4, idx, xyz_lo, feat_lo, out, grouped_xyz);
        else if (lpr == 16) group_concat_vec_kernel<16, R><<<grid, kCopyThreads, 0, st>>>(n, c4, nsample, rpc, xyz, new_xyz, p4, idx, xyz_lo, feat_lo, out, grouped_xyz);
        else group_concat_vec_kernel<32, R><<<grid, kCopyThreads, 0, st>>>(n, c4, nsample, rpc, xyz, new_xyz, p4, idx, xyz_lo, feat_lo, out, grouped_xyz);
        return finish_launch();
    }
    const int lpr = w <= 4 ? 4 : (w <= 8 ? 8 : (w <= 16 ? 16 : 32));
    const unsigned rows_per_block = (kCopyThreads / 32) * (32 / lpr) * 2;  // R = 2 rows per lane group and trip
    unsigned gx = (rpc + rows_per_block - 1) / rows_per_block;
    const unsigned cap = (148u * 32u + b - 1) / b;  // enough CTAs to fill the machine, then grid-stride
    if (gx > cap) gx = cap;
    if (gx < 1) gx = 1;
    dim3 grid(gx, b, 1);
#define PN2_GROUP_ROWS(L) \
    group_rows_kernel<L, HAS_XYZ><<<grid, kCopyThreads, 0, st>>>(n, c, nsample, rpc, xyz, new_xyz, points, idx, xyz_lo, feat_lo, out, grouped_xyz)
    if (lpr == 4) PN2_GROUP_ROWS(4);
    else if (lpr == 8) PN2_GROUP_ROWS(8);
    else if (lpr == 16) PN2_GROUP_ROWS(16);
    else PN2_GROUP_ROWS(32);
#undef PN2_GROUP_ROWS
    return finish_launch();
}

// ---- group_point_grad: atomic scatter-add (vector red.global.add.v4.f32 when c % 4 == 0) -------
template <typename IndexT>
__global__ void __launch_bounds__(kCopyThreads)
group_point_grad_vec4_kernel(int n, int c4, IndexT rows_per_cloud, IndexT total_vec,
                             const float4* __restrict__ grad_out, const int* __restrict__ idx,
                             float4* __restrict__ grad_points) {
    const IndexT stride = (IndexT)gridDim.x * kCopyThreads;
    for (IndexT v = (IndexT)blockIdx.x * kCopyThreads + threadIdx.x; v < total_vec; v += stride) {
        const IndexT row = v / (IndexT)c4;
        const int l = (int)(v - row * (IndexT)c4);
        const IndexT cloud = row / rows_per_cloud;
        const int a = __ldg(idx + row);
        const float4 g = __ldcs(grad_out + v);
        atomicAdd(grad_points + ((size_t)cloud * n + a) * c4 + l, g);  // red.global.add.v4.f32 (sm_90+)
    }
}

template <typename IndexT>
__global__ void __launch_bounds__(kCopyThreads)
group_point_grad_scalar_kernel(int n, int c, IndexT rows_per_cloud, IndexT total,
                               const float* __restrict__ grad_out, const int* __restrict__ idx,
                               float* __restrict__ grad_points) {
    const IndexT stride = (IndexT)gridDim.x * kCopyThreads;
    for (IndexT e = (IndexT)blockIdx.x * kCopyThreads + threadIdx.x; e < total; e += stride) {
        const IndexT row = e / (IndexT)c;
        const int l = (int)(e - row * (IndexT)c);
        const IndexT cloud = row / rows_per_cloud;
        const int a = __ldg(idx + row);
        atomicAdd(grad_points + ((size_t)cloud * n + a) * c + l, __ldcs(grad_out + e));
    }
}

// ---- selection_sort: one warp per (b,m) row ------------------------------------------------------
// k rounds of "find the first minimum of v[s..n) (strict '<'), swap it into position s", indices
// carried along — the same permutation the reference's thread-per-row loop produces, with the
// argmin parallelised across the warp on the key (value, position).
__global__ void __launch_bounds__(kCopyThreads)
selection_sort_kernel(int n, int k, long long rows, const float* __restrict__ dist, int* __restrict__ outi,
                      float* __restrict__ out) {
    const int lane = threadIdx.x & 31;
    const long long warp = ((long long)blockIdx.x * kCopyThreads + threadIdx.x) >> 5;
    if (warp >= rows) return;
    const float* src = dist + warp * n;
    float* v = out + warp * n;
    int* ix = outi + warp * n;
    for (int s = lane; s < n; s += 32) {
        v[s] = src[s];
        ix[s] = s;
    }
    __syncwarp();
    const int rounds = k < n ? k : n;
    for (int s = 0; s < rounds; ++s) {
        float bv = 0.f;
        int bt = -1;
        for (int t = s + lane; t < n; t += 32) {
            const float x = v[t];
            if (bt < 0 || x < bv) {  // ascending t within a lane: strict '<' keeps the earliest
                bv = x;
                bt = t;
            }
        }
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) {
            const float ov = __shfl_xor_sync(kFullMask, bv, off);
            const int ot = __shfl_xor_sync(kFullMask, bt, off);
            // NaN-free total order on (value, position); lanes without candidates carry bt = -1
            const bool take = (ot >= 0) && (bt < 0 || ov < bv || (ov == bv && ot < bt));
            if (take) {
                bv = ov;
                bt = ot;
            }
        }
        if (lane == 0 && bt != s && bt >= 0) {
            const float tv = v[bt];
            v[bt] = v[s];
            v[s] = tv;
            const int ti = ix[bt];
            ix[bt] = ix[s];
            ix[s] = ti;
        }
        __syncwarp();
    }
}

static unsigned grid_for(unsigned long long work_items, unsigned per_block) {
    unsigned long long blocks = (work_items + per_block - 1) / per_block;
    const unsigned long long cap = 148ull * 64;  // grid-stride beyond this
    if (blocks > cap) blocks = cap;
    if (blocks < 1) blocks = 1;
    return (unsigned)blocks;
}


// ---- 16-bit features (pn2_*_h) -------------------------------------------------------------------
// A gather copies bits, so pn2_group_point_h hands every layout the float32 kernels already move — c even with
// 4-byte aligned bases: rows of c/2 words, float4 rows when c % 8 == 0 — to pn2_group_point.  What is left here:
// odd c / 2-byte aligned rows, and the concat tail, whose centred xyz is computed in float32 and rounded once.
// group_rows_h_kernel is group_rows_kernel with 2-byte elements (U = 8: the same bytes in flight per lane).
template <int LPR, bool HAS_XYZ, int DT>
__global__ void __launch_bounds__(kCopyThreads)
group_rows_h_kernel(int n, int c, int nsample, unsigned rows_per_cloud, const float* __restrict__ xyz,
                    const float* __restrict__ new_xyz, const unsigned short* __restrict__ points,
                    const int* __restrict__ idx, int xyz_lo, int feat_lo, unsigned short* __restrict__ out,
                    float* __restrict__ grouped_xyz) {
    constexpr int RPW = 32 / LPR;
    const int lane = threadIdx.x & 31, g = lane % LPR, sub = lane / LPR;
    const unsigned cloud = blockIdx.y;
    const int w = c + (HAS_XYZ ? 3 : 0);
    const unsigned warps = (gridDim.x * kCopyThreads) >> 5;
    const unsigned warp = (blockIdx.x * kCopyThreads + threadIdx.x) >> 5;
    const size_t cloud_row0 = (size_t)cloud * rows_per_cloud;
    const int* __restrict__ cidx = idx + cloud_row0;
    const unsigned short* __restrict__ cpts = points ? points + (size_t)cloud * n * c : nullptr;
    const float* __restrict__ cxyz = HAS_XYZ ? xyz + (size_t)cloud * n * 3 : nullptr;
    constexpr int R = 2, U = 8;
    for (unsigned r0 = (warp * RPW + sub) * R; r0 < rows_per_cloud; r0 += warps * RPW * R) {
        const unsigned short* __restrict__ src[R];
        unsigned short* __restrict__ d[R];
        bool ok[R];
#pragma unroll
        for (int rr = 0; rr < R; ++rr) {
            const unsigned r = r0 + rr;
            ok[rr] = r < rows_per_cloud;
            const int a = ok[rr] ? __ldg(cidx + r) : 0;
            unsigned short* __restrict__ dst = out + (cloud_row0 + r) * w;
            src[rr] = cpts ? cpts + (size_t)a * c : nullptr;
            d[rr] = dst + feat_lo;
            if (HAS_XYZ && ok[rr] && g < 3) {
                const size_t ctr = (size_t)cloud * (rows_per_cloud / (unsigned)nsample) + r / (unsigned)nsample;
                const float v = __fsub_rn(__ldg(cxyz + (size_t)a * 3 + g), __ldg(new_xyz + ctr * 3 + g));
                __stcs(dst + xyz_lo + g, f_to_h<DT>(v));
                if (grouped_xyz) __stcs(grouped_xyz + (cloud_row0 + r) * 3 + g, v);
            }
        }
        for (int l0 = g; l0 < c; l0 += LPR * U) {
            unsigned short v[R][U];
#pragma unroll
            for (int rr = 0; rr < R; ++rr)
#pragma unroll
                for (int u = 0; u < U; ++u)
                    if (ok[rr] && l0 + u * LPR < c) v[rr][u] = __ldg(src[rr] + l0 + u * LPR);
#pragma unroll
            for (int rr = 0; rr < R; ++rr)
#pragma unroll
                for (int u = 0; u < U; ++u)
                    if (ok[rr] && l0 + u * LPR < c) __stcs(d[rr] + l0 + u * LPR, v[rr][u]);
        }
    }
}

// The concat tail with 16-bit features, c % 8 == 0: 16-byte gathers of 8 values AND 16-byte stores.  Output rows are
// 3 + c values wide, so a row's feature segment starts `head` = 0..7 values before a 16-byte boundary, differently
// for every row.  As in group_concat_vec_kernel, lane k loads source vector k, gets vector k+1 from its neighbour
// (the last lane of a pass loads it), and stores the aligned output vector that starts `head` values into the
// segment: words q = head/2 .. q+4 of the pair, funnel-shifted by 16 bits when head is odd.  The head values, the
// 8 - head tail values and the 3 centred xyz of a row are scalar stores.  R rows' gathers are in flight before the
// first store.
template <int LPR, int R, int DT>
__global__ void __launch_bounds__(kCopyThreads, 4)
group_concat_h_vec_kernel(int n, int c8, int nsample, unsigned rows_per_cloud, const float* __restrict__ xyz,
                          const float* __restrict__ new_xyz, const uint4* __restrict__ points, const int* __restrict__ idx,
                          int xyz_lo, int feat_lo, unsigned short* __restrict__ out, float* __restrict__ grouped_xyz) {
    constexpr int RPW = 32 / LPR;
    const int lane = threadIdx.x & 31, g = lane % LPR, sub = lane / LPR;
    const unsigned cloud = blockIdx.y;
    const unsigned warps = (gridDim.x * kCopyThreads) >> 5;
    const unsigned warp = (blockIdx.x * kCopyThreads + threadIdx.x) >> 5;
    const size_t cloud_row0 = (size_t)cloud * rows_per_cloud;
    const unsigned m = rows_per_cloud / (unsigned)nsample;
    const int c = 8 * c8;
    const size_t w = (size_t)c + 3;
    const int* __restrict__ cidx = idx + cloud_row0;
    const uint4* __restrict__ cpts = points + (size_t)cloud * n * c8;
    const float* __restrict__ cxyz = xyz + (size_t)cloud * n * 3;
    const float* __restrict__ cctr = new_xyz + (size_t)cloud * m * 3;
    for (unsigned r0 = (warp * RPW + sub) * R; r0 < rows_per_cloud; r0 += warps * RPW * R) {
        const uint4* __restrict__ src[R];
        unsigned short* __restrict__ fdst[R];
        int head[R];
        bool ok[R];
#pragma unroll
        for (int rr = 0; rr < R; ++rr) {
            const unsigned r = r0 + rr;
            ok[rr] = r < rows_per_cloud;
            const int a = ok[rr] ? __ldg(cidx + r) : 0;
            src[rr] = cpts + (size_t)a * c8;
            const size_t obase = (cloud_row0 + r) * w;
            fdst[rr] = out + obase + feat_lo;
            head[rr] = (int)((8u - (unsigned)((obase + (size_t)feat_lo) & 7u)) & 7u);
            // scalar slots: t < 3 the centred xyz, then head value t-3 or tail value c-8+(t-3) (11 slots)
            if (ok[rr]) {
                for (int t = g; t < 11; t += LPR) {
                    const int h = head[rr];
                    if (t < 3) {
                        const float val =
                            __fsub_rn(__ldg(cxyz + (size_t)a * 3 + t), __ldg(cctr + (size_t)(r / (unsigned)nsample) * 3 + t));
                        __stcs(out + obase + xyz_lo + t, f_to_h<DT>(val));
                        if (grouped_xyz) __stcs(grouped_xyz + (cloud_row0 + r) * 3 + t, val);
                    } else if (h != 0) {
                        const int e = t - 3 < h ? t - 3 : c - 8 + (t - 3);
                        __stcs(fdst[rr] + e, __ldg(reinterpret_cast<const unsigned short*>(src[rr]) + e));
                    }
                }
            }
        }
        for (int k0 = 0; k0 < c8; k0 += LPR) {
            const int k = k0 + g;
            uint4 v[R], nx[R];
#pragma unroll
            for (int rr = 0; rr < R; ++rr) {
                v[rr] = make_uint4(0u, 0u, 0u, 0u);
                if (ok[rr] && k < c8) v[rr] = __ldg(src[rr] + k);
            }
#pragma unroll
            for (int rr = 0; rr < R; ++rr) {
                nx[rr].x = __shfl_down_sync(kFullMask, v[rr].x, 1, LPR);
                nx[rr].y = __shfl_down_sync(kFullMask, v[rr].y, 1, LPR);
                nx[rr].z = __shfl_down_sync(kFullMask, v[rr].z, 1, LPR);
                nx[rr].w = __shfl_down_sync(kFullMask, v[rr].w, 1, LPR);
                if (g == LPR - 1 && ok[rr] && k + 1 < c8 && head[rr] != 0) nx[rr] = __ldg(src[rr] + k + 1);
            }
#pragma unroll
            for (int rr = 0; rr < R; ++rr) {
                if (!ok[rr] || k >= c8) continue;
                const int h = head[rr];
                unsigned short* __restrict__ d = fdst[rr];
                if (h == 0) {
                    __stcs(reinterpret_cast<uint4*>(d) + k, v[rr]);
                    continue;
                }
                if (k + 1 < c8) {  // values [h + 8k, h + 8k + 8) of the segment
                    const unsigned W[8] = {v[rr].x, v[rr].y, v[rr].z, v[rr].w, nx[rr].x, nx[rr].y, nx[rr].z, nx[rr].w};
                    const int q = h >> 1;
                    const unsigned sh = (unsigned)(h & 1) * 16u;
                    unsigned s5[5];
#pragma unroll
                    for (int i = 0; i < 5; ++i) s5[i] = q == 0 ? W[i] : (q == 1 ? W[i + 1] : (q == 2 ? W[i + 2] : W[i + 3]));
                    uint4 o;
                    o.x = __funnelshift_r(s5[0], s5[1], sh);
                    o.y = __funnelshift_r(s5[1], s5[2], sh);
                    o.z = __funnelshift_r(s5[2], s5[3], sh);
                    o.w = __funnelshift_r(s5[3], s5[4], sh);
                    __stcs(reinterpret_cast<uint4*>(d + h + 8 * k), o);
                }
            }
        }
    }
}

template <bool HAS_XYZ, int DT>
static int launch_group_rows_h(int b, int n, int c, int m, int nsample, const float* xyz, const float* new_xyz,
                               const unsigned short* points, const int* idx, int xyz_lo, int feat_lo, unsigned short* out,
                               float* grouped_xyz, cudaStream_t st) {
    const unsigned rpc = (unsigned)m * (unsigned)nsample;
    const unsigned cap = (148u * 32u + b - 1) / b;  // enough CTAs to fill the machine, then grid-stride
    if (HAS_XYZ && c > 0 && c % 8 == 0 && aligned16(points) && aligned16(out)) {
        const int c8 = c / 8;
        // lanes per row: the widest that leaves the fewest lanes idle in the row's last pass (C = 320: 40 vectors
        // are 5 full passes of 8 lanes, not 32 + 8 of 32 lanes)
        int lpr = 8;
        for (int l = 16; l <= 32; l *= 2)
            if ((c8 + l - 1) / l * l <= (c8 + lpr - 1) / lpr * lpr) lpr = l;
        constexpr int R = 2;
        const unsigned rows_per_block = (kCopyThreads / 32) * (32 / lpr) * R;
        unsigned gx = (rpc + rows_per_block - 1) / rows_per_block;
        if (gx > cap) gx = cap;
        if (gx < 1) gx = 1;
        dim3 grid(gx, b, 1);
        const uint4* p8 = reinterpret_cast<const uint4*>(points);
        if (lpr == 8) group_concat_h_vec_kernel<8, R, DT><<<grid, kCopyThreads, 0, st>>>(n, c8, nsample, rpc, xyz, new_xyz, p8, idx, xyz_lo, feat_lo, out, grouped_xyz);
        else if (lpr == 16) group_concat_h_vec_kernel<16, R, DT><<<grid, kCopyThreads, 0, st>>>(n, c8, nsample, rpc, xyz, new_xyz, p8, idx, xyz_lo, feat_lo, out, grouped_xyz);
        else group_concat_h_vec_kernel<32, R, DT><<<grid, kCopyThreads, 0, st>>>(n, c8, nsample, rpc, xyz, new_xyz, p8, idx, xyz_lo, feat_lo, out, grouped_xyz);
        return finish_launch();
    }
    const int w = c + (HAS_XYZ ? 3 : 0);
    const int lpr = w <= 4 ? 4 : (w <= 8 ? 8 : (w <= 16 ? 16 : 32));
    const unsigned rows_per_block = (kCopyThreads / 32) * (32 / lpr) * 2;
    unsigned gx = (rpc + rows_per_block - 1) / rows_per_block;
    if (gx > cap) gx = cap;
    if (gx < 1) gx = 1;
    dim3 grid(gx, b, 1);
#define PN2_GROUP_ROWS_H(L) \
    group_rows_h_kernel<L, HAS_XYZ, DT><<<grid, kCopyThreads, 0, st>>>(n, c, nsample, rpc, xyz, new_xyz, points, idx, xyz_lo, feat_lo, out, grouped_xyz)
    if (lpr == 4) PN2_GROUP_ROWS_H(4);
    else if (lpr == 8) PN2_GROUP_ROWS_H(8);
    else if (lpr == 16) PN2_GROUP_ROWS_H(16);
    else PN2_GROUP_ROWS_H(32);
#undef PN2_GROUP_ROWS_H
    return finish_launch();
}

// group_point_grad with a 16-bit grad_out: widened exactly, float atomics into float32 grad_points.  VEC: 4 channels
// per thread (8-byte loads, red.global.add.v4.f32), c % 4 == 0.
template <typename IndexT, int DT, bool VEC>
__global__ void __launch_bounds__(kCopyThreads)
group_point_grad_h_kernel(int n, int c, IndexT rows_per_cloud, IndexT total, const unsigned short* __restrict__ grad_out,
                          const int* __restrict__ idx, float* __restrict__ grad_points) {
    constexpr int W = VEC ? 4 : 1;
    const int cw = c / W;
    const IndexT stride = (IndexT)gridDim.x * kCopyThreads;
    for (IndexT e = (IndexT)blockIdx.x * kCopyThreads + threadIdx.x; e < total; e += stride) {
        const IndexT row = e / (IndexT)cw;
        const int l = (int)(e - row * (IndexT)cw) * W;
        const IndexT cloud = row / rows_per_cloud;
        const int a = __ldg(idx + row);
        float* gp = grad_points + ((size_t)cloud * n + a) * c + l;
        if (VEC) {
            const uint2 u = __ldcs(reinterpret_cast<const uint2*>(grad_out) + e);
            const float2 lo = h2_to_f2<DT>(u.x), hi = h2_to_f2<DT>(u.y);
            atomicAdd(reinterpret_cast<float4*>(gp), make_float4(lo.x, lo.y, hi.x, hi.y));
        } else {
            atomicAdd(gp, h_to_f<DT>(__ldcs(grad_out + e)));
        }
    }
}

template <int DT>
static int group_point_grad_h(int b, int n, int c, int m, int nsample, const unsigned short* grad_out, const int* idx,
                              float* grad_points, cudaStream_t st) {
    const unsigned long long rpc = (unsigned long long)m * nsample;
    const unsigned long long total = (unsigned long long)b * rpc * c;
    if (c % 4 == 0 && (reinterpret_cast<uintptr_t>(grad_out) & 7u) == 0 && aligned16(grad_points)) {
        const unsigned long long tv = total / 4;
        const unsigned grid = grid_for(tv, kCopyThreads);
        if (tv < (1ull << 31))
            group_point_grad_h_kernel<unsigned, DT, true><<<grid, kCopyThreads, 0, st>>>(n, c, (unsigned)rpc, (unsigned)tv, grad_out, idx, grad_points);
        else
            group_point_grad_h_kernel<unsigned long long, DT, true><<<grid, kCopyThreads, 0, st>>>(n, c, rpc, tv, grad_out, idx, grad_points);
    } else {
        const unsigned grid = grid_for(total, kCopyThreads);
        if (total < (1ull << 31))
            group_point_grad_h_kernel<unsigned, DT, false><<<grid, kCopyThreads, 0, st>>>(n, c, (unsigned)rpc, (unsigned)total, grad_out, idx, grad_points);
        else
            group_point_grad_h_kernel<unsigned long long, DT, false><<<grid, kCopyThreads, 0, st>>>(n, c, rpc, total, grad_out, idx, grad_points);
    }
    return finish_launch();
}

static bool aligned4(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 3u) == 0; }


}  // namespace pn2

extern "C" {

int pn2_gather_point(int b, int n, int m, const float* inp, const int* idx, float* out, void* stream) {
    using namespace pn2;
    if (b < 0 || n <= 0 || m < 0) return (int)cudaErrorInvalidValue;
    if (b == 0 || m == 0) return 0;
    if (!inp || !idx || !out) return (int)cudaErrorInvalidValue;
    const long long total = (long long)b * m;
    gather_point_kernel<<<grid_for(total, kCopyThreads), kCopyThreads, 0, as_stream(stream)>>>(n, m, total, inp, idx, out);
    return finish_launch();
}

int pn2_gather_point_grad(int b, int n, int m, const float* out_g, const int* idx, float* inp_g, void* stream) {
    using namespace pn2;
    if (b < 0 || n <= 0 || m < 0) return (int)cudaErrorInvalidValue;
    if (b == 0 || m == 0) return 0;
    if (!out_g || !idx || !inp_g) return (int)cudaErrorInvalidValue;
    const long long total = (long long)b * m;
    gather_point_grad_kernel<<<grid_for(total, kCopyThreads), kCopyThreads, 0, as_stream(stream)>>>(n, m, total, out_g, idx, inp_g);
    return finish_launch();
}

int pn2_group_point(int b, int n, int c, int m, int nsample, const float* points, const int* idx, float* out,
                    void* stream) {
    using namespace pn2;
    if (b < 0 || n <= 0 || c < 0 || m < 0 || nsample < 0) return (int)cudaErrorInvalidValue;
    const unsigned long long rows = (unsigned long long)b * m * nsample;
    const unsigned long long total = rows * c;
    if (total == 0) return 0;
    if (!points || !idx || !out) return (int)cudaErrorInvalidValue;
    cudaStream_t st = as_stream(stream);
    const unsigned long long rpc = (unsigned long long)m * nsample;
    if (c % 4 == 0 && aligned16(points) && aligned16(out)) {
        const unsigned long long tv = total / 4;
        static int mode = -1, ctas_per_sm = 0;
        if (mode < 0) {  // tuning hooks: PN2_GROUP_MODE 0 = row-batched (default), 1 = flat one-vector-per-thread
            const char* e = getenv("PN2_GROUP_MODE");
            mode = e ? atoi(e) : 0;
            const char* gq = getenv("PN2_GROUP_CTAS");
            ctas_per_sm = gq ? atoi(gq) : 16;
        }
        if (mode == 0 && rpc < (1ull << 32) && b <= 65535) {
            const int c4 = c / 4;
            const int lpr = c4 <= 4 ? 4 : (c4 <= 8 ? 8 : (c4 <= 16 ? 16 : 32));
            constexpr int R = 4;
            const unsigned rows_per_block = (kCopyThreads / 32) * (32 / lpr) * R;
            unsigned gx = (unsigned)((rpc + rows_per_block - 1) / rows_per_block);
            const unsigned cap = (148u * (unsigned)ctas_per_sm + b - 1) / b;
            if (gx > cap) gx = cap;
            if (gx < 1) gx = 1;
            dim3 grid(gx, b, 1);
            if (lpr == 4) group_rows_vec4_kernel<4, R><<<grid, kCopyThreads, 0, st>>>(n, c4, (unsigned)rpc, (const float4*)points, idx, (float4*)out);
            else if (lpr == 8) group_rows_vec4_kernel<8, R><<<grid, kCopyThreads, 0, st>>>(n, c4, (unsigned)rpc, (const float4*)points, idx, (float4*)out);
            else if (lpr == 16) group_rows_vec4_kernel<16, R><<<grid, kCopyThreads, 0, st>>>(n, c4, (unsigned)rpc, (const float4*)points, idx, (float4*)out);
            else group_rows_vec4_kernel<32, R><<<grid, kCopyThreads, 0, st>>>(n, c4, (unsigned)rpc, (const float4*)points, idx, (float4*)out);
            return finish_launch();
        }
        unsigned long long blocks = (tv + kCopyThreads - 1) / kCopyThreads;
        const unsigned long long cap = 148ull * (unsigned long long)ctas_per_sm;
        const unsigned grid = (unsigned)(blocks > cap ? cap : (blocks < 1 ? 1 : blocks));
        if (tv < (1ull << 31))
            group_point_vec4_kernel<unsigned, 1><<<grid, kCopyThreads, 0, st>>>(n, c / 4, (unsigned)rpc, (unsigned)tv, (const float4*)points, idx, (float4*)out);
        else
            group_point_vec4_kernel<unsigned long long, 1><<<grid, kCopyThreads, 0, st>>>(n, c / 4, rpc, tv, (const float4*)points, idx, (float4*)out);
    } else {
        if (rpc >= (1ull << 32) || b > 65535) return (int)cudaErrorInvalidValue;
        return launch_group_rows<false>(b, n, c, m, nsample, nullptr, nullptr, points, idx, 0, 0, out, nullptr, st);
    }
    return finish_launch();
}

int pn2_group_point_grad(int b, int n, int c, int m, int nsample, const float* grad_out, const int* idx,
                         float* grad_points, void* stream) {
    using namespace pn2;
    if (b < 0 || n <= 0 || c < 0 || m < 0 || nsample < 0) return (int)cudaErrorInvalidValue;
    const unsigned long long rows = (unsigned long long)b * m * nsample;
    const unsigned long long total = rows * c;
    if (total == 0) return 0;
    if (!grad_out || !idx || !grad_points) return (int)cudaErrorInvalidValue;
    cudaStream_t st = as_stream(stream);
    const unsigned long long rpc = (unsigned long long)m * nsample;
    if (c % 4 == 0 && aligned16(grad_out) && aligned16(grad_points)) {
        const unsigned long long tv = total / 4;
        const unsigned grid = grid_for(tv, kCopyThreads);
        if (tv < (1ull << 31))
            group_point_grad_vec4_kernel<unsigned><<<grid, kCopyThreads, 0, st>>>(
                n, c / 4, (unsigned)rpc, (unsigned)tv, (const float4*)grad_out, idx, (float4*)grad_points);
        else
            group_point_grad_vec4_kernel<unsigned long long><<<grid, kCopyThreads, 0, st>>>(
                n, c / 4, rpc, tv, (const float4*)grad_out, idx, (float4*)grad_points);
    } else {
        const unsigned grid = grid_for(total, kCopyThreads);
        if (total < (1ull << 31))
            group_point_grad_scalar_kernel<unsigned><<<grid, kCopyThreads, 0, st>>>(n, c, (unsigned)rpc, (unsigned)total, grad_out, idx, grad_points);
        else
            group_point_grad_scalar_kernel<unsigned long long><<<grid, kCopyThreads, 0, st>>>(n, c, rpc, total, grad_out, idx, grad_points);
    }
    return finish_launch();
}

int pn2_group_concat(int b, int n, int c, int m, int nsample, const float* xyz, const float* new_xyz,
                     const float* points, const int* idx, int xyz_first, float* out, float* grouped_xyz,
                     void* stream) {
    using namespace pn2;
    if (b < 0 || n <= 0 || c < 0 || m < 0 || nsample < 0) return (int)cudaErrorInvalidValue;
    const unsigned long long rpc = (unsigned long long)m * nsample;
    if (b == 0 || rpc == 0) return 0;
    if (!xyz || !new_xyz || !idx || !out || (c > 0 && !points)) return (int)cudaErrorInvalidValue;
    if (rpc >= (1ull << 32) || b > 65535) return (int)cudaErrorInvalidValue;
    const int xyz_lo = xyz_first ? 0 : c, feat_lo = xyz_first ? 3 : 0;
    return launch_group_rows<true>(b, n, c, m, nsample, xyz, new_xyz, points, idx, xyz_lo, feat_lo, out, grouped_xyz,
                                   as_stream(stream));
}

int pn2_selection_sort(int b, int n, int m, int k, const float* dist, int* outi, float* out, void* stream) {
    using namespace pn2;
    if (b < 0 || n <= 0 || m < 0 || k <= 0) return (int)cudaErrorInvalidValue;
    const long long rows = (long long)b * m;
    if (rows == 0) return 0;
    if (!dist || !outi || !out) return (int)cudaErrorInvalidValue;
    const unsigned long long blocks = ((unsigned long long)rows * 32 + kCopyThreads - 1) / kCopyThreads;
    if (blocks > 0x7fffffffull) return (int)cudaErrorInvalidValue;
    selection_sort_kernel<<<(unsigned)blocks, kCopyThreads, 0, as_stream(stream)>>>(n, k, rows, dist, outi, out);
    return finish_launch();
}

int pn2_group_point_h(int dtype, int b, int n, int c, int m, int nsample, const void* points, const int* idx, void* out,
                      void* stream) {
    using namespace pn2;
    if (!valid_half_dtype(dtype)) return (int)cudaErrorInvalidValue;
    if (b < 0 || n <= 0 || c < 0 || m < 0 || nsample < 0) return (int)cudaErrorInvalidValue;
    const unsigned long long rpc = (unsigned long long)m * nsample;
    if ((unsigned long long)b * rpc * c == 0) return 0;
    if (!points || !idx || !out) return (int)cudaErrorInvalidValue;
    // the bytes do not depend on the element type: even rows on 4-byte aligned bases are rows of c/2 float32 words
    if (c % 2 == 0 && aligned4(points) && aligned4(out))
        return pn2_group_point(b, n, c / 2, m, nsample, static_cast<const float*>(points), idx, static_cast<float*>(out), stream);
    if (rpc >= (1ull << 32) || b > 65535) return (int)cudaErrorInvalidValue;
    return launch_group_rows_h<false, PN2_DTYPE_BF16>(b, n, c, m, nsample, nullptr, nullptr, static_cast<const unsigned short*>(points),
                                                      idx, 0, 0, static_cast<unsigned short*>(out), nullptr, as_stream(stream));
}

int pn2_group_point_grad_h(int dtype, int b, int n, int c, int m, int nsample, const void* grad_out, const int* idx,
                           float* grad_points, void* stream) {
    using namespace pn2;
    if (!valid_half_dtype(dtype)) return (int)cudaErrorInvalidValue;
    if (b < 0 || n <= 0 || c < 0 || m < 0 || nsample < 0) return (int)cudaErrorInvalidValue;
    if ((unsigned long long)b * m * nsample * c == 0) return 0;
    if (!grad_out || !idx || !grad_points) return (int)cudaErrorInvalidValue;
    const unsigned short* g = static_cast<const unsigned short*>(grad_out);
    if (dtype == PN2_DTYPE_BF16) return group_point_grad_h<PN2_DTYPE_BF16>(b, n, c, m, nsample, g, idx, grad_points, as_stream(stream));
    return group_point_grad_h<PN2_DTYPE_F16>(b, n, c, m, nsample, g, idx, grad_points, as_stream(stream));
}

int pn2_group_concat_h(int dtype, int b, int n, int c, int m, int nsample, const float* xyz, const float* new_xyz,
                       const void* points, const int* idx, int xyz_first, void* out, float* grouped_xyz, void* stream) {
    using namespace pn2;
    if (!valid_half_dtype(dtype)) return (int)cudaErrorInvalidValue;
    if (b < 0 || n <= 0 || c < 0 || m < 0 || nsample < 0) return (int)cudaErrorInvalidValue;
    const unsigned long long rpc = (unsigned long long)m * nsample;
    if (b == 0 || rpc == 0) return 0;
    if (!xyz || !new_xyz || !idx || !out || (c > 0 && !points)) return (int)cudaErrorInvalidValue;
    if (rpc >= (1ull << 32) || b > 65535) return (int)cudaErrorInvalidValue;
    const int xyz_lo = xyz_first ? 0 : c, feat_lo = xyz_first ? 3 : 0;
    const unsigned short* p = static_cast<const unsigned short*>(points);
    unsigned short* o = static_cast<unsigned short*>(out);
    if (dtype == PN2_DTYPE_BF16)
        return launch_group_rows_h<true, PN2_DTYPE_BF16>(b, n, c, m, nsample, xyz, new_xyz, p, idx, xyz_lo, feat_lo, o, grouped_xyz, as_stream(stream));
    return launch_group_rows_h<true, PN2_DTYPE_F16>(b, n, c, m, nsample, xyz, new_xyz, p, idx, xyz_lo, feat_lo, o, grouped_xyz, as_stream(stream));
}

}  // extern "C"
