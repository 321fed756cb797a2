// interpolate.cu — three_nn, three_interpolate (+grad) and the fused feature-propagation front
// end, for sm_100a.
//
// Replaces the CPU-only functions of the reference (tf_ops/3d_interpolation/tf_interpolate.cpp):
//   threenn_cpu :60-103, threeinterpolate_cpu :107-127, threeinterpolate_grad_cpu :131-153
// — which TensorFlow runs on the host with D2H/H2D copies around them — with device kernels.
//
// three_nn is bit-exact with the reference's x86 arithmetic: squared distance without
// contraction (pn2::d2_nofma), strict '<' three-way insertion in ascending known index (earlier
// index wins ties), +inf / index 0 for missing neighbours.  three_interpolate evaluates
// ((p1*w1 + p2*w2) + p3*w3) with every operation rounded on its own, i.e. also bit-exact (the
// contract only asks for 1e-5 abs).
#include <math.h>

#include <atomic>

#include "pn2_common.cuh"

namespace pn2 {

constexpr int kNnThreads = 128;
constexpr int kNnTile = 2048;  // known points per shared-memory tile (24 KB as pairs)

struct Top3 {
    float d1, d2, d3;
    int i1, i2, i3;
};

__device__ __forceinline__ void top3_init(Top3& t) {
    t.d1 = t.d2 = t.d3 = INFINITY;
    t.i1 = t.i2 = t.i3 = 0;
}

// Branch-free insertion (selects only): the reference's strict '<' cascade (tf_interpolate.cpp:74-89).
// A candidate that is not < d3 leaves the state untouched.
__device__ __forceinline__ void top3_insert(Top3& t, float d, int k) {
    const bool c3 = d < t.d3, c2 = d < t.d2, c1 = d < t.d1;  // c1 => c2 => c3 (d1 <= d2 <= d3)
    const float nd3 = c2 ? t.d2 : d;
    const int ni3 = c2 ? t.i2 : k;
    const float nd2 = c1 ? t.d1 : d;
    const int ni2 = c1 ? t.i1 : k;
    t.d3 = c3 ? nd3 : t.d3;
    t.i3 = c3 ? ni3 : t.i3;
    t.d2 = c2 ? nd2 : t.d2;
    t.i2 = c2 ? ni2 : t.i2;
    t.d1 = c1 ? d : t.d1;
    t.i1 = c1 ? k : t.i1;
}

// packed FP32x2 helpers (SASS FADD2 / FMUL2): two known points per instruction for the differences
// and the squares, IEEE round-to-nearest per half
__device__ __forceinline__ unsigned long long nn_pack(float a, float b) {
    unsigned long long r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(a), "f"(b));
    return r;
}
__device__ __forceinline__ void nn_unpack(unsigned long long v, float& a, float& b) {
    asm("mov.b64 {%0, %1}, %2;" : "=f"(a), "=f"(b) : "l"(v));
}
__device__ __forceinline__ unsigned long long nn_sub2(unsigned long long a, unsigned long long b) {
    unsigned long long r;
    asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
__device__ __forceinline__ unsigned long long nn_mul2(unsigned long long a, unsigned long long b) {
    unsigned long long r;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
constexpr int kNnPairs = kNnTile / 2;

// Shared-memory tile of known points stored as PAIRS: s_xy[i] = (x0, x1, y0, y1) of points 2i, 2i+1,
// s_z[i] = (z0, z1).  The tail up to a multiple of 2 pairs is +inf (distance +inf never passes '<').
struct KnownTile {
    ulonglong2 xy[kNnPairs];
    unsigned long long z[kNnPairs];
};

__device__ __forceinline__ int stage_known(KnownTile& tile, const float* __restrict__ known, int base, int m, int tid,
                                           int nthreads) {
    const int tn = min(kNnTile, m - base);
    const int tp_pad = (((tn + 1) >> 1) + 1) & ~1;  // pairs, rounded up to an even count
    float* sxy = reinterpret_cast<float*>(tile.xy);
    float* sz = reinterpret_cast<float*>(tile.z);
    for (int p = tid; p < 2 * tp_pad; p += nthreads) {
        float x = INFINITY, y = INFINITY, z = INFINITY;
        if (p < tn) {
            const float* s = known + (size_t)(base + p) * 3;
            x = s[0];
            y = s[1];
            z = s[2];
        }
        const int pi = p >> 1, par = p & 1;
        sxy[4 * pi + par] = x;
        sxy[4 * pi + 2 + par] = y;
        sz[2 * pi + par] = z;
    }
    return tp_pad;
}

// Scan one tile.  Candidates are offered in ascending known index; the (rare, per-lane) insertion
// sits behind a warp-uniform vote so the common path is distance math + one compare per point.
__device__ __forceinline__ void scan_tile(Top3& t, const KnownTile& tile, int tp_pad, int base, float ux, float uy,
                                          float uz) {
    const unsigned long long UX = nn_pack(ux, ux), UY = nn_pack(uy, uy), UZ = nn_pack(uz, uz);
    for (int p = 0; p < tp_pad; p += 2) {
        float d[4];
#pragma unroll
        for (int u = 0; u < 2; ++u) {
            const ulonglong2 xy = tile.xy[p + u];
            const unsigned long long zz = tile.z[p + u];
            const unsigned long long dx = nn_sub2(xy.x, UX), dy = nn_sub2(xy.y, UY), dz = nn_sub2(zz, UZ);
            // squares packed, sums scalar: ptxas contracts mul.rn.f32x2 + add.rn.f32x2 into FFMA2
            // (CUDA 12.9, even with -fmad=false or when the add is spelled fma(a,1,b)), which would
            // skip the rounding of the products that the reference's x86 code performs; the scalar
            // __fadd_rn intrinsic is never contracted
            float xx0, xx1, yy0, yy1, zz0, zz1;
            nn_unpack(nn_mul2(dx, dx), xx0, xx1);
            nn_unpack(nn_mul2(dy, dy), yy0, yy1);
            nn_unpack(nn_mul2(dz, dz), zz0, zz1);
            d[2 * u] = __fadd_rn(__fadd_rn(xx0, yy0), zz0);
            d[2 * u + 1] = __fadd_rn(__fadd_rn(xx1, yy1), zz1);
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            if (__any_sync(kFullMask, d[u] < t.d3)) top3_insert(t, d[u], base + 2 * p + u);
        }
    }
}

// One thread per unknown point; known points broadcast from shared memory.
__global__ void __launch_bounds__(kNnThreads)
three_nn_kernel(int n, int m, const float* __restrict__ xyz1, const float* __restrict__ xyz2,
                float* __restrict__ dist, int* __restrict__ idx) {
    __shared__ KnownTile s_tile;
    const int tid = threadIdx.x;
    const int cloud = blockIdx.y;
    const int j = blockIdx.x * kNnThreads + tid;
    const bool valid = j < n;
    const float* __restrict__ known = xyz2 + (size_t)cloud * m * 3;
    float ux = 0.f, uy = 0.f, uz = 0.f;
    if (valid) {
        const float* u = xyz1 + ((size_t)cloud * n + j) * 3;
        ux = u[0];
        uy = u[1];
        uz = u[2];
    }
    Top3 t;
    top3_init(t);
    for (int base = 0; base < m; base += kNnTile) {
        if (base) __syncthreads();
        const int tp_pad = stage_known(s_tile, known, base, m, tid, kNnThreads);
        __syncthreads();
        scan_tile(t, s_tile, tp_pad, base, ux, uy, uz);
    }
    if (valid) {
        float* dd = dist + ((size_t)cloud * n + j) * 3;
        int* ii = idx + ((size_t)cloud * n + j) * 3;
        dd[0] = t.d1; dd[1] = t.d2; dd[2] = t.d3;
        ii[0] = t.i1; ii[1] = t.i2; ii[2] = t.i3;
    }
}

// ---- three_interpolate ---------------------------------------------------------------------------
__device__ __forceinline__ float interp3(float p1, float p2, float p3, float w1, float w2, float w3) {
    return __fadd_rn(__fadd_rn(__fmul_rn(p1, w1), __fmul_rn(p2, w2)), __fmul_rn(p3, w3));
}

// 8 16-bit values of each of three rows (16-byte vectors): widened exactly, interp3, one rounding each
template <int DT>
__device__ __forceinline__ unsigned interp3_h2(unsigned a, unsigned b, unsigned c, float w1, float w2, float w3) {
    const float2 x = h2_to_f2<DT>(a), y = h2_to_f2<DT>(b), z = h2_to_f2<DT>(c);
    return f2_to_h2<DT>(interp3(x.x, y.x, z.x, w1, w2, w3), interp3(x.y, y.y, z.y, w1, w2, w3));
}
template <int DT>
__device__ __forceinline__ uint4 interp3_h8(uint4 a, uint4 b, uint4 c, float w1, float w2, float w3) {
    return make_uint4(interp3_h2<DT>(a.x, b.x, c.x, w1, w2, w3), interp3_h2<DT>(a.y, b.y, c.y, w1, w2, w3),
                      interp3_h2<DT>(a.z, b.z, c.z, w1, w2, w3), interp3_h2<DT>(a.w, b.w, c.w, w1, w2, w3));
}

constexpr int kItThreads = 256;

// One thread per output float4 (U = 1).  Measured in round 2 (profiles/r2_interp_experiments.txt): U = 4 outputs in
// flight per thread costs 96 registers and quarter occupancy (40 us against 27 us at 16 x 8192 <- 1024, C = 128);
// staging channel slices of the known features in shared memory is worse still (73 us: one 160 KB CTA per SM
// cannot hide its own slice load).  The kernel moves 78 MB in 27 us; 8 us of that is the fixed cost every
// kernel shows in this harness (launch + cold TLB/L2 after the flush), see DESIGN.md section 4.
template <typename IndexT, int U>
__global__ void __launch_bounds__(kItThreads)
three_interp_vec4_kernel(int m, int c4, IndexT rows_per_cloud, IndexT total_vec, const float4* __restrict__ points,
                         const int* __restrict__ idx, const float* __restrict__ weight, float4* __restrict__ out) {
    const IndexT stride = (IndexT)gridDim.x * kItThreads;
    for (IndexT v0 = (IndexT)blockIdx.x * kItThreads + threadIdx.x; v0 < total_vec; v0 += stride * U) {
        int i1[U], i2[U], i3[U];
        float w1[U], w2[U], w3[U];
        const float4* pb[U];
        bool ok[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const IndexT v = v0 + (IndexT)u * stride;
            ok[u] = v < total_vec;
            const IndexT row = ok[u] ? v / (IndexT)c4 : 0;
            const int l = ok[u] ? (int)(v - row * (IndexT)c4) : 0;
            const IndexT cloud = row / rows_per_cloud;
            i1[u] = __ldg(idx + (size_t)row * 3 + 0);
            i2[u] = __ldg(idx + (size_t)row * 3 + 1);
            i3[u] = __ldg(idx + (size_t)row * 3 + 2);
            w1[u] = __ldg(weight + (size_t)row * 3 + 0);
            w2[u] = __ldg(weight + (size_t)row * 3 + 1);
            w3[u] = __ldg(weight + (size_t)row * 3 + 2);
            pb[u] = points + (size_t)cloud * m * c4 + l;
        }
        float4 a[U], b[U], c[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            if (ok[u]) {
                a[u] = __ldg(pb[u] + (size_t)i1[u] * c4);
                b[u] = __ldg(pb[u] + (size_t)i2[u] * c4);
                c[u] = __ldg(pb[u] + (size_t)i3[u] * c4);
            }
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
            if (ok[u]) {
                float4 o;
                o.x = interp3(a[u].x, b[u].x, c[u].x, w1[u], w2[u], w3[u]);
                o.y = interp3(a[u].y, b[u].y, c[u].y, w1[u], w2[u], w3[u]);
                o.z = interp3(a[u].z, b[u].z, c[u].z, w1[u], w2[u], w3[u]);
                o.w = interp3(a[u].w, b[u].w, c[u].w, w1[u], w2[u], w3[u]);
                st_stream_f4(out + v0 + (IndexT)u * stride, o);
            }
        }
    }
}

template <typename IndexT>
__global__ void __launch_bounds__(kItThreads)
three_interp_scalar_kernel(int m, int c, IndexT rows_per_cloud, IndexT total, const float* __restrict__ points,
                           const int* __restrict__ idx, const float* __restrict__ weight, float* __restrict__ out) {
    const IndexT stride = (IndexT)gridDim.x * kItThreads;
    for (IndexT e = (IndexT)blockIdx.x * kItThreads + threadIdx.x; e < total; e += stride) {
        const IndexT row = e / (IndexT)c;
        const int l = (int)(e - row * (IndexT)c);
        const IndexT cloud = row / rows_per_cloud;
        const int* ii = idx + (size_t)row * 3;
        const float* w = weight + (size_t)row * 3;
        const float* pb = points + (size_t)cloud * m * c + l;
        out[e] = interp3(__ldg(pb + (size_t)__ldg(ii + 0) * c), __ldg(pb + (size_t)__ldg(ii + 1) * c),
                         __ldg(pb + (size_t)__ldg(ii + 2) * c), __ldg(w + 0), __ldg(w + 1), __ldg(w + 2));
    }
}

// grad_points[b, idx[b,j,t], l] += grad_out[b,j,l] * weight[b,j,t]
template <typename IndexT>
__global__ void __launch_bounds__(kItThreads)
three_interp_grad_vec4_kernel(int m, int c4, IndexT rows_per_cloud, IndexT total_vec,
                              const float4* __restrict__ grad_out, const int* __restrict__ idx,
                              const float* __restrict__ weight, float4* __restrict__ grad_points) {
    const IndexT stride = (IndexT)gridDim.x * kItThreads;
    for (IndexT v = (IndexT)blockIdx.x * kItThreads + threadIdx.x; v < total_vec; v += stride) {
        const IndexT row = v / (IndexT)c4;
        const int l = (int)(v - row * (IndexT)c4);
        const IndexT cloud = row / rows_per_cloud;
        const float4 g = __ldcs(grad_out + v);
        float4* gb = grad_points + (size_t)cloud * m * c4 + l;
#pragma unroll
        for (int t = 0; t < 3; ++t) {
            const int i = __ldg(idx + (size_t)row * 3 + t);
            const float w = __ldg(weight + (size_t)row * 3 + t);
            atomicAdd(gb + (size_t)i * c4,
                      make_float4(__fmul_rn(g.x, w), __fmul_rn(g.y, w), __fmul_rn(g.z, w), __fmul_rn(g.w, w)));
        }
    }
}

template <typename IndexT>
__global__ void __launch_bounds__(kItThreads)
three_interp_grad_scalar_kernel(int m, int c, IndexT rows_per_cloud, IndexT total, const float* __restrict__ grad_out,
                                const int* __restrict__ idx, const float* __restrict__ weight,
                                float* __restrict__ grad_points) {
    const IndexT stride = (IndexT)gridDim.x * kItThreads;
    for (IndexT e = (IndexT)blockIdx.x * kItThreads + threadIdx.x; e < total; e += stride) {
        const IndexT row = e / (IndexT)c;
        const int l = (int)(e - row * (IndexT)c);
        const IndexT cloud = row / rows_per_cloud;
        const float g = __ldcs(grad_out + e);
        float* gb = grad_points + (size_t)cloud * m * c + l;
#pragma unroll
        for (int t = 0; t < 3; ++t)
            atomicAdd(gb + (size_t)__ldg(idx + (size_t)row * 3 + t) * c, __fmul_rn(g, __ldg(weight + (size_t)row * 3 + t)));
    }
}

// ---- fused FP front end: three_nn -> inverse-distance weights -> three_interpolate -> concat -----
// utils/pointnet_util.py:211-219.  G lanes share one unknown point: lane g scans the known points of
// pairs p = g, g+G, ... (ascending index inside the lane), the G partial top-3 lists are merged by a
// shuffle butterfly under (distance, index) — exactly the order the reference's strict '<' scan over
// ascending indices produces — so small layers (64 or 256 unknown points per cloud) still fill the
// machine: a CTA covers 128/G points.  Phase 2 writes the CTA's rows of the output
// [interpolated (c2) | points1 (c1)] with consecutive lanes on consecutive channels; dist / idx /
// weight never touch HBM unless the caller asks for them, and the concat of :219 is not a separate pass.
__device__ __forceinline__ void top3_insert_lex(Top3& t, float d, int k) {
    // like top3_insert, with ties broken by the smaller index (candidates arrive out of index order)
    const bool c3 = d < t.d3 || (d == t.d3 && k < t.i3), c2 = d < t.d2 || (d == t.d2 && k < t.i2),
               c1 = d < t.d1 || (d == t.d1 && k < t.i1);
    const float nd3 = c2 ? t.d2 : d;
    const int ni3 = c2 ? t.i2 : k;
    const float nd2 = c1 ? t.d1 : d;
    const int ni2 = c1 ? t.i1 : k;
    t.d3 = c3 ? nd3 : t.d3;
    t.i3 = c3 ? ni3 : t.i3;
    t.d2 = c2 ? nd2 : t.d2;
    t.i2 = c2 ? ni2 : t.i2;
    t.d1 = c1 ? d : t.d1;
    t.i1 = c1 ? k : t.i1;
}

// Phase 2 of fp_front_kernel for 16-bit features: 16-byte loads of 8 values when c2 and c1 are multiples of 8 and the
// rows are 16-byte aligned, else one value per lane.
template <int DT, int PPB>
__device__ __forceinline__ void fp_front_phase2_h(int rows, int c2, int c1, const unsigned short* __restrict__ pb,
                                                  const unsigned short* __restrict__ p1, unsigned short* __restrict__ ob,
                                                  const int (&s_i)[PPB][3], const float (&s_w)[PPB][3], int tid) {
    const int cw = c2 + c1;
    const bool vec = ((c2 | c1) & 7) == 0 &&
                     ((reinterpret_cast<uintptr_t>(pb) | reinterpret_cast<uintptr_t>(ob) | reinterpret_cast<uintptr_t>(p1)) & 15u) == 0;
    if (vec) {
        const int c28 = c2 >> 3, cw8 = cw >> 3, c18 = c1 >> 3;
        const uint4* pb8 = reinterpret_cast<const uint4*>(pb);
        const uint4* p18 = reinterpret_cast<const uint4*>(p1);
        uint4* ob8 = reinterpret_cast<uint4*>(ob);
        for (int e = tid; e < rows * cw8; e += kNnThreads) {
            const int r = e / cw8, l = e - r * cw8;
            uint4 o;
            if (l < c28) {
                const uint4 a = __ldg(pb8 + (size_t)s_i[r][0] * c28 + l), b = __ldg(pb8 + (size_t)s_i[r][1] * c28 + l),
                            cc = __ldg(pb8 + (size_t)s_i[r][2] * c28 + l);
                o = interp3_h8<DT>(a, b, cc, s_w[r][0], s_w[r][1], s_w[r][2]);
            } else {
                o = __ldcs(p18 + (size_t)r * c18 + (l - c28));
            }
            __stcs(ob8 + e, o);
        }
    } else {
        for (int e = tid; e < rows * cw; e += kNnThreads) {
            const int r = e / cw, l = e - r * cw;
            unsigned short o;
            if (l < c2)
                o = f_to_h<DT>(interp3(h_to_f<DT>(__ldg(pb + (size_t)s_i[r][0] * c2 + l)), h_to_f<DT>(__ldg(pb + (size_t)s_i[r][1] * c2 + l)),
                                       h_to_f<DT>(__ldg(pb + (size_t)s_i[r][2] * c2 + l)), s_w[r][0], s_w[r][1], s_w[r][2]));
            else
                o = __ldcs(p1 + (size_t)r * c1 + (l - c2));
            ob[e] = o;
        }
    }
}

// lane g of G scans pairs g, g+G, ... of the tile (2 points per pair)
template <int G>
__device__ __forceinline__ void scan_tile_strided(Top3& t, const KnownTile& tile, int tp_pad, int base, int g, float ux, float uy,
                                                  float uz) {
    const unsigned long long UX = nn_pack(ux, ux), UY = nn_pack(uy, uy), UZ = nn_pack(uz, uz);
    for (int p = g; p < tp_pad; p += G) {
        const ulonglong2 xy = tile.xy[p];
        const unsigned long long zz = tile.z[p];
        const unsigned long long dx = nn_sub2(xy.x, UX), dy = nn_sub2(xy.y, UY), dz = nn_sub2(zz, UZ);
        float xx0, xx1, yy0, yy1, zz0, zz1;
        nn_unpack(nn_mul2(dx, dx), xx0, xx1);
        nn_unpack(nn_mul2(dy, dy), yy0, yy1);
        nn_unpack(nn_mul2(dz, dz), zz0, zz1);
        const float d0 = __fadd_rn(__fadd_rn(xx0, yy0), zz0), d1 = __fadd_rn(__fadd_rn(xx1, yy1), zz1);
        if (d0 < t.d3) top3_insert(t, d0, base + 2 * p);
        if (d1 < t.d3) top3_insert(t, d1, base + 2 * p + 1);
    }
}

// DT: feature type of points1 / points2 / out (0 = float32, or PN2_DTYPE_BF16 / PN2_DTYPE_F16: values widened exactly,
// interp3 in float32, one rounding); phase 1 does not depend on it.
template <int G, int DT>
__global__ void __launch_bounds__(kNnThreads)
fp_front_kernel(int n, int m, int c2, int c1, const float* __restrict__ xyz1, const float* __restrict__ xyz2,
                const feat_t<DT>* __restrict__ points1, const feat_t<DT>* __restrict__ points2, feat_t<DT>* __restrict__ out,
                float* __restrict__ dist_o, int* __restrict__ idx_o, float* __restrict__ weight_o) {
    constexpr int PPB = kNnThreads / G;  // unknown points per CTA
    __shared__ KnownTile s_tile;
    __shared__ int s_i[PPB][3];
    __shared__ float s_w[PPB][3];
    const int tid = threadIdx.x;
    const int g = tid % G, slot = tid / G;
    const int cloud = blockIdx.y;
    const int j0 = blockIdx.x * PPB;
    const int j = j0 + slot;
    const bool valid = j < n;
    const float* __restrict__ known = xyz2 + (size_t)cloud * m * 3;
    float ux = 0.f, uy = 0.f, uz = 0.f;
    if (valid) {
        const float* u = xyz1 + ((size_t)cloud * n + j) * 3;
        ux = __ldg(u);
        uy = __ldg(u + 1);
        uz = __ldg(u + 2);
    }
    Top3 t;
    top3_init(t);
    for (int base = 0; base < m; base += kNnTile) {
        if (base) __syncthreads();
        const int tp_pad = stage_known(s_tile, known, base, m, tid, kNnThreads);
        __syncthreads();
        if (G == 1) scan_tile(t, s_tile, tp_pad, base, ux, uy, uz);
        else scan_tile_strided<G>(t, s_tile, tp_pad, base, g, ux, uy, uz);
    }
    if (G > 1) {  // merge the G partial lists of this point (all lanes end with the merged list)
#pragma unroll
        for (int o = 1; o < G; o <<= 1) {
            const float e1 = __shfl_xor_sync(kFullMask, t.d1, o), e2 = __shfl_xor_sync(kFullMask, t.d2, o),
                        e3 = __shfl_xor_sync(kFullMask, t.d3, o);
            const int f1 = __shfl_xor_sync(kFullMask, t.i1, o), f2 = __shfl_xor_sync(kFullMask, t.i2, o),
                      f3 = __shfl_xor_sync(kFullMask, t.i3, o);
            // +inf entries are the (inf, 0) filler of an unfilled slot: never insert them (index 0 would win ties)
            if (e1 < INFINITY) top3_insert_lex(t, e1, f1);
            if (e2 < INFINITY) top3_insert_lex(t, e2, f2);
            if (e3 < INFINITY) top3_insert_lex(t, e3, f3);
        }
    }
    // dist = max(dist, 1e-10); norm = sum(1/dist); weight = (1/dist)/norm   (pointnet_util.py:212-215)
    const float r1 = __fdiv_rn(1.0f, fmaxf(t.d1, 1e-10f));
    const float r2 = __fdiv_rn(1.0f, fmaxf(t.d2, 1e-10f));
    const float r3 = __fdiv_rn(1.0f, fmaxf(t.d3, 1e-10f));
    const float norm = __fadd_rn(__fadd_rn(r1, r2), r3);
    const float w1 = __fdiv_rn(r1, norm), w2 = __fdiv_rn(r2, norm), w3 = __fdiv_rn(r3, norm);
    if (g == 0) {
        s_i[slot][0] = t.i1; s_i[slot][1] = t.i2; s_i[slot][2] = t.i3;
        s_w[slot][0] = w1;   s_w[slot][1] = w2;   s_w[slot][2] = w3;
        if (valid) {
            const size_t o = ((size_t)cloud * n + j) * 3;
            if (dist_o) { dist_o[o] = t.d1; dist_o[o + 1] = t.d2; dist_o[o + 2] = t.d3; }
            if (idx_o) { idx_o[o] = t.i1; idx_o[o + 1] = t.i2; idx_o[o + 2] = t.i3; }
            if (weight_o) { weight_o[o] = w1; weight_o[o + 1] = w2; weight_o[o + 2] = w3; }
        }
    }
    __syncthreads();
    if (!out) return;
    const int rows = min(PPB, n - j0);
    const int cw = c2 + c1;  // output row width
    const feat_t<DT>* __restrict__ pb = points2 + (size_t)cloud * m * c2;
    const feat_t<DT>* __restrict__ p1 = points1 ? points1 + ((size_t)cloud * n + j0) * c1 : nullptr;
    feat_t<DT>* __restrict__ ob = out + ((size_t)cloud * n + j0) * cw;
    if constexpr (DT != 0) {
        fp_front_phase2_h<DT>(rows, c2, c1, pb, p1, ob, s_i, s_w, tid);
        return;
    } else {
    const bool vec = ((c2 | c1) & 3) == 0 &&
                     ((reinterpret_cast<uintptr_t>(pb) | reinterpret_cast<uintptr_t>(ob) | reinterpret_cast<uintptr_t>(p1)) & 15u) == 0;
    if (vec) {
        const int c24 = c2 >> 2, cw4 = cw >> 2, c14 = c1 >> 2;
        const float4* pb4 = reinterpret_cast<const float4*>(pb);
        const float4* p14 = reinterpret_cast<const float4*>(p1);
        float4* ob4 = reinterpret_cast<float4*>(ob);
        for (int e = tid; e < rows * cw4; e += kNnThreads) {
            const int r = e / cw4, l = e - r * cw4;
            float4 o;
            if (l < c24) {
                const float4 a = __ldg(pb4 + (size_t)s_i[r][0] * c24 + l), b = __ldg(pb4 + (size_t)s_i[r][1] * c24 + l),
                             cc = __ldg(pb4 + (size_t)s_i[r][2] * c24 + l);
                const float x1 = s_w[r][0], x2 = s_w[r][1], x3 = s_w[r][2];
                o.x = interp3(a.x, b.x, cc.x, x1, x2, x3);
                o.y = interp3(a.y, b.y, cc.y, x1, x2, x3);
                o.z = interp3(a.z, b.z, cc.z, x1, x2, x3);
                o.w = interp3(a.w, b.w, cc.w, x1, x2, x3);
            } else {
                o = __ldcs(p14 + (size_t)r * c14 + (l - c24));  // points1, read once
            }
            st_stream_f4(ob4 + e, o);
        }
    } else {
        for (int e = tid; e < rows * cw; e += kNnThreads) {
            const int r = e / cw, l = e - r * cw;
            float o;
            if (l < c2)
                o = interp3(__ldg(pb + (size_t)s_i[r][0] * c2 + l), __ldg(pb + (size_t)s_i[r][1] * c2 + l),
                            __ldg(pb + (size_t)s_i[r][2] * c2 + l), s_w[r][0], s_w[r][1], s_w[r][2]);
            else
                o = __ldcs(p1 + (size_t)r * c1 + (l - c2));
            ob[e] = o;
        }
    }
    }
}

template <int G, int DT>
static int launch_fp_front(int b, int n, int m, int c2, int c1, const float* xyz1, const float* xyz2, const feat_t<DT>* points1,
                           const feat_t<DT>* points2, feat_t<DT>* out, float* dist, int* idx, float* weight, cudaStream_t st) {
    constexpr int PPB = kNnThreads / G;
    dim3 grid((n + PPB - 1) / PPB, b, 1);
    fp_front_kernel<G, DT><<<grid, kNnThreads, 0, st>>>(n, m, c2, c1, xyz1, xyz2, points1, points2, out, dist, idx, weight);
    return finish_launch();
}

template <int DT>
static int fp_front_dispatch(int b, int n, int m, int c2, int c1, const float* xyz1, const float* xyz2, const feat_t<DT>* points1,
                             const feat_t<DT>* points2, feat_t<DT>* out, float* dist, int* idx, float* weight, cudaStream_t st) {
    // lanes per unknown point: as many as it takes to put ~2 CTAs on every SM (a CTA covers 128/G points),
    // but never more lanes than there are pairs of known points to share
    const long long pts = (long long)b * n;
    int G = 1;
    while (G < 32 && pts * G < 2LL * 148 * kNnThreads && 2 * G <= (m + 1) / 2) G *= 2;
    switch (G) {
        case 1: return launch_fp_front<1, DT>(b, n, m, c2, c1, xyz1, xyz2, points1, points2, out, dist, idx, weight, st);
        case 2: return launch_fp_front<2, DT>(b, n, m, c2, c1, xyz1, xyz2, points1, points2, out, dist, idx, weight, st);
        case 4: return launch_fp_front<4, DT>(b, n, m, c2, c1, xyz1, xyz2, points1, points2, out, dist, idx, weight, st);
        case 8: return launch_fp_front<8, DT>(b, n, m, c2, c1, xyz1, xyz2, points1, points2, out, dist, idx, weight, st);
        case 16: return launch_fp_front<16, DT>(b, n, m, c2, c1, xyz1, xyz2, points1, points2, out, dist, idx, weight, st);
        default: return launch_fp_front<32, DT>(b, n, m, c2, c1, xyz1, xyz2, points1, points2, out, dist, idx, weight, st);
    }
}

// ---- three_interpolate_grad without atomics: an inverse index, then one warp per known point ------
// grad_points[b,i,:] = sum over the entries e = 3j+t with idx[b,j,t] == i of grad_out[b,j,:] * weight[b,j,t],
// accumulated in ASCENDING e — the very order threeinterpolate_grad_cpu (tf_interpolate.cpp:131-153: j outer,
// t = 1,2,3 inner) adds them, each product and sum rounded on its own — so the result is not only
// deterministic but bit-identical to the reference's CPU function, and grad_points needs no zero-fill.
// Build: count entries per known point (int atomics), exclusive scan per cloud, fill the CSR lists (order
// inside a list is arbitrary), then every warp sorts its own list (<= 128 entries: bitonic sort in
// registers; longer lists — degenerate layers where most unknown points share a neighbour — are served
// by an index-ordered scan of the cloud's entries instead).
constexpr int kInvThreads = 256;
constexpr int kInvSortCap = 256;

__global__ void __launch_bounds__(kInvThreads)
inv_count_kernel(int n3, int m, long long total, const int* __restrict__ idx, int* __restrict__ cnt) {
    for (long long e = (long long)blockIdx.x * kInvThreads + threadIdx.x; e < total; e += (long long)gridDim.x * kInvThreads) {
        const long long cloud = e / n3;
        atomicAdd(cnt + cloud * (m + 1) + __ldg(idx + e), 1);
    }
}

// one CTA per cloud: off[i] = exclusive prefix of cnt[i], i = 0..m (off[m] = 3n); cur[i] = off[i]
__global__ void __launch_bounds__(1024)
inv_scan_kernel(int m, int* __restrict__ cnt_off, int* __restrict__ cur) {
    __shared__ int s_w[32];
    __shared__ int s_carry;
    int* __restrict__ c = cnt_off + (size_t)blockIdx.x * (m + 1);
    int* __restrict__ cu = cur + (size_t)blockIdx.x * m;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) s_carry = 0;
    __syncthreads();
    for (int base = 0; base <= m; base += 1024) {
        const int i = base + tid;
        const int v = (i < m) ? c[i] : 0;
        int incl = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int t = __shfl_up_sync(kFullMask, incl, o);
            if (lane >= o) incl += t;
        }
        if (lane == 31) s_w[warp] = incl;
        __syncthreads();
        int wv = s_w[lane], winc = wv;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int t = __shfl_up_sync(kFullMask, winc, o);
            if (lane >= o) winc += t;
        }
        const int carry = s_carry;
        const int excl = carry + __shfl_sync(kFullMask, winc - wv, warp) + incl - v;
        if (i <= m) c[i] = excl;
        if (i < m) cu[i] = excl;
        __syncthreads();
        if (tid == 1023) s_carry = excl + v;
        __syncthreads();
    }
}

__global__ void __launch_bounds__(kInvThreads)
inv_fill_kernel(int n3, int m, long long total, const int* __restrict__ idx, int* __restrict__ cur, int* __restrict__ entries) {
    for (long long e = (long long)blockIdx.x * kInvThreads + threadIdx.x; e < total; e += (long long)gridDim.x * kInvThreads) {
        const long long cloud = e / n3;
        const int pos = atomicAdd(cur + cloud * m + __ldg(idx + e), 1);
        entries[cloud * n3 + pos] = (int)(e - cloud * n3);
    }
}

// count + scan + fill of one cloud in ONE CTA, with the counters and cursors in shared memory (m <= 16000): the
// inverse index of a layer costs one launch instead of two memsets and three kernels.
constexpr int kInvBuildMaxM = 16000;
__global__ void __launch_bounds__(1024)
inv_build_kernel(int n3, int m, const int* __restrict__ idx, int* __restrict__ off, int* __restrict__ entries,
                 int* __restrict__ long_queue) {
    extern __shared__ int s_c[];  // [m + 1]: counts -> exclusive offsets (kept as the fill cursors)
    __shared__ int s_w[32];
    __shared__ int s_carry;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const long long cloud = blockIdx.x;
    const int* __restrict__ cidx = idx + cloud * n3;
    for (int i = tid; i <= m; i += 1024) s_c[i] = 0;
    if (tid == 0) {
        s_carry = 0;
        if (cloud == 0) long_queue[0] = 0;
    }
    __syncthreads();
    for (int e = tid; e < n3; e += 1024) atomicAdd(&s_c[__ldg(cidx + e)], 1);
    __syncthreads();
    int* __restrict__ o = off + cloud * (m + 1);
    for (int base = 0; base <= m; base += 1024) {
        const int i = base + tid;
        const int v = (i < m) ? s_c[i] : 0;
        int incl = v;
#pragma unroll
        for (int sft = 1; sft < 32; sft <<= 1) {
            const int t = __shfl_up_sync(kFullMask, incl, sft);
            if (lane >= sft) incl += t;
        }
        if (lane == 31) s_w[warp] = incl;
        __syncthreads();
        int wv = s_w[lane], winc = wv;
#pragma unroll
        for (int sft = 1; sft < 32; sft <<= 1) {
            const int t = __shfl_up_sync(kFullMask, winc, sft);
            if (lane >= sft) winc += t;
        }
        const int excl = s_carry + __shfl_sync(kFullMask, winc - wv, warp) + incl - v;
        if (i <= m) {
            o[i] = excl;
            s_c[i] = excl;
        }
        __syncthreads();
        if (tid == 1023) s_carry = excl + v;
        __syncthreads();
    }
    int* __restrict__ ent = entries + cloud * n3;
    for (int e = tid; e < n3; e += 1024) ent[atomicAdd(&s_c[__ldg(cidx + e)], 1)] = e;
}

// 4 consecutive entries / one entry of grad_out, widened exactly to float32 (DT = 0: float32 grad_out)
template <int DT>
__device__ __forceinline__ float4 ld_grad4(const feat_t<DT>* __restrict__ p) {
    if constexpr (DT == 0) {
        return __ldg(reinterpret_cast<const float4*>(p));
    } else {
        const uint2 u = __ldg(reinterpret_cast<const uint2*>(p));
        const float2 lo = h2_to_f2<DT>(u.x), hi = h2_to_f2<DT>(u.y);
        return make_float4(lo.x, lo.y, hi.x, hi.y);
    }
}
template <int DT>
__device__ __forceinline__ float ld_grad1(const feat_t<DT>* __restrict__ p) {
    if constexpr (DT == 0) return __ldg(p);
    else return h_to_f<DT>(__ldg(p));
}

// one warp per known point (b, i); lanes over channels (4 channels per lane when VEC).  Lists longer than kInvSortCap
// are queued for inv_long_kernel.  DT: grad_out's type (0 = float32); sums are float32 either way.
template <int DT, bool VEC>
__global__ void __launch_bounds__(kInvThreads)
inv_gather_kernel(int n, int c, int m, long long warps_total, const feat_t<DT>* __restrict__ grad_out,
                  const float* __restrict__ weight, const int* __restrict__ off, const int* __restrict__ entries,
                  float* __restrict__ grad_points, int* __restrict__ long_queue) {
    __shared__ int s_e[kInvThreads / 32][kInvSortCap];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const long long gw = ((long long)blockIdx.x * kInvThreads + threadIdx.x) >> 5;
    if (gw >= warps_total) return;
    const long long cloud = gw / m;
    const int i = (int)(gw - cloud * m);
    const int n3 = 3 * n;
    const int* __restrict__ o = off + cloud * (m + 1);
    const int beg = o[i], len = o[i + 1] - beg;
    if (len > kInvSortCap) {  // warp-uniform
        if (lane == 0) long_queue[1 + atomicAdd(long_queue, 1)] = (int)gw;  // the order of the queue does not matter
        return;
    }
    const feat_t<DT>* __restrict__ go = grad_out + (size_t)cloud * n * c;
    const float* __restrict__ wt = weight + (size_t)cloud * n3;
    float* __restrict__ gp = grad_points + ((size_t)cloud * m + i) * c;
    {
        int key[8];
#pragma unroll
        for (int q = 0; q < 8; ++q) key[q] = (32 * q + lane < len) ? __ldg(entries + cloud * n3 + beg + 32 * q + lane) : 0x7fffffff;
        const int nreg = (len + 31) >> 5;
        if (nreg <= 1) bitonic_sort_keys<1, 8>(key, lane);
        else if (nreg == 2) bitonic_sort_keys<2, 8>(key, lane);
        else if (nreg <= 4) bitonic_sort_keys<4, 8>(key, lane);
        else bitonic_sort_keys<8, 8>(key, lane);
#pragma unroll
        for (int q = 0; q < 8; ++q)
            if (32 * q + lane < len) s_e[wib][32 * q + lane] = key[q];
        __syncwarp();
    }
    constexpr int W = VEC ? 4 : 1;
    for (int l0 = 0; l0 < c; l0 += 32 * W) {  // 128 (VEC) or 32 channels per pass
        const int l = l0 + lane * W;
        if (l >= c) continue;
        float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
#pragma unroll 4
        for (int sidx = 0; sidx < len; ++sidx) {
            const int e = s_e[wib][sidx];
            const float w = __ldg(wt + e);
            const feat_t<DT>* __restrict__ src = go + (size_t)(e / 3) * c + l;
            if (VEC) {
                const float4 g = ld_grad4<DT>(src);
                a0 = __fadd_rn(a0, __fmul_rn(g.x, w));
                a1 = __fadd_rn(a1, __fmul_rn(g.y, w));
                a2 = __fadd_rn(a2, __fmul_rn(g.z, w));
                a3 = __fadd_rn(a3, __fmul_rn(g.w, w));
            } else {
                a0 = __fadd_rn(a0, __fmul_rn(ld_grad1<DT>(src), w));
            }
        }
        if (VEC) *reinterpret_cast<float4*>(gp + l) = make_float4(a0, a1, a2, a3);
        else gp[l] = a0;
    }
}

// Long lists (most unknown points share a neighbour: coincident points, m < 3, ...): one CTA per list.  The
// cloud's 3n entries are cut into 8 consecutive pieces, one per warp; each warp walks its piece in index order
// (coalesced index loads + ballot), adds the entries that point at i in that order, and the 8 partial sums are
// combined in piece order — a fixed association, hence deterministic (it differs from one long sequential sum
// only in rounding; short lists, the normal case, are bit-identical to the reference's loop).
template <int DT, bool VEC>
__global__ void __launch_bounds__(kInvThreads)
inv_long_kernel(int n, int c, int m, const feat_t<DT>* __restrict__ grad_out, const int* __restrict__ idx,
                const float* __restrict__ weight, const int* __restrict__ long_queue, float* __restrict__ grad_points) {
    constexpr int NW = kInvThreads / 32;
    constexpr int W = VEC ? 4 : 1;
    __shared__ float s_part[NW][32 * W];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int nq = long_queue[0];
    const int n3 = 3 * n;
    const int piece = (n3 + NW - 1) / NW;
    for (int q = blockIdx.x; q < nq; q += gridDim.x) {
        const long long gw = long_queue[1 + q];
        const long long cloud = gw / m;
        const int i = (int)(gw - cloud * m);
        const feat_t<DT>* __restrict__ go = grad_out + (size_t)cloud * n * c;
        const float* __restrict__ wt = weight + (size_t)cloud * n3;
        const int* __restrict__ cidx = idx + cloud * n3;
        float* __restrict__ gp = grad_points + ((size_t)cloud * m + i) * c;
        const int e_lo = warp * piece, e_hi = min(n3, e_lo + piece);
        for (int l0 = 0; l0 < c; l0 += 32 * W) {
            const int l = l0 + lane * W;
            const bool act = l < c;
            float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
            for (int base = e_lo; base < e_hi; base += 32) {
                const int e = base + lane;
                unsigned hit = __ballot_sync(kFullMask, e < e_hi && __ldg(cidx + e) == i);
                while (hit) {  // up to 4 matching entries at a time: their rows are loaded together, then added in order
                    int ee[4];
                    float w[4];
                    float4 g[4];
#pragma unroll
                    for (int u = 0; u < 4; ++u) {
                        ee[u] = -1;
                        if (hit) {
                            ee[u] = base + __ffs(hit) - 1;
                            hit &= hit - 1;
                        }
                    }
#pragma unroll
                    for (int u = 0; u < 4; ++u) {
                        g[u] = make_float4(0.f, 0.f, 0.f, 0.f);
                        w[u] = 0.f;
                        if (ee[u] >= 0 && act) {
                            w[u] = __ldg(wt + ee[u]);
                            const feat_t<DT>* __restrict__ src = go + (size_t)(ee[u] / 3) * c + l;
                            if (VEC) g[u] = ld_grad4<DT>(src);
                            else g[u].x = ld_grad1<DT>(src);
                        }
                    }
#pragma unroll
                    for (int u = 0; u < 4; ++u) {
                        if (ee[u] >= 0 && act) {
                            a0 = __fadd_rn(a0, __fmul_rn(g[u].x, w[u]));
                            if (VEC) {
                                a1 = __fadd_rn(a1, __fmul_rn(g[u].y, w[u]));
                                a2 = __fadd_rn(a2, __fmul_rn(g[u].z, w[u]));
                                a3 = __fadd_rn(a3, __fmul_rn(g[u].w, w[u]));
                            }
                        }
                    }
                }
            }
            s_part[warp][lane * W] = a0;
            if (VEC) {
                s_part[warp][lane * W + 1] = a1;
                s_part[warp][lane * W + 2] = a2;
                s_part[warp][lane * W + 3] = a3;
            }
            __syncthreads();
            if (warp == 0 && act) {
#pragma unroll
                for (int u = 0; u < W; ++u) {
                    float t = s_part[0][lane * W + u];
#pragma unroll
                    for (int p = 1; p < NW; ++p) t = __fadd_rn(t, s_part[p][lane * W + u]);
                    gp[l + u] = t;
                }
            }
            __syncthreads();
        }
    }
}

static unsigned it_grid(unsigned long long work_items, unsigned per_block) {
    unsigned long long blocks = (work_items + per_block - 1) / per_block;
    const unsigned long long cap = 148ull * 64;
    if (blocks > cap) blocks = cap;
    if (blocks < 1) blocks = 1;
    return (unsigned)blocks;
}

static bool al16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

// ---- 16-bit features (pn2_*_h) -------------------------------------------------------------------
// three_interpolate: one thread per 8 output values (16-byte loads of each of the three rows) when c % 8 == 0 and the
// bases are 16-byte aligned, else one per value.  Values widened exactly, interp3 in float32, one rounding.
template <typename IndexT, int DT>
__global__ void __launch_bounds__(kItThreads)
three_interp_h_vec8_kernel(int m, int c8, IndexT rows_per_cloud, IndexT total_vec, const uint4* __restrict__ points,
                           const int* __restrict__ idx, const float* __restrict__ weight, uint4* __restrict__ out) {
    const IndexT stride = (IndexT)gridDim.x * kItThreads;
    for (IndexT v = (IndexT)blockIdx.x * kItThreads + threadIdx.x; v < total_vec; v += stride) {
        const IndexT row = v / (IndexT)c8;
        const int l = (int)(v - row * (IndexT)c8);
        const IndexT cloud = row / rows_per_cloud;
        const int i1 = __ldg(idx + (size_t)row * 3 + 0), i2 = __ldg(idx + (size_t)row * 3 + 1), i3 = __ldg(idx + (size_t)row * 3 + 2);
        const float w1 = __ldg(weight + (size_t)row * 3 + 0), w2 = __ldg(weight + (size_t)row * 3 + 1),
                    w3 = __ldg(weight + (size_t)row * 3 + 2);
        const uint4* pb = points + (size_t)cloud * m * c8 + l;
        const uint4 a = __ldg(pb + (size_t)i1 * c8), b = __ldg(pb + (size_t)i2 * c8), c = __ldg(pb + (size_t)i3 * c8);
        __stcs(out + v, interp3_h8<DT>(a, b, c, w1, w2, w3));
    }
}

template <typename IndexT, int DT>
__global__ void __launch_bounds__(kItThreads)
three_interp_h_scalar_kernel(int m, int c, IndexT rows_per_cloud, IndexT total, const unsigned short* __restrict__ points,
                             const int* __restrict__ idx, const float* __restrict__ weight, unsigned short* __restrict__ out) {
    const IndexT stride = (IndexT)gridDim.x * kItThreads;
    for (IndexT e = (IndexT)blockIdx.x * kItThreads + threadIdx.x; e < total; e += stride) {
        const IndexT row = e / (IndexT)c;
        const int l = (int)(e - row * (IndexT)c);
        const IndexT cloud = row / rows_per_cloud;
        const int* ii = idx + (size_t)row * 3;
        const float* w = weight + (size_t)row * 3;
        const unsigned short* pb = points + (size_t)cloud * m * c + l;
        out[e] = f_to_h<DT>(interp3(h_to_f<DT>(__ldg(pb + (size_t)__ldg(ii + 0) * c)), h_to_f<DT>(__ldg(pb + (size_t)__ldg(ii + 1) * c)),
                                    h_to_f<DT>(__ldg(pb + (size_t)__ldg(ii + 2) * c)), __ldg(w + 0), __ldg(w + 1), __ldg(w + 2)));
    }
}

template <int DT>
static int three_interp_h(int b, int m, int c, int n, const unsigned short* points, const int* idx, const float* weight,
                          unsigned short* out, cudaStream_t st) {
    const unsigned long long total = (unsigned long long)b * n * c;
    if (c % 8 == 0 && al16(points) && al16(out)) {
        const unsigned long long tv = total / 8;
        const unsigned grid = it_grid(tv, kItThreads);
        const uint4* p8 = reinterpret_cast<const uint4*>(points);
        uint4* o8 = reinterpret_cast<uint4*>(out);
        if (tv < (1ull << 31))
            three_interp_h_vec8_kernel<unsigned, DT><<<grid, kItThreads, 0, st>>>(m, c / 8, (unsigned)n, (unsigned)tv, p8, idx, weight, o8);
        else
            three_interp_h_vec8_kernel<unsigned long long, DT><<<grid, kItThreads, 0, st>>>(m, c / 8, (unsigned long long)n, tv, p8, idx, weight, o8);
    } else {
        const unsigned grid = it_grid(total, kItThreads);
        if (total < (1ull << 31))
            three_interp_h_scalar_kernel<unsigned, DT><<<grid, kItThreads, 0, st>>>(m, c, (unsigned)n, (unsigned)total, points, idx, weight, out);
        else
            three_interp_h_scalar_kernel<unsigned long long, DT><<<grid, kItThreads, 0, st>>>(m, c, (unsigned long long)n, total, points, idx, weight, out);
    }
    return finish_launch();
}

// grad_points[b, idx[b,j,t], l] += grad_out[b,j,l] * weight[b,j,t] with a 16-bit grad_out, float atomics into float32.
// VEC: 4 channels per thread (8-byte loads, red.global.add.v4.f32), c % 4 == 0.
template <typename IndexT, int DT, bool VEC>
__global__ void __launch_bounds__(kItThreads)
three_interp_grad_h_kernel(int m, int c, IndexT rows_per_cloud, IndexT total, const unsigned short* __restrict__ grad_out,
                           const int* __restrict__ idx, const float* __restrict__ weight, float* __restrict__ grad_points) {
    constexpr int W = VEC ? 4 : 1;
    const int cw = c / W;
    const IndexT stride = (IndexT)gridDim.x * kItThreads;
    for (IndexT e = (IndexT)blockIdx.x * kItThreads + threadIdx.x; e < total; e += stride) {
        const IndexT row = e / (IndexT)cw;
        const int l = (int)(e - row * (IndexT)cw) * W;
        const IndexT cloud = row / rows_per_cloud;
        float4 g;
        if (VEC) {
            const uint2 u = __ldcs(reinterpret_cast<const uint2*>(grad_out) + e);
            const float2 lo = h2_to_f2<DT>(u.x), hi = h2_to_f2<DT>(u.y);
            g = make_float4(lo.x, lo.y, hi.x, hi.y);
        } else {
            g.x = h_to_f<DT>(__ldcs(grad_out + e));
        }
        float* gb = grad_points + (size_t)cloud * m * c + l;
#pragma unroll
        for (int t = 0; t < 3; ++t) {
            const int i = __ldg(idx + (size_t)row * 3 + t);
            const float w = __ldg(weight + (size_t)row * 3 + t);
            if (VEC)
                atomicAdd(reinterpret_cast<float4*>(gb + (size_t)i * c),
                          make_float4(__fmul_rn(g.x, w), __fmul_rn(g.y, w), __fmul_rn(g.z, w), __fmul_rn(g.w, w)));
            else
                atomicAdd(gb + (size_t)i * c, __fmul_rn(g.x, w));
        }
    }
}

template <int DT>
static int three_interp_grad_h(int b, int n, int c, int m, const unsigned short* grad_out, const int* idx, const float* weight,
                               float* grad_points, cudaStream_t st) {
    const unsigned long long total = (unsigned long long)b * n * c;
    if (c % 4 == 0 && (reinterpret_cast<uintptr_t>(grad_out) & 7u) == 0 && al16(grad_points)) {
        const unsigned long long tv = total / 4;
        const unsigned grid = it_grid(tv, kItThreads);
        if (tv < (1ull << 31))
            three_interp_grad_h_kernel<unsigned, DT, true><<<grid, kItThreads, 0, st>>>(m, c, (unsigned)n, (unsigned)tv, grad_out, idx, weight, grad_points);
        else
            three_interp_grad_h_kernel<unsigned long long, DT, true><<<grid, kItThreads, 0, st>>>(m, c, (unsigned long long)n, tv, grad_out, idx, weight, grad_points);
    } else {
        const unsigned grid = it_grid(total, kItThreads);
        if (total < (1ull << 31))
            three_interp_grad_h_kernel<unsigned, DT, false><<<grid, kItThreads, 0, st>>>(m, c, (unsigned)n, (unsigned)total, grad_out, idx, weight, grad_points);
        else
            three_interp_grad_h_kernel<unsigned long long, DT, false><<<grid, kItThreads, 0, st>>>(m, c, (unsigned long long)n, total, grad_out, idx, weight, grad_points);
    }
    return finish_launch();
}

// pn2_three_interpolate_grad_det for a float32 (DT = 0) or 16-bit grad_out: the inverse index does not depend on it
template <int DT>
static int three_interp_grad_det(int b, int n, int c, int m, const feat_t<DT>* grad_out, const int* idx, const float* weight,
                                 float* grad_points, void* workspace, size_t workspace_bytes, void* stream) {
    if (b < 0 || m <= 0 || c < 0 || n < 0) return (int)cudaErrorInvalidValue;
    if ((unsigned long long)b * m * c == 0) return 0;
    if (!grad_points) return (int)cudaErrorInvalidValue;
    cudaStream_t st = as_stream(stream);
    if (n == 0) return (int)cudaMemsetAsync(grad_points, 0, sizeof(float) * (size_t)b * m * c, st);
    if (!grad_out || !idx || !weight || !workspace) return (int)cudaErrorInvalidValue;
    if (workspace_bytes < ::pn2_three_interpolate_grad_det_workspace_bytes(b, n, m) || (long long)n * 3 > 0x7fffffffLL)
        return (int)cudaErrorInvalidValue;
    int* off = static_cast<int*>(workspace);
    int* cur = off + (size_t)b * (m + 1);
    int* entries = cur + (size_t)b * m;
    int* long_queue = entries + (size_t)b * 3 * (size_t)n;  // [0] = count, then (cloud * m + i) of every list > kInvSortCap
    int launches = 2;
    if (m <= kInvBuildMaxM) {
        static std::atomic<unsigned long long> attr_done{0ull};
        int dev = 0;
        cudaError_t e = cudaGetDevice(&dev);
        if (e != cudaSuccess) return (int)e;
        if (dev >= 64 || !(attr_done.load(std::memory_order_acquire) & (1ull << dev))) {
            e = cudaFuncSetAttribute(inv_build_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(int) * (kInvBuildMaxM + 1));
            if (e != cudaSuccess) return (int)e;
            if (dev < 64) attr_done.fetch_or(1ull << dev, std::memory_order_release);
        }
        inv_build_kernel<<<b, 1024, sizeof(int) * (size_t)(m + 1), st>>>(3 * n, m, idx, off, entries, long_queue);
        launches += 1;
    } else {
        cudaError_t e = cudaMemsetAsync(off, 0, sizeof(int) * (size_t)b * (m + 1), st);
        if (e == cudaSuccess) e = cudaMemsetAsync(long_queue, 0, sizeof(int), st);
        if (e != cudaSuccess) return (int)e;
        const long long total = (long long)b * n * 3;
        const unsigned g1 = it_grid((unsigned long long)total, kInvThreads);
        inv_count_kernel<<<g1, kInvThreads, 0, st>>>(3 * n, m, total, idx, off);
        inv_scan_kernel<<<b, 1024, 0, st>>>(m, off, cur);
        inv_fill_kernel<<<g1, kInvThreads, 0, st>>>(3 * n, m, total, idx, cur, entries);
        launches += 3;
    }
    const long long warps = (long long)b * m;
    const unsigned long long blocks = ((unsigned long long)warps * 32 + kInvThreads - 1) / kInvThreads;
    if (blocks > 0x7fffffffull) return (int)cudaErrorInvalidValue;
    // long lists: a fixed grid walks the queue (usually empty: the CTAs read one word and leave)
    const unsigned long_grid = 148u * 2u;
    // VEC: 4 channels per lane (16-byte float32 / 8-byte 16-bit loads)
    const uintptr_t galign = DT == 0 ? 15u : 7u;
    if (c % 4 == 0 && (reinterpret_cast<uintptr_t>(grad_out) & galign) == 0 && al16(grad_points)) {
        inv_gather_kernel<DT, true><<<(unsigned)blocks, kInvThreads, 0, st>>>(n, c, m, warps, grad_out, weight, off, entries, grad_points, long_queue);
        inv_long_kernel<DT, true><<<long_grid, kInvThreads, 0, st>>>(n, c, m, grad_out, idx, weight, long_queue, grad_points);
    } else {
        inv_gather_kernel<DT, false><<<(unsigned)blocks, kInvThreads, 0, st>>>(n, c, m, warps, grad_out, weight, off, entries, grad_points, long_queue);
        inv_long_kernel<DT, false><<<long_grid, kInvThreads, 0, st>>>(n, c, m, grad_out, idx, weight, long_queue, grad_points);
    }
    count_launch(launches - 1);
    return finish_launch();
}


}  // namespace pn2

extern "C" {

int pn2_three_nn(int b, int n, int m, const float* xyz1, const float* xyz2, float* dist, int* idx, void* stream) {
    using namespace pn2;
    if (b < 0 || n < 0 || m < 0) return (int)cudaErrorInvalidValue;
    if (b == 0 || n == 0) return 0;
    if (!xyz1 || (m > 0 && !xyz2) || !dist || !idx) return (int)cudaErrorInvalidValue;
    if (b > 65535) return (int)cudaErrorInvalidValue;
    dim3 grid((n + kNnThreads - 1) / kNnThreads, b, 1);
    three_nn_kernel<<<grid, kNnThreads, 0, as_stream(stream)>>>(n, m, xyz1, xyz2, dist, idx);
    return finish_launch();
}

int pn2_three_interpolate(int b, int m, int c, int n, const float* points, const int* idx, const float* weight,
                          float* out, void* stream) {
    using namespace pn2;
    if (b < 0 || m <= 0 || c < 0 || n < 0) return (int)cudaErrorInvalidValue;
    const unsigned long long total = (unsigned long long)b * n * c;
    if (total == 0) return 0;
    if (!points || !idx || !weight || !out) return (int)cudaErrorInvalidValue;
    cudaStream_t st = as_stream(stream);
    if (c % 4 == 0 && al16(points) && al16(out)) {
        const unsigned long long tv = total / 4;
        const unsigned grid = it_grid(tv, kItThreads);
        if (tv < (1ull << 31))
            three_interp_vec4_kernel<unsigned, 1><<<grid, kItThreads, 0, st>>>(m, c / 4, (unsigned)n, (unsigned)tv, (const float4*)points, idx, weight, (float4*)out);
        else
            three_interp_vec4_kernel<unsigned long long, 1><<<grid, kItThreads, 0, st>>>(m, c / 4, (unsigned long long)n, tv, (const float4*)points, idx, weight, (float4*)out);
    } else {
        const unsigned grid = it_grid(total, kItThreads);
        if (total < (1ull << 31))
            three_interp_scalar_kernel<unsigned><<<grid, kItThreads, 0, st>>>(m, c, (unsigned)n, (unsigned)total, points, idx, weight, out);
        else
            three_interp_scalar_kernel<unsigned long long><<<grid, kItThreads, 0, st>>>(m, c, (unsigned long long)n, total, points, idx, weight, out);
    }
    return finish_launch();
}

int pn2_three_interpolate_grad(int b, int n, int c, int m, const float* grad_out, const int* idx, const float* weight,
                               float* grad_points, void* stream) {
    using namespace pn2;
    if (b < 0 || m <= 0 || c < 0 || n < 0) return (int)cudaErrorInvalidValue;
    const unsigned long long total = (unsigned long long)b * n * c;
    if (total == 0) return 0;
    if (!grad_out || !idx || !weight || !grad_points) return (int)cudaErrorInvalidValue;
    cudaStream_t st = as_stream(stream);
    if (c % 4 == 0 && al16(grad_out) && al16(grad_points)) {
        const unsigned long long tv = total / 4;
        const unsigned grid = it_grid(tv, kItThreads);
        if (tv < (1ull << 31))
            three_interp_grad_vec4_kernel<unsigned><<<grid, kItThreads, 0, st>>>(m, c / 4, (unsigned)n, (unsigned)tv, (const float4*)grad_out, idx, weight, (float4*)grad_points);
        else
            three_interp_grad_vec4_kernel<unsigned long long><<<grid, kItThreads, 0, st>>>(m, c / 4, (unsigned long long)n, tv, (const float4*)grad_out, idx, weight, (float4*)grad_points);
    } else {
        const unsigned grid = it_grid(total, kItThreads);
        if (total < (1ull << 31))
            three_interp_grad_scalar_kernel<unsigned><<<grid, kItThreads, 0, st>>>(m, c, (unsigned)n, (unsigned)total, grad_out, idx, weight, grad_points);
        else
            three_interp_grad_scalar_kernel<unsigned long long><<<grid, kItThreads, 0, st>>>(m, c, (unsigned long long)n, total, grad_out, idx, weight, grad_points);
    }
    return finish_launch();
}

int pn2_three_nn_interpolate(int b, int n, int m, int c, const float* xyz1, const float* xyz2, const float* points2,
                             float* out, float* dist, int* idx, float* weight, void* stream) {
    using namespace pn2;
    if (b < 0 || n < 0 || m <= 0 || c < 0) return (int)cudaErrorInvalidValue;
    if (b == 0 || n == 0) return 0;
    if (!xyz1 || !xyz2 || (c > 0 && (!points2 || !out))) return (int)cudaErrorInvalidValue;
    if (b > 65535) return (int)cudaErrorInvalidValue;
    return fp_front_dispatch<0>(b, n, m, c, 0, xyz1, xyz2, nullptr, points2, c > 0 ? out : nullptr, dist, idx, weight, as_stream(stream));
}

int pn2_fp_interpolate_concat(int b, int n, int m, int c2, int c1, const float* xyz1, const float* xyz2, const float* points1,
                              const float* points2, float* out, void* stream) {
    using namespace pn2;
    if (b < 0 || n < 0 || m <= 0 || c2 <= 0 || c1 < 0) return (int)cudaErrorInvalidValue;
    if (b == 0 || n == 0) return 0;
    if (!xyz1 || !xyz2 || !points2 || !out || (c1 > 0 && !points1)) return (int)cudaErrorInvalidValue;
    if (b > 65535) return (int)cudaErrorInvalidValue;
    return fp_front_dispatch<0>(b, n, m, c2, c1, xyz1, xyz2, c1 > 0 ? points1 : nullptr, points2, out, nullptr, nullptr, nullptr,
                             as_stream(stream));
}

size_t pn2_three_interpolate_grad_det_workspace_bytes(int b, int n, int m) {
    if (b <= 0 || n <= 0 || m <= 0) return 0;
    // offsets (b, m+1) + cursors (b, m) + entries (b, 3n) + queue of long lists (1 + b * ceil(3n / (cap+1))), ints
    const size_t longs = (size_t)b * ((3 * (size_t)n) / (pn2::kInvSortCap + 1) + 1);
    return sizeof(int) * ((size_t)b * (m + 1) + (size_t)b * m + (size_t)b * 3 * (size_t)n + 1 + longs);
}

int pn2_three_interpolate_grad_det(int b, int n, int c, int m, const float* grad_out, const int* idx, const float* weight,
                                   float* grad_points, void* workspace, size_t workspace_bytes, void* stream) {
    return pn2::three_interp_grad_det<0>(b, n, c, m, grad_out, idx, weight, grad_points, workspace, workspace_bytes, stream);
}

int pn2_three_interpolate_h(int dtype, int b, int m, int c, int n, const void* points, const int* idx, const float* weight,
                            void* out, void* stream) {
    using namespace pn2;
    if (!valid_half_dtype(dtype)) return (int)cudaErrorInvalidValue;
    if (b < 0 || m <= 0 || c < 0 || n < 0) return (int)cudaErrorInvalidValue;
    if ((unsigned long long)b * n * c == 0) return 0;
    if (!points || !idx || !weight || !out) return (int)cudaErrorInvalidValue;
    const unsigned short* p = static_cast<const unsigned short*>(points);
    unsigned short* o = static_cast<unsigned short*>(out);
    if (dtype == PN2_DTYPE_BF16) return three_interp_h<PN2_DTYPE_BF16>(b, m, c, n, p, idx, weight, o, as_stream(stream));
    return three_interp_h<PN2_DTYPE_F16>(b, m, c, n, p, idx, weight, o, as_stream(stream));
}

int pn2_three_interpolate_grad_h(int dtype, int b, int n, int c, int m, const void* grad_out, const int* idx,
                                 const float* weight, float* grad_points, void* stream) {
    using namespace pn2;
    if (!valid_half_dtype(dtype)) return (int)cudaErrorInvalidValue;
    if (b < 0 || m <= 0 || c < 0 || n < 0) return (int)cudaErrorInvalidValue;
    if ((unsigned long long)b * n * c == 0) return 0;
    if (!grad_out || !idx || !weight || !grad_points) return (int)cudaErrorInvalidValue;
    const unsigned short* g = static_cast<const unsigned short*>(grad_out);
    if (dtype == PN2_DTYPE_BF16) return three_interp_grad_h<PN2_DTYPE_BF16>(b, n, c, m, g, idx, weight, grad_points, as_stream(stream));
    return three_interp_grad_h<PN2_DTYPE_F16>(b, n, c, m, g, idx, weight, grad_points, as_stream(stream));
}

int pn2_three_interpolate_grad_det_h(int dtype, int b, int n, int c, int m, const void* grad_out, const int* idx,
                                     const float* weight, float* grad_points, void* workspace, size_t workspace_bytes,
                                     void* stream) {
    using namespace pn2;
    const unsigned short* g = static_cast<const unsigned short*>(grad_out);
    if (dtype == PN2_DTYPE_BF16)
        return three_interp_grad_det<PN2_DTYPE_BF16>(b, n, c, m, g, idx, weight, grad_points, workspace, workspace_bytes, stream);
    if (dtype == PN2_DTYPE_F16)
        return three_interp_grad_det<PN2_DTYPE_F16>(b, n, c, m, g, idx, weight, grad_points, workspace, workspace_bytes, stream);
    return (int)cudaErrorInvalidValue;
}

int pn2_three_nn_interpolate_h(int dtype, int b, int n, int m, int c, const float* xyz1, const float* xyz2, const void* points2,
                               void* out, float* dist, int* idx, float* weight, void* stream) {
    using namespace pn2;
    if (!valid_half_dtype(dtype)) return (int)cudaErrorInvalidValue;
    if (b < 0 || n < 0 || m <= 0 || c < 0) return (int)cudaErrorInvalidValue;
    if (b == 0 || n == 0) return 0;
    if (!xyz1 || !xyz2 || (c > 0 && (!points2 || !out))) return (int)cudaErrorInvalidValue;
    if (b > 65535) return (int)cudaErrorInvalidValue;
    const unsigned short* p2 = static_cast<const unsigned short*>(points2);
    unsigned short* o = c > 0 ? static_cast<unsigned short*>(out) : nullptr;
    if (dtype == PN2_DTYPE_BF16)
        return fp_front_dispatch<PN2_DTYPE_BF16>(b, n, m, c, 0, xyz1, xyz2, nullptr, p2, o, dist, idx, weight, as_stream(stream));
    return fp_front_dispatch<PN2_DTYPE_F16>(b, n, m, c, 0, xyz1, xyz2, nullptr, p2, o, dist, idx, weight, as_stream(stream));
}

int pn2_fp_interpolate_concat_h(int dtype, int b, int n, int m, int c2, int c1, const float* xyz1, const float* xyz2,
                                const void* points1, const void* points2, void* out, void* stream) {
    using namespace pn2;
    if (!valid_half_dtype(dtype)) return (int)cudaErrorInvalidValue;
    if (b < 0 || n < 0 || m <= 0 || c2 <= 0 || c1 < 0) return (int)cudaErrorInvalidValue;
    if (b == 0 || n == 0) return 0;
    if (!xyz1 || !xyz2 || !points2 || !out || (c1 > 0 && !points1)) return (int)cudaErrorInvalidValue;
    if (b > 65535) return (int)cudaErrorInvalidValue;
    const unsigned short* p1 = c1 > 0 ? static_cast<const unsigned short*>(points1) : nullptr;
    const unsigned short* p2 = static_cast<const unsigned short*>(points2);
    unsigned short* o = static_cast<unsigned short*>(out);
    if (dtype == PN2_DTYPE_BF16)
        return fp_front_dispatch<PN2_DTYPE_BF16>(b, n, m, c2, c1, xyz1, xyz2, p1, p2, o, nullptr, nullptr, nullptr, as_stream(stream));
    return fp_front_dispatch<PN2_DTYPE_F16>(b, n, m, c2, c1, xyz1, xyz2, p1, p2, o, nullptr, nullptr, nullptr, as_stream(stream));
}

}  // extern "C"
