// pn2_common.cuh — shared device/host helpers for libpn2_b200 (sm_100a only).
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <type_traits>

#include "pn2_api.h"

namespace pn2 {

constexpr unsigned kFullMask = 0xffffffffu;

// ---- launch accounting (pn2_launch_count) --------------------------------------------------
extern unsigned long long g_launch_count;
inline void count_launch(int k = 1) { __atomic_fetch_add(&g_launch_count, (unsigned long long)k, __ATOMIC_RELAXED); }

inline int finish_launch() {
    count_launch();
    return (int)cudaGetLastError();
}

inline cudaStream_t as_stream(void* s) { return reinterpret_cast<cudaStream_t>(s); }

inline unsigned ceil_div_u(unsigned long long a, unsigned long long b) { return (unsigned)((a + b - 1) / b); }

// ---- arithmetic contracts --------------------------------------------------------------------
// Squared distance exactly as nvcc contracts the reference's FPS and ball-query source
// (tf_sampling_g.cu:142, tf_grouping_g.cu:24; SASS: FMUL dy*dy, FFMA dx, FFMA dz).  Written with
// explicit round-to-nearest intrinsics so no compiler version or surrounding code can change it.
__device__ __forceinline__ float d2_fma_pattern(float ax, float ay, float az, float bx, float by, float bz) {
    const float dx = __fsub_rn(ax, bx), dy = __fsub_rn(ay, by), dz = __fsub_rn(az, bz);
    return __fmaf_rn(dz, dz, __fmaf_rn(dx, dx, __fmul_rn(dy, dy)));
}

// Squared distance exactly as x86-64 g++ -O2 (no FMA) evaluates threenn_cpu's expression
// (tf_interpolate.cpp:73): ((dx*dx + dy*dy) + dz*dz), each operation rounded on its own.
__device__ __forceinline__ float d2_nofma(float ax, float ay, float az, float bx, float by, float bz) {
    const float dx = __fsub_rn(ax, bx), dy = __fsub_rn(ay, by), dz = __fsub_rn(az, bz);
    return __fadd_rn(__fadd_rn(__fmul_rn(dx, dx), __fmul_rn(dy, dy)), __fmul_rn(dz, dz));
}

// ---- warp helpers ----------------------------------------------------------------------------
// Batch-level rule of the uniform-grid ball query, evaluated identically by the grid kernel and by
// the brute-force kernel (each warp on its own, no barrier): the two kernels run back to back on one
// stream, so splitting a batch between them only pays when the grid serves a fair share of it
// (measured: 10 of 32 clouds pays, 2 of 32 costs 20 us).  `flags` is
// the per-cloud flag word written by bq_grid_build_kernel, one every `stride` ints; batches larger
// than 1024 clouds are judged on their first 1024.
__device__ __forceinline__ bool batch_uses_grid(const int* __restrict__ flags, size_t stride, int b) {
    const int lane = threadIdx.x & 31;
    const int bb = b < 1024 ? b : 1024;
    int cnt = 0;
    for (int c = lane; c < bb; c += 32) cnt += (__ldg(flags + (size_t)c * stride) != 0) ? 1 : 0;
    cnt = __reduce_add_sync(kFullMask, cnt);
    return 4 * cnt >= bb;
}

__device__ __forceinline__ unsigned warp_max_u32(unsigned v) { return __reduce_max_sync(kFullMask, v); }

// Lexicographic max of (hi, lo) pairs over the warp; every lane gets the result.
__device__ __forceinline__ void warp_max_pair(unsigned& hi, unsigned& lo) {
    const unsigned mh = warp_max_u32(hi);
    const unsigned ml = warp_max_u32(hi == mh ? lo : 0u);
    hi = mh;
    lo = ml;
}

// Ascending bitonic sort of 32*K ints held K per lane (element i = register i/32 of lane i%32; K <= KMAX, a power of 2).
template <int K, int KMAX>
__device__ __forceinline__ void bitonic_sort_keys(int (&key)[KMAX], int lane) {
#pragma unroll
    for (int size = 2; size <= 32 * K; size <<= 1) {
#pragma unroll
        for (int stride = size >> 1; stride > 0; stride >>= 1) {
            if (stride >= 32) {  // partner in the same lane, another register
                const int js = stride >> 5;
#pragma unroll
                for (int j = 0; j < K; ++j) {
                    if ((j & js) == 0) {
                        const bool up = (((32 * j) & size) == 0);  // lane bits are below 32 <= stride < size: direction depends on j only
                        const int a = key[j], b = key[j | js];
                        const bool sw = up ? (a > b) : (a < b);
                        key[j] = sw ? b : a;
                        key[j | js] = sw ? a : b;
                    }
                }
            } else {
#pragma unroll
                for (int j = 0; j < K; ++j) {
                    const int i = 32 * j + lane;
                    const int other = __shfl_xor_sync(kFullMask, key[j], stride);
                    const bool up = ((i & size) == 0), lower = ((lane & stride) == 0);
                    // the lower element of an ascending pair keeps the minimum
                    key[j] = (up == lower) ? min(key[j], other) : max(key[j], other);
                }
            }
        }
    }
}

// brute-force ball query launcher (ball_query.cu); clouds whose grid_params[cloud*grid_stride] != 0
// are skipped (they are served by the uniform-grid kernels of ball_query_grid.cu)
int launch_ball_query_brute(int b, int n, int m, float thr, int nsample, const float* xyz1, const float* xyz2,
                            int* idx, int* pts_cnt, const int* grid_params, int grid_stride, cudaStream_t st);

// farthest point sampling dispatch (fps.cu), shared with the fused set-abstraction layer (sa_fused.cu).
// sentinel != 0: single-CTA plans only (ask fps_single_cta first) — the kernel pre-fills `out` with -1 and
// signals programmatic launch completion so that a dependent grid can consume the picks as they appear.
int fps_dispatch(int b, int n, int m, const float* inp, float* temp, int* out, float* new_xyz, int sentinel, cudaStream_t st);
bool fps_single_cta(int b, int n);
size_t fps_scratch_bytes(int b, int n);

// ---- 16-bit features (the pn2_*_h entry points) -------------------------------------------------
// DT = 0 for float32, PN2_DTYPE_BF16 or PN2_DTYPE_F16; 16-bit values travel as their bit patterns.
template <int DT>
using feat_t = std::conditional_t<DT == 0, float, unsigned short>;

inline bool valid_half_dtype(int dt) { return dt == PN2_DTYPE_BF16 || dt == PN2_DTYPE_F16; }

// exact widening
template <int DT>
__device__ __forceinline__ float h_to_f(unsigned short u) {
    if (DT == PN2_DTYPE_BF16) return __uint_as_float((unsigned)u << 16);
    return __half2float(__ushort_as_half(u));
}
// one rounding, to nearest-even
template <int DT>
__device__ __forceinline__ unsigned short f_to_h(float f) {
    if (DT == PN2_DTYPE_BF16) return __bfloat16_as_ushort(__float2bfloat16_rn(f));
    return __half_as_ushort(__float2half_rn(f));
}
// a word of two 16-bit values: element 2i is the low half
template <int DT>
__device__ __forceinline__ float2 h2_to_f2(unsigned w) {
    return make_float2(h_to_f<DT>((unsigned short)(w & 0xffffu)), h_to_f<DT>((unsigned short)(w >> 16)));
}
template <int DT>
__device__ __forceinline__ unsigned f2_to_h2(float lo, float hi) {
    return (unsigned)f_to_h<DT>(lo) | ((unsigned)f_to_h<DT>(hi) << 16);
}

// ---- streaming memory ops ---------------------------------------------------------------------
__device__ __forceinline__ void st_stream_f4(float4* p, float4 v) { __stcs(p, v); }
__device__ __forceinline__ void st_stream_i4(int4* p, int4 v) { __stcs(p, v); }

}  // namespace pn2
