// pm_common.cuh — shared helpers for libplatymatch_b200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <map>
#include <mutex>
#include "../../include/platymatch_b200.h"

void pm_set_error(const char *fmt, ...);
void pm_count_launches(int n);

#define PM_CUDA_TRY(expr)                                                                     \
    do {                                                                                      \
        cudaError_t _e = (expr);                                                              \
        if (_e != cudaSuccess) {                                                              \
            pm_set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #expr, cudaGetErrorString(_e)); \
            return PM_ERR_CUDA;                                                               \
        }                                                                                     \
    } while (0)

#define PM_LAUNCH_CHECK_N(n)                                                                   \
    do {                                                                                      \
        pm_count_launches(n);                                                                 \
        cudaError_t _e = cudaGetLastError();                                                  \
        if (_e != cudaSuccess) {                                                              \
            pm_set_error("%s:%d: kernel launch -> %s", __FILE__, __LINE__, cudaGetErrorString(_e)); \
            return PM_ERR_CUDA;                                                               \
        }                                                                                     \
    } while (0)

#define PM_LAUNCH_CHECK() PM_LAUNCH_CHECK_N(1)

// Refuses an argument in the name of the entry point fn (host helpers take their entry point's name)
#define PM_REQUIRE_AS(fn, cond, msg)                                           \
    do {                                                                       \
        if (!(cond)) {                                                         \
            pm_set_error("%s: invalid argument: %s", fn, msg);                \
            return PM_ERR_INVALID_ARGUMENT;                                    \
        }                                                                      \
    } while (0)

#define PM_REQUIRE(cond, msg) PM_REQUIRE_AS(__func__, cond, msg)

static inline cudaStream_t pm_stream(void *s) { return reinterpret_cast<cudaStream_t>(s); }

// Two byte ranges overlap (sizes up to 2^64 and beyond, no wrap-around)
static inline bool pm_ranges_overlap(const void *a, unsigned __int128 abytes, const void *b, unsigned __int128 bbytes) {
    const unsigned __int128 a0 = (uintptr_t)a, b0 = (uintptr_t)b;
    return !(a0 + abytes <= b0 || b0 + bbytes <= a0);
}

// A launch of `tiles` CTAs in a 1-D grid (at most 2^31 - 1); fn's `what` (its output / volume) is nz x ny x nx.
static inline int pm_check_grid_1d(const char *fn, const char *what, unsigned long long tiles, int nz, int ny, int nx) {
    if (tiles <= 0x7fffffffull) return PM_OK;
    pm_set_error("%s: %s of %d x %d x %d needs more than 2^31 - 1 CTAs", fn, what, nz, ny, nx);
    return PM_ERR_UNSUPPORTED;
}

// CTAs of a grid-stride streaming kernel over `want` CTAs of work: ONE wave of resident CTAs at most (SM count x the
// kernel's occupancy at `threads` per CTA), so that no second wave starts ragged.  The occupancy is queried once per
// (kernel, device).
static inline int pm_resident_wave(const void *kernel, int threads, int dev, int sms, size_t want, int *blocks) {
    static std::mutex mu;
    static std::map<std::pair<const void *, int>, int> occupancy;
    std::lock_guard<std::mutex> g(mu);
    int &occ = occupancy[{kernel, dev}];
    if (occ < 1) {
        PM_CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kernel, threads, 0));
        occ = occ < 1 ? 1 : occ;
    }
    *blocks = (int)(want < (size_t)sms * occ ? (want ? want : 1) : (size_t)sms * occ);
    return PM_OK;
}

// Volumes of the label and resample entry points.  dtype codes: PM_LABEL_I32 (int32_t), PM_LABEL_U16 (uint16_t) and,
// for the resample entry points (F32), PM_RESAMPLE_F32 (float).
static inline bool pm_volume_dtype_ok(int dtype, bool f32) {
    return dtype == PM_LABEL_I32 || dtype == PM_LABEL_U16 || (f32 && dtype == PM_RESAMPLE_F32);
}

// f(T{}) with T the element type of `dtype`, a code the entry point has accepted (pm_volume_dtype_ok)
template <bool F32, typename F> static inline int pm_volume_dispatch(int dtype, F &&f) {
    if constexpr (F32) {
        if (dtype == PM_RESAMPLE_F32) return f(float{});
    }
    return dtype == PM_LABEL_I32 ? f(int32_t{}) : f(uint16_t{});
}

// src [sz][sy][sx] and dst [dz][dy][dx] of the resample entry point fn, elements of an accepted `dtype`: every extent
// >= 1, each volume below 2^63 bytes, the two disjoint (in-place is not supported).  dst_bytes = the size of dst.
static inline int pm_check_volume_pair(const char *fn, int dtype, const void *src, int sz, int sy, int sx,
                                       const void *dst, int dz, int dy, int dx, unsigned __int128 &dst_bytes) {
    PM_REQUIRE_AS(fn, sz >= 1 && sy >= 1 && sx >= 1 && dz >= 1 && dy >= 1 && dx >= 1, "every extent must be >= 1");
    const unsigned __int128 es = dtype == PM_LABEL_U16 ? 2 : 4;
    const unsigned __int128 src_bytes = (unsigned __int128)sz * sy * sx * es;
    dst_bytes = (unsigned __int128)dz * dy * dx * es;
    PM_REQUIRE_AS(fn, src_bytes < ((unsigned __int128)1 << 63) && dst_bytes < ((unsigned __int128)1 << 63),
                  "volume too large");
    PM_REQUIRE_AS(fn, !pm_ranges_overlap(src, src_bytes, dst, dst_bytes),
                  "src and dst overlap (in-place is not supported)");
    return PM_OK;
}

__device__ __forceinline__ double pm_warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// Block-wide float64 sum (all threads get the result).  blockDim.x multiple of 32, <= 1024.
__device__ __forceinline__ double pm_block_sum(double v, double *smem32) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
    v = pm_warp_sum(v);
    __syncthreads();
    if (lane == 0) smem32[warp] = v;
    __syncthreads();
    double r = (lane < nw) ? smem32[lane] : 0.0;
    r = pm_warp_sum(r);
    return r;
}

#include "pm_linalg.cuh"   // pm_solve_right_4x4, pm_jacobi_sym4, pm_affine_from_normal_eq, pm_similar_from_moments
