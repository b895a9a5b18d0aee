// pm_sample.cuh — the volume sampler of the resample kernels (pm_resample.cu, pm_spline.cu; DESIGN §8 rows 5 and 8).
//
// Given a source coordinate c (z, y, x) in voxel index space, the value scipy.ndimage.map_coordinates(src, c, order,
// mode='constant', cval) gives there:
//   any c_h NaN, < 0 or > n_h - 1                    -> cval
//   order 0: src[floor(c + 0.5)]                     (round half up)
//   order 1: trilinear with weights c - floor(c) and 1 - (c - floor(c)), float64, neighbours clamped to n_h - 1
//   result -> dtype: float32 rounds to nearest; integers round half away from zero and saturate (as scipy casts)
// Offsets are 64-bit.  Source loads go through the read-only path.
#pragma once
#include "pm_common.cuh"

// scipy's cast of a float64 result to the output dtype
template <typename T> __device__ __forceinline__ T pm_rs_cast(double v);
template <> __device__ __forceinline__ float pm_rs_cast<float>(double v) { return __double2float_rn(v); }
template <> __device__ __forceinline__ int32_t pm_rs_cast<int32_t>(double v) {
    const double r = v < 0.0 ? v - 0.5 : v + 0.5;                 // round half away from zero, then truncate
    if (!(r >= -2147483648.0)) return INT32_MIN;                  // (NaN too)
    if (r >= 2147483648.0) return INT32_MAX;
    return (int32_t)r;
}
template <> __device__ __forceinline__ uint16_t pm_rs_cast<uint16_t>(double v) {
    const double r = v < 0.0 ? v - 0.5 : v + 0.5;
    if (!(r >= 1.0)) return 0;                                    // (NaN too)
    if (r >= 65535.0) return 65535;
    return (uint16_t)(unsigned)r;
}

// One output voxel: `valid` false (a pad lane past the row's end) or c outside the source -> cv (= cast of cval).
template <typename T, int ORDER>
__device__ __forceinline__ T pm_rs_sample(const T *__restrict__ src, const int (&n)[3], const double (&c)[3], bool valid,
                                          T cv) {
    bool in = valid;
#pragma unroll
    for (int h = 0; h < 3; ++h) in &= c[h] >= 0.0 && c[h] <= (double)(n[h] - 1);       // false for NaN
    if (!in) return cv;
    const int sy = n[1], sx = n[2];
    if (ORDER == 0) {
        const int iz = __double2int_rd(__dadd_rn(c[0], 0.5));
        const int iy = __double2int_rd(__dadd_rn(c[1], 0.5));
        const int ix = __double2int_rd(__dadd_rn(c[2], 0.5));
        return __ldg(src + ((size_t)iz * sy + iy) * sx + ix);
    } else {
        int i0[3], i1[3];
        double w1[3], w0[3];
#pragma unroll
        for (int h = 0; h < 3; ++h) {
            i0[h] = __double2int_rd(c[h]);
            i1[h] = min(i0[h] + 1, n[h] - 1);
            w1[h] = c[h] - (double)i0[h];
            w0[h] = 1.0 - w1[h];
        }
        const size_t r00 = ((size_t)i0[0] * sy + i0[1]) * sx, r01 = ((size_t)i0[0] * sy + i1[1]) * sx;
        const size_t r10 = ((size_t)i1[0] * sy + i0[1]) * sx, r11 = ((size_t)i1[0] * sy + i1[1]) * sx;
        const double v000 = (double)(__ldg(src + r00 + i0[2])), v001 = (double)(__ldg(src + r00 + i1[2]));
        const double v010 = (double)(__ldg(src + r01 + i0[2])), v011 = (double)(__ldg(src + r01 + i1[2]));
        const double v100 = (double)(__ldg(src + r10 + i0[2])), v101 = (double)(__ldg(src + r10 + i1[2]));
        const double v110 = (double)(__ldg(src + r11 + i0[2])), v111 = (double)(__ldg(src + r11 + i1[2]));
        const double a0 = (v000 * w0[2] + v001 * w1[2]) * w0[1] + (v010 * w0[2] + v011 * w1[2]) * w1[1];
        const double a1 = (v100 * w0[2] + v101 * w1[2]) * w0[1] + (v110 * w0[2] + v111 * w1[2]) * w1[1];
        return pm_rs_cast<T>(a0 * w0[0] + a1 * w1[0]);
    }
}

// 4 consecutive x outputs starting at p: one vector store when all 4 are in the row and p is aligned, else scalars
template <typename T> __device__ __forceinline__ void pm_rs_store4(T *p, const T (&v)[4]) {
    if constexpr (sizeof(T) == 4) {
        uint4 q;
        memcpy(&q, v, 16);
        __stcs(reinterpret_cast<uint4 *>(p), q);
    } else {
        uint2 q;
        memcpy(&q, v, 8);
        __stcs(reinterpret_cast<uint2 *>(p), q);
    }
}

template <typename T> __device__ __forceinline__ void pm_rs_store_quad(T *p, const T (&v)[4], unsigned left) {
    if (left >= 4 && (reinterpret_cast<size_t>(p) & (4 * sizeof(T) - 1)) == 0) {
        pm_rs_store4(p, v);
    } else {
#pragma unroll
        for (int e = 0; e < 4; ++e)
            if ((unsigned)e < left) p[e] = v[e];
    }
}
