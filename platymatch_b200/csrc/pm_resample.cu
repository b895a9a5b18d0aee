// pm_resample.cu — resample a volume into another grid through a 4 x 4 affine map (SURVEY §8f row 5).
//
// Reference: platymatch/_dock_widget.py:1095-1130 (EvaluateMetrics._export_transformed_image) resamples the moving
// image into the fixed image's grid with the registration transform (through SimpleITK).  The contract here is
// scipy.ndimage.affine_transform(src, M[:3, :3], offset=M[:3, 3], output_shape, order, mode='constant', cval) in
// voxel index space, order 0 (nearest) or 1 (trilinear):
//   c_h = ((z * M[h][0] + y * M[h][1]) + x * M[h][2]) + M[h][3]      float64, this association, no FMA contraction
//   any c_h NaN, < 0 or > n_h - 1                    -> cval
//   order 0: src[floor(c + 0.5)]                     (round half up)
//   order 1: trilinear with weights c - floor(c) and 1 - (c - floor(c)), float64, neighbours clamped to n_h - 1
//   result -> dtype: float32 rounds to nearest; integers round half away from zero and saturate (as scipy casts)
//
// One thread makes 4 consecutive x outputs (one 16-byte store for int32 / float32, 8 bytes for uint16).  The row
// partials z * M[h][0] + y * M[h][1] are computed once per thread, so a voxel costs one multiply and two adds per
// source axis for its coordinates.  Source loads go through the read-only path; outputs are streamed (never re-read).
#include "pm_common.cuh"

// CTA tile: PM_RS_QX quads of x outputs x PM_RS_BY rows x PM_RS_BZ planes = 256 threads, tiles in raster order.
// Row-linear (128 quads = 512 x outputs, two rows) against 3-D bricks, on one B200 (1000 W power limit), 384 x 512 x
// 512 volumes under 12 degrees about x, scale 1.03 (tools/resample_bench.py, 160 MB L2 flush before each call):
//   int32 order 0    rows 512 x 2 x 1: 0.249 ms   bricks 64 x 4 x 4: 0.253 ms   bricks 32 x 8 x 4: 0.255 ms
//   uint16 order 1   rows 512 x 2 x 1: 0.675 ms   bricks 64 x 4 x 4: 0.680 ms   bricks 32 x 8 x 4: 0.683 ms
// The order hardly matters: the kernel is bound by its FP64 pipe, not by L2 misses (DESIGN §8, row 5).
constexpr int PM_RS_QX = 128, PM_RS_BY = 2, PM_RS_BZ = 1;
static_assert(PM_RS_QX * PM_RS_BY * PM_RS_BZ == 256, "one CTA is 256 threads");

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

template <typename T, int ORDER>
__global__ void __launch_bounds__(256) pm_resample_kernel(const T *__restrict__ src, int sz, int sy, int sx,
                                                          const double *__restrict__ M, double cval,
                                                          T *__restrict__ dst, int dz, int dy, int dx,
                                                          unsigned tiles_x, unsigned tiles_y) {
    const unsigned b = blockIdx.x, t2 = b / tiles_x;
    const unsigned tx = b - t2 * tiles_x, ty = t2 % tiles_y, tz = t2 / tiles_y;
    const unsigned q = threadIdx.x % PM_RS_QX, r = threadIdx.x / PM_RS_QX;
    const unsigned z = tz * PM_RS_BZ + r / PM_RS_BY, y = ty * PM_RS_BY + r % PM_RS_BY;
    const unsigned x0 = (tx * PM_RS_QX + q) * 4u;
    if (z >= (unsigned)dz || y >= (unsigned)dy || x0 >= (unsigned)dx) return;
    const int n[3] = {sz, sy, sx};
    double row[3], m2[3], m3[3];
#pragma unroll
    for (int h = 0; h < 3; ++h) {
        row[h] = __dadd_rn(__dmul_rn((double)z, __ldg(M + 4 * h)), __dmul_rn((double)y, __ldg(M + 4 * h + 1)));
        m2[h] = __ldg(M + 4 * h + 2);
        m3[h] = __ldg(M + 4 * h + 3);
    }
    const T cv = pm_rs_cast<T>(cval);
    T out[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) {
        const double x = (double)(x0 + e);
        double c[3];
        bool in = x0 + e < (unsigned)dx;
#pragma unroll
        for (int h = 0; h < 3; ++h) {
            c[h] = __dadd_rn(__dadd_rn(row[h], __dmul_rn(x, m2[h])), m3[h]);
            in &= c[h] >= 0.0 && c[h] <= (double)(n[h] - 1);       // false for NaN
        }
        out[e] = cv;
        if (!in) continue;
        if (ORDER == 0) {
            const int iz = __double2int_rd(__dadd_rn(c[0], 0.5));
            const int iy = __double2int_rd(__dadd_rn(c[1], 0.5));
            const int ix = __double2int_rd(__dadd_rn(c[2], 0.5));
            out[e] = __ldg(src + ((size_t)iz * sy + iy) * sx + ix);
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
            out[e] = pm_rs_cast<T>(a0 * w0[0] + a1 * w1[0]);
        }
    }
    T *p = dst + ((size_t)z * dy + y) * dx + x0;
    if (x0 + 3 < (unsigned)dx && (reinterpret_cast<size_t>(p) & (4 * sizeof(T) - 1)) == 0) {
        pm_rs_store4(p, out);
    } else {
#pragma unroll
        for (int e = 0; e < 4; ++e)
            if (x0 + e < (unsigned)dx) p[e] = out[e];
    }
}

template <typename T>
static int pm_resample_run(const T *src, int sz, int sy, int sx, const double *M, int order, double cval, T *dst,
                           int dz, int dy, int dx, cudaStream_t s) {
    const unsigned long long tiles_x = ((unsigned long long)dx + 4 * PM_RS_QX - 1) / (4 * PM_RS_QX);
    const unsigned long long tiles_y = ((unsigned long long)dy + PM_RS_BY - 1) / PM_RS_BY;
    const unsigned long long tiles_z = ((unsigned long long)dz + PM_RS_BZ - 1) / PM_RS_BZ;
    const unsigned long long tiles = tiles_x * tiles_y * tiles_z;
    if (tiles > 0x7fffffffull) {
        pm_set_error("pm_resample_affine: output of %d x %d x %d needs more than 2^31 - 1 CTAs", dz, dy, dx);
        return PM_ERR_UNSUPPORTED;
    }
    if (order == 0)
        pm_resample_kernel<T, 0><<<(unsigned)tiles, 256, 0, s>>>(src, sz, sy, sx, M, cval, dst, dz, dy, dx,
                                                                 (unsigned)tiles_x, (unsigned)tiles_y);
    else
        pm_resample_kernel<T, 1><<<(unsigned)tiles, 256, 0, s>>>(src, sz, sy, sx, M, cval, dst, dz, dy, dx,
                                                                 (unsigned)tiles_x, (unsigned)tiles_y);
    PM_LAUNCH_CHECK();
    return PM_OK;
}

extern "C" int pm_resample_affine(const void *src, int dtype, int sz, int sy, int sx, const double *M, int order,
                                  double cval, void *dst, int dz, int dy, int dx, void *stream) {
    PM_REQUIRE(src && M && dst, "null pointer");
    PM_REQUIRE(dtype == PM_LABEL_I32 || dtype == PM_LABEL_U16 || dtype == PM_RESAMPLE_F32,
               "dtype must be PM_LABEL_I32, PM_LABEL_U16 or PM_RESAMPLE_F32");
    PM_REQUIRE(order == 0 || order == 1, "order must be 0 or 1");
    PM_REQUIRE(sz >= 1 && sy >= 1 && sx >= 1 && dz >= 1 && dy >= 1 && dx >= 1, "every extent must be >= 1");
    const unsigned __int128 es = dtype == PM_LABEL_U16 ? 2 : 4;
    const unsigned __int128 src_bytes = (unsigned __int128)sz * sy * sx * es, dst_bytes = (unsigned __int128)dz * dy * dx * es;
    PM_REQUIRE(src_bytes < ((unsigned __int128)1 << 63) && dst_bytes < ((unsigned __int128)1 << 63), "volume too large");
    const unsigned __int128 s0 = (uintptr_t)src, d0 = (uintptr_t)dst;
    PM_REQUIRE(s0 + src_bytes <= d0 || d0 + dst_bytes <= s0, "src and dst overlap (in-place is not supported)");
    if (dtype == PM_LABEL_I32)
        return pm_resample_run((const int32_t *)src, sz, sy, sx, M, order, cval, (int32_t *)dst, dz, dy, dx,
                               pm_stream(stream));
    if (dtype == PM_LABEL_U16)
        return pm_resample_run((const uint16_t *)src, sz, sy, sx, M, order, cval, (uint16_t *)dst, dz, dy, dx,
                               pm_stream(stream));
    return pm_resample_run((const float *)src, sz, sy, sx, M, order, cval, (float *)dst, dz, dy, dx, pm_stream(stream));
}
