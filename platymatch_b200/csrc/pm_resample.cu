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
#include "pm_sample.cuh"    // the sampler (bounds test, order 0 / 1, cast), shared with pm_spline.cu

// CTA tile: PM_RS_QX quads of x outputs x PM_RS_BY rows x PM_RS_BZ planes = 256 threads, tiles in raster order.
// Row-linear (128 quads = 512 x outputs, two rows) against 3-D bricks, on one B200 (1000 W power limit), 384 x 512 x
// 512 volumes under 12 degrees about x, scale 1.03 (tools/resample_bench.py, 160 MB L2 flush before each call):
//   int32 order 0    rows 512 x 2 x 1: 0.249 ms   bricks 64 x 4 x 4: 0.253 ms   bricks 32 x 8 x 4: 0.255 ms
//   uint16 order 1   rows 512 x 2 x 1: 0.675 ms   bricks 64 x 4 x 4: 0.680 ms   bricks 32 x 8 x 4: 0.683 ms
// The order hardly matters: the kernel is bound by its FP64 pipe, not by L2 misses (DESIGN §8, row 5).
constexpr int PM_RS_QX = 128, PM_RS_BY = 2, PM_RS_BZ = 1;
static_assert(PM_RS_QX * PM_RS_BY * PM_RS_BZ == 256, "one CTA is 256 threads");

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
#pragma unroll
        for (int h = 0; h < 3; ++h) c[h] = __dadd_rn(__dadd_rn(row[h], __dmul_rn(x, m2[h])), m3[h]);
        out[e] = pm_rs_sample<T, ORDER>(src, n, c, x0 + e < (unsigned)dx, cv);
    }
    pm_rs_store_quad(dst + ((size_t)z * dy + y) * dx + x0, out, (unsigned)dx - x0);
}

template <typename T>
static int pm_resample_run(const T *src, int sz, int sy, int sx, const double *M, int order, double cval, T *dst,
                           int dz, int dy, int dx, cudaStream_t s) {
    const unsigned long long tiles_x = ((unsigned long long)dx + 4 * PM_RS_QX - 1) / (4 * PM_RS_QX);
    const unsigned long long tiles_y = ((unsigned long long)dy + PM_RS_BY - 1) / PM_RS_BY;
    const unsigned long long tiles_z = ((unsigned long long)dz + PM_RS_BZ - 1) / PM_RS_BZ;
    const unsigned long long tiles = tiles_x * tiles_y * tiles_z;
    if (int rc = pm_check_grid_1d("pm_resample_affine", "output", tiles, dz, dy, dx)) return rc;
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
    PM_REQUIRE(pm_volume_dtype_ok(dtype, true), "dtype must be PM_LABEL_I32, PM_LABEL_U16 or PM_RESAMPLE_F32");
    PM_REQUIRE(order == 0 || order == 1, "order must be 0 or 1");
    unsigned __int128 dst_bytes;
    if (int rc = pm_check_volume_pair(__func__, dtype, src, sz, sy, sx, dst, dz, dy, dx, dst_bytes)) return rc;
    return pm_volume_dispatch<true>(dtype, [&](auto t) {
        using T = decltype(t);
        return pm_resample_run((const T *)src, sz, sy, sx, M, order, cval, (T *)dst, dz, dy, dx, pm_stream(stream));
    });
}
