// pm_spline.cu — a 3-D smoothing thin-plate spline (the biharmonic kernel r): its system matrix, its value at points and
// the volume warp through it (DESIGN §8 row 8).
//
// A spline with centres y_k (k < K) and coefficients c [(K + 4) x 3] maps a point x (z, y, x) to
//   f(x) = sum_k c_k * (-||x - y_k||) + c_K + sum_h c_{K+1+h} * (x_h - shift_h) / scale_h
// which is scipy.interpolate.RBFInterpolator(y, d, kernel='linear', degree=1, smoothing) with scipy's monomial order and
// its shift = (min + max) / 2, scale = (max - min) / 2 (0 -> 1) per axis, computed on the host.  Its coefficients solve
// [-R + lambda I, P; P^T, 0] c = [d; 0] (R_ij = ||y_i - y_j||), whose matrix pm_spline_system writes.
//
// Every kernel takes its distances from one routine (pm_sp_zy, pm_sp_phi): -sqrt((dz * dz + dy * dy) + dx * dx) with
// explicit float64 intrinsics, no FMA contraction, correctly rounded square root.  The evaluation (pm_sp_accumulate,
// pm_sp_finish) is shared by pm_spline_eval and pm_resample_spline: centres in ascending index order, each term one FMA
// into a per-axis accumulator, then the constant and the three polynomial terms.  So the two give the same coordinate
// bits, and both are deterministic.
//
// pm_resample_spline is an N-body pass: a CTA owns 1024 outputs (32 quads of x x 8 rows), each thread 4 consecutive x
// voxels (12 float64 accumulators); the centres and their coefficients (48 B each) are staged through shared memory 256
// at a time, and every thread reads each one as a broadcast.  The 4 voxels of a thread share z and y, so dz * dz + dy *
// dy is computed once per centre for the 4.  The coordinate then goes to the row-5 sampler (pm_sample.cuh).
#include "pm_sample.cuh"

constexpr int PM_SP_QX = 32, PM_SP_BY = 8;          // warp tile: 128 x outputs x 8 rows = 256 threads x 4 voxels
constexpr int PM_SP_CHUNK = 256;                    // centres staged per round (one per thread, 12 KB)
static_assert(PM_SP_QX * PM_SP_BY == 256 && PM_SP_CHUNK == 256, "one CTA is 256 threads, one centre each");

struct __align__(16) PmSpCentre {
    double y[3], c[3];
};

__device__ __forceinline__ double pm_sp_zy(double dz, double dy) { return __dadd_rn(__dmul_rn(dz, dz), __dmul_rn(dy, dy)); }
// -||d||, with zy = pm_sp_zy(dz, dy)
__device__ __forceinline__ double pm_sp_phi(double zy, double dx) { return -__dsqrt_rn(__dadd_rn(zy, __dmul_rn(dx, dx))); }

__device__ __forceinline__ void pm_sp_accumulate(double (&acc)[3], const double (&c)[3], double phi) {
#pragma unroll
    for (int j = 0; j < 3; ++j) acc[j] = __fma_rn(c[j], phi, acc[j]);
}

// f(p) from the kernel sums: + c_K, then + c_{K+1+h} * (p_h - shift_h) / scale_h for h = 0, 1, 2
__device__ __forceinline__ void pm_sp_finish(double (&f)[3], const double (&acc)[3], const double (&p)[3],
                                             const double *__restrict__ tail, const double *__restrict__ shift_scale) {
#pragma unroll
    for (int j = 0; j < 3; ++j) f[j] = __dadd_rn(acc[j], __ldg(tail + j));
#pragma unroll
    for (int h = 0; h < 3; ++h) {
        const double q = __ddiv_rn(__dsub_rn(p[h], __ldg(shift_scale + h)), __ldg(shift_scale + 3 + h));
#pragma unroll
        for (int j = 0; j < 3; ++j) f[j] = __fma_rn(__ldg(tail + 3 * (1 + h) + j), q, f[j]);
    }
}

// centres [base, base + 256) of the spline into shared memory (the caller syncs before and after)
__device__ __forceinline__ void pm_sp_stage(PmSpCentre *s, const double *__restrict__ centres,
                                            const double *__restrict__ coeffs, int base, int k) {
    const int i = base + (int)threadIdx.x;
    if (i < k) {
        PmSpCentre v;
#pragma unroll
        for (int j = 0; j < 3; ++j) {
            v.y[j] = __ldg(centres + 3 * (size_t)i + j);
            v.c[j] = __ldg(coeffs + 3 * (size_t)i + j);
        }
        s[threadIdx.x] = v;
    }
}

// ---- the system matrix ----------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) pm_spline_system_kernel(const double *__restrict__ y, int k,
                                                               const double *__restrict__ shift_scale, double smoothing,
                                                               double *__restrict__ lhs, long long ld) {
    const int m = k + 4;
    const int j = blockIdx.x * 32 + (threadIdx.x & 31);
    const int i = blockIdx.y * 8 + (threadIdx.x >> 5);
    if (i >= m || j >= m) return;
    double v;
    if (i < k && j < k) {
        const double dz = __dsub_rn(__ldg(y + 3 * (size_t)i), __ldg(y + 3 * (size_t)j));
        const double dy = __dsub_rn(__ldg(y + 3 * (size_t)i + 1), __ldg(y + 3 * (size_t)j + 1));
        const double dx = __dsub_rn(__ldg(y + 3 * (size_t)i + 2), __ldg(y + 3 * (size_t)j + 2));
        v = pm_sp_phi(pm_sp_zy(dz, dy), dx);
        if (i == j) v = __dadd_rn(v, smoothing);
    } else if (i < k || j < k) {                     // polynomial blocks: [1, (y - shift) / scale] and its transpose
        const int r = i < k ? i : j, h = (i < k ? j : i) - k;
        v = h == 0 ? 1.0
                   : __ddiv_rn(__dsub_rn(__ldg(y + 3 * (size_t)r + h - 1), __ldg(shift_scale + h - 1)),
                               __ldg(shift_scale + 2 + h));
    } else {
        v = 0.0;
    }
    lhs[(size_t)i * ld + j] = v;
}

// ---- f at n points --------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) pm_spline_eval_kernel(const double *__restrict__ centres,
                                                             const double *__restrict__ coeffs, int k,
                                                             const double *__restrict__ shift_scale,
                                                             const double *__restrict__ pts, long long n,
                                                             double *__restrict__ out) {
    __shared__ PmSpCentre s[PM_SP_CHUNK];
    const long long i = (long long)blockIdx.x * 256 + threadIdx.x;
    const bool active = i < n;
    double p[3] = {0.0, 0.0, 0.0};
    if (active)
#pragma unroll
        for (int h = 0; h < 3; ++h) p[h] = __ldg(pts + 3 * i + h);
    double acc[3] = {0.0, 0.0, 0.0};
    for (int base = 0; base < k; base += PM_SP_CHUNK) {
        __syncthreads();
        pm_sp_stage(s, centres, coeffs, base, k);
        __syncthreads();
        const int cnt = min(PM_SP_CHUNK, k - base);
#pragma unroll 4
        for (int t = 0; t < cnt; ++t) {
            const PmSpCentre q = s[t];
            const double zy = pm_sp_zy(__dsub_rn(p[0], q.y[0]), __dsub_rn(p[1], q.y[1]));
            pm_sp_accumulate(acc, q.c, pm_sp_phi(zy, __dsub_rn(p[2], q.y[2])));
        }
    }
    if (!active) return;
    double f[3];
    pm_sp_finish(f, acc, p, coeffs + 3 * (size_t)k, shift_scale);
#pragma unroll
    for (int j = 0; j < 3; ++j) out[3 * i + j] = f[j];
}

// ---- the volume warp ------------------------------------------------------------------------------------------------
template <typename T, int ORDER>
__global__ void __launch_bounds__(256) pm_resample_spline_kernel(const T *__restrict__ src, int sz, int sy, int sx,
                                                                 const double *__restrict__ centres,
                                                                 const double *__restrict__ coeffs, int k,
                                                                 const double *__restrict__ shift_scale, double cval,
                                                                 T *__restrict__ dst, int dz, int dy, int dx,
                                                                 unsigned tiles_x, unsigned tiles_y) {
    __shared__ PmSpCentre s[PM_SP_CHUNK];
    const unsigned b = blockIdx.x, t2 = b / tiles_x;
    const unsigned tx = b - t2 * tiles_x, ty = t2 % tiles_y, z = t2 / tiles_y;
    const unsigned y = ty * PM_SP_BY + threadIdx.x / PM_SP_QX;
    const unsigned x0 = (tx * PM_SP_QX + threadIdx.x % PM_SP_QX) * 4u;
    // threads past the grid's edge stage centres with the others and write nothing
    const bool active = y < (unsigned)dy && x0 < (unsigned)dx;
    const double pz = (double)z, py = (double)y;
    double px[4], acc[4][3];
#pragma unroll
    for (int e = 0; e < 4; ++e) {
        px[e] = (double)(x0 + e);
        acc[e][0] = acc[e][1] = acc[e][2] = 0.0;
    }
    for (int base = 0; base < k; base += PM_SP_CHUNK) {
        __syncthreads();
        pm_sp_stage(s, centres, coeffs, base, k);
        __syncthreads();
        const int cnt = min(PM_SP_CHUNK, k - base);
#pragma unroll 2
        for (int t = 0; t < cnt; ++t) {
            const PmSpCentre q = s[t];
            const double zy = pm_sp_zy(__dsub_rn(pz, q.y[0]), __dsub_rn(py, q.y[1]));
#pragma unroll
            for (int e = 0; e < 4; ++e) pm_sp_accumulate(acc[e], q.c, pm_sp_phi(zy, __dsub_rn(px[e], q.y[2])));
        }
    }
    if (!active) return;
    const int n[3] = {sz, sy, sx};
    const T cv = pm_rs_cast<T>(cval);
    T out[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) {
        const double p[3] = {pz, py, px[e]};
        double c[3];
        pm_sp_finish(c, acc[e], p, coeffs + 3 * (size_t)k, shift_scale);
        out[e] = pm_rs_sample<T, ORDER>(src, n, c, x0 + e < (unsigned)dx, cv);
    }
    pm_rs_store_quad(dst + ((size_t)z * dy + y) * dx + x0, out, (unsigned)dx - x0);
}

template <typename T>
static int pm_resample_spline_run(const T *src, int sz, int sy, int sx, const double *centres, const double *coeffs,
                                  int k, const double *shift_scale, int order, double cval, T *dst, int dz, int dy,
                                  int dx, cudaStream_t s) {
    const unsigned long long tiles_x = ((unsigned long long)dx + 4 * PM_SP_QX - 1) / (4 * PM_SP_QX);
    const unsigned long long tiles_y = ((unsigned long long)dy + PM_SP_BY - 1) / PM_SP_BY;
    const unsigned long long tiles = tiles_x * tiles_y * (unsigned long long)dz;
    if (int rc = pm_check_grid_1d("pm_resample_spline", "output", tiles, dz, dy, dx)) return rc;
    if (order == 0)
        pm_resample_spline_kernel<T, 0><<<(unsigned)tiles, 256, 0, s>>>(src, sz, sy, sx, centres, coeffs, k, shift_scale,
                                                                        cval, dst, dz, dy, dx, (unsigned)tiles_x,
                                                                        (unsigned)tiles_y);
    else
        pm_resample_spline_kernel<T, 1><<<(unsigned)tiles, 256, 0, s>>>(src, sz, sy, sx, centres, coeffs, k, shift_scale,
                                                                        cval, dst, dz, dy, dx, (unsigned)tiles_x,
                                                                        (unsigned)tiles_y);
    PM_LAUNCH_CHECK();
    return PM_OK;
}

// bytes of the spline's device arrays: centres [k][3], coeffs [k + 4][3], shift_scale [6]
static inline unsigned __int128 pm_sp_centre_bytes(int k) { return (unsigned __int128)k * 24; }
static inline unsigned __int128 pm_sp_coeff_bytes(int k) { return ((unsigned __int128)k + 4) * 24; }

extern "C" int pm_spline_system(const double *centres, int k, const double *shift_scale, double smoothing, double *lhs,
                                long long ld, void *stream) {
    PM_REQUIRE(centres && shift_scale && lhs, "null pointer");
    PM_REQUIRE(k >= 1, "k must be >= 1");
    PM_REQUIRE(k <= (1 << 30) - 4, "k too large");
    PM_REQUIRE(ld >= (long long)k + 4, "ld must be >= k + 4");
    PM_REQUIRE(smoothing >= 0.0 && smoothing <= 1.7976931348623157e308, "smoothing must be finite and >= 0");
    const unsigned __int128 lhs_bytes = ((unsigned __int128)ld * (k + 3) + k + 4) * 8;
    PM_REQUIRE(lhs_bytes < ((unsigned __int128)1 << 63), "matrix too large");
    PM_REQUIRE(!pm_ranges_overlap(lhs, lhs_bytes, centres, pm_sp_centre_bytes(k)) &&
                   !pm_ranges_overlap(lhs, lhs_bytes, shift_scale, 48),
               "lhs overlaps an input");
    const int m = k + 4;
    const dim3 grid((m + 31) / 32, (m + 7) / 8);
    PM_REQUIRE(grid.y <= 65535u, "k too large");
    pm_spline_system_kernel<<<grid, 256, 0, pm_stream(stream)>>>(centres, k, shift_scale, smoothing, lhs, ld);
    PM_LAUNCH_CHECK();
    return PM_OK;
}

extern "C" int pm_spline_eval(const double *centres, const double *coeffs, int k, const double *shift_scale,
                              const double *pts, long long n, double *out, void *stream) {
    PM_REQUIRE(centres && coeffs && shift_scale && pts && out, "null pointer");
    PM_REQUIRE(k >= 1, "k must be >= 1");
    PM_REQUIRE(n >= 1, "n must be >= 1");
    PM_REQUIRE(n <= ((long long)1 << 38), "n too large");
    const unsigned __int128 out_bytes = (unsigned __int128)n * 24;
    PM_REQUIRE(!pm_ranges_overlap(out, out_bytes, pts, out_bytes) &&
                   !pm_ranges_overlap(out, out_bytes, centres, pm_sp_centre_bytes(k)) &&
                   !pm_ranges_overlap(out, out_bytes, coeffs, pm_sp_coeff_bytes(k)) &&
                   !pm_ranges_overlap(out, out_bytes, shift_scale, 48),
               "out overlaps an input");
    const unsigned long long blocks = ((unsigned long long)n + 255) / 256;
    pm_spline_eval_kernel<<<(unsigned)blocks, 256, 0, pm_stream(stream)>>>(centres, coeffs, k, shift_scale, pts, n, out);
    PM_LAUNCH_CHECK();
    return PM_OK;
}

extern "C" int pm_resample_spline(const void *src, int dtype, int sz, int sy, int sx, const double *centres,
                                  const double *coeffs, int k, const double *shift_scale, int order, double cval,
                                  void *dst, int dz, int dy, int dx, void *stream) {
    PM_REQUIRE(src && centres && coeffs && shift_scale && dst, "null pointer");
    PM_REQUIRE(pm_volume_dtype_ok(dtype, true), "dtype must be PM_LABEL_I32, PM_LABEL_U16 or PM_RESAMPLE_F32");
    PM_REQUIRE(order == 0 || order == 1, "order must be 0 or 1");
    PM_REQUIRE(k >= 1, "k must be >= 1");
    unsigned __int128 dst_bytes;
    if (int rc = pm_check_volume_pair(__func__, dtype, src, sz, sy, sx, dst, dz, dy, dx, dst_bytes)) return rc;
    PM_REQUIRE(!pm_ranges_overlap(dst, dst_bytes, centres, pm_sp_centre_bytes(k)) &&
                   !pm_ranges_overlap(dst, dst_bytes, coeffs, pm_sp_coeff_bytes(k)) &&
                   !pm_ranges_overlap(dst, dst_bytes, shift_scale, 48),
               "dst overlaps the spline");
    return pm_volume_dispatch<true>(dtype, [&](auto t) {
        using T = decltype(t);
        return pm_resample_spline_run((const T *)src, sz, sy, sx, centres, coeffs, k, shift_scale, order, cval, (T *)dst,
                                      dz, dy, dx, pm_stream(stream));
    });
}
