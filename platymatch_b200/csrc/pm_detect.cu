// pm_detect.cu — nuclei detection in an intensity volume by scale-space LoG minima (SURVEY §2 row 10).
//
// Reference: platymatch/detect_nuclei/ss_log.py (find_spheres :83-87, sphere_log :25-35, suppress_intersecting_spheres
// :53-64).  The reference's exact parameters are not available to this project, so the contract is this project's own
// (DESIGN §8 row 6, restated in tests/detect_oracle.py); agreement with the reference's DetectNuclei output is unverified.
//
//   pass      one separable 1-D correlation along one axis, float64 weights, mode 'reflect' (period 2n, as scipy's
//             correlate1d extends a line), float64 accumulation in scipy's symmetric order, float32 result
//   otsu      min / max, np.histogram's 256-bin binning of float32 data with float32 edges, skimage's threshold_otsu
//   minima    strict (value, linear index) minimum over the 3x3x3x3 scale-space neighbourhood and above threshold
//   suppress  greedy sphere-overlap suppression in priority order, as a fixed point over a uniform grid
//
// This file is compiled with -fmad=false: the threshold and the lens volumes must round like numpy's float64.
#include "pm_common.cuh"

#include <math.h>

// ---- separable pass ---------------------------------------------------------------------------------------------
// A CTA owns 32 lines x 64 positions along the axis.  Lane = line, warp = 8 consecutive positions (PM_DT_R) of that
// line.  The tile plus its 2 lw halo is staged once in shared memory as float64 (each input converted once); every
// thread then slides two register windows (left / right taps) over it: 2 shared loads and 3 FP64 operations per tap
// pair and output.  Lines along x are rows of the tile (odd row stride: conflict-free), lines along y or z are 32
// consecutive x (coalesced loads and stores).
constexpr int PM_DT_R = 8, PM_DT_WARPS = 8, PM_DT_TL = PM_DT_R * PM_DT_WARPS;
constexpr int PM_DT_MAX_LW = 384;   // (64 + 2 * 384 + 1) x 32 x 8 bytes = 213 KB of shared memory

__device__ __forceinline__ int pm_dt_reflect(int i, int n) {
    if (n == 1) return 0;
    const int p = 2 * n;
    int m = i % p;
    if (m < 0) m += p;
    return m < n ? m : p - 1 - m;
}

template <int AXIS>
__global__ void __launch_bounds__(256, 2) pm_detect_pass_kernel(const float *__restrict__ src, int nz, int ny, int nx,
                                                             const double *__restrict__ w, int lw,
                                                             const float *__restrict__ t0, const float *__restrict__ t1,
                                                             float scale, float *__restrict__ dst, unsigned tiles_a,
                                                             unsigned lines_x) {
    extern __shared__ double s_tile[];
    const int lane = threadIdx.x & 31, g = threadIdx.x >> 5;
    const unsigned ta = blockIdx.x % tiles_a, tl = blockIdx.x / tiles_a;
    const int n_a = AXIS == 0 ? nz : AXIS == 1 ? ny : nx;
    const size_t stride_a = AXIS == 0 ? (size_t)ny * nx : AXIS == 1 ? (size_t)nx : 1;
    const int W = PM_DT_TL + 2 * lw, S = AXIS == 2 ? (W | 1) : 32;
    const int a0 = (int)ta * PM_DT_TL;
    // offset of the first element of line l of this tile, or ~0 when the tile's line l lies outside the volume
    const unsigned q = AXIS == 2 ? 0u : tl % lines_x, o = AXIS == 2 ? 0u : tl / lines_x;  // o = z (AXIS 1), y (AXIS 0)
    auto line = [&](int l) -> size_t {
        if (AXIS == 2) {
            const size_t r = (size_t)tl * 32 + l;
            return r < (size_t)nz * ny ? r * nx : ~(size_t)0;
        }
        const int x = (int)q * 32 + l;
        return x < nx ? (AXIS == 1 ? (size_t)o * ny * nx : (size_t)o * nx) + x : ~(size_t)0;
    };
    for (int e = threadIdx.x; e < 32 * W; e += 256) {
        const int l = AXIS == 2 ? e / W : e & 31, a = AXIS == 2 ? e - l * W : e >> 5;
        const size_t lb = line(l);
        s_tile[AXIS == 2 ? l * S + a : a * 32 + l] =
            lb == ~(size_t)0 ? 0.0 : (double)__ldg(src + lb + (size_t)pm_dt_reflect(a0 - lw + a, n_a) * stride_a);
    }
    __syncthreads();
    const size_t base = line(lane);
    if (base == ~(size_t)0) return;
    const int p0 = g * PM_DT_R + lw;                                 // tile position of this thread's first output
    if (a0 + p0 - lw >= n_a) return;
    const double *sl = AXIS == 2 ? s_tile + lane * S : s_tile + lane;
    const int ss = AXIS == 2 ? 1 : 32;
    double acc[PM_DT_R], lf[PM_DT_R], rt[PM_DT_R];
    const double w0 = __ldg(w);
#pragma unroll
    for (int r = 0; r < PM_DT_R; ++r) {
        acc[r] = __dmul_rn(sl[(p0 + r) * ss], w0);
        lf[r] = sl[(p0 + r - lw) * ss];
        rt[r] = sl[(p0 + r + lw) * ss];
    }
    // scipy's order: centre first, then the tap pairs from the outermost inwards
    for (int j = lw; j >= 1; --j) {
        const double wj = __ldg(w + j);
#pragma unroll
        for (int r = 0; r < PM_DT_R; ++r) acc[r] = __dadd_rn(acc[r], __dmul_rn(__dadd_rn(lf[r], rt[r]), wj));
        if (j > 1) {
#pragma unroll
            for (int r = 0; r < PM_DT_R - 1; ++r) lf[r] = lf[r + 1];
            lf[PM_DT_R - 1] = sl[(p0 + PM_DT_R - j) * ss];
#pragma unroll
            for (int r = PM_DT_R - 1; r > 0; --r) rt[r] = rt[r - 1];
            rt[0] = sl[(p0 + j - 1) * ss];
        }
    }
#pragma unroll
    for (int r = 0; r < PM_DT_R; ++r) {
        const int a = a0 + g * PM_DT_R + r;
        if (a >= n_a) break;
        const size_t i = base + (size_t)a * stride_a;
        float v = __double2float_rn(acc[r]);
        if (t0) v = __fmul_rn(scale, __fadd_rn(__fadd_rn(__ldg(t0 + i), __ldg(t1 + i)), v));
        dst[i] = v;
    }
}

template <int AXIS>
static int pm_detect_pass_run(const float *src, int nz, int ny, int nx, const double *w, int lw, const float *t0,
                              const float *t1, float scale, float *dst, cudaStream_t s) {
    const int n_a = AXIS == 0 ? nz : AXIS == 1 ? ny : nx;
    const unsigned long long tiles_a = ((unsigned long long)n_a + PM_DT_TL - 1) / PM_DT_TL;
    const unsigned long long lines_x = ((unsigned long long)nx + 31) / 32;
    const unsigned long long tiles_l = AXIS == 2 ? ((unsigned long long)nz * ny + 31) / 32
                                                 : lines_x * (unsigned long long)(AXIS == 1 ? nz : ny);
    const unsigned long long tiles = tiles_a * tiles_l;
    if (tiles > 0x7fffffffull) {
        pm_set_error("pm_detect_pass: volume of %d x %d x %d needs more than 2^31 - 1 CTAs", nz, ny, nx);
        return PM_ERR_UNSUPPORTED;
    }
    const int W = PM_DT_TL + 2 * lw;
    const size_t smem = (size_t)32 * (AXIS == 2 ? (W | 1) : W) * sizeof(double);
    if (smem > 48 * 1024)
        PM_CUDA_TRY(cudaFuncSetAttribute(pm_detect_pass_kernel<AXIS>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         (int)smem));
    pm_detect_pass_kernel<AXIS><<<(unsigned)tiles, 256, smem, s>>>(src, nz, ny, nx, w, lw, t0, t1, scale, dst,
                                                                     (unsigned)tiles_a, (unsigned)lines_x);
    PM_LAUNCH_CHECK();
    return PM_OK;
}

static bool pm_dt_disjoint(const void *a, size_t abytes, const void *b, size_t bbytes) {
    const uintptr_t x = (uintptr_t)a, y = (uintptr_t)b;
    return x + abytes <= y || y + bbytes <= x;
}

extern "C" int pm_detect_pass(const float *src, int nz, int ny, int nx, int axis, const double *weights, int lw,
                              const float *t0, const float *t1, float scale, float *dst, void *stream) {
    PM_REQUIRE(src && weights && dst, "null pointer");
    PM_REQUIRE((t0 == nullptr) == (t1 == nullptr), "t0 and t1 must both be given or both be NULL");
    PM_REQUIRE(nz >= 1 && ny >= 1 && nx >= 1, "every extent must be >= 1");
    PM_REQUIRE(axis >= 0 && axis <= 2, "axis must be 0 (z), 1 (y) or 2 (x)");
    PM_REQUIRE(lw >= 0 && lw <= PM_DT_MAX_LW, "lw must be in [0, 384]");
    const unsigned __int128 nbytes = (unsigned __int128)nz * ny * nx * sizeof(float);
    PM_REQUIRE(nbytes < ((unsigned __int128)1 << 62), "volume too large");
    PM_REQUIRE(pm_dt_disjoint(src, (size_t)nbytes, dst, (size_t)nbytes), "src and dst overlap (in-place is not supported)");
    PM_REQUIRE(!t0 || (pm_dt_disjoint(t0, (size_t)nbytes, dst, (size_t)nbytes) &&
                       pm_dt_disjoint(t1, (size_t)nbytes, dst, (size_t)nbytes)),
               "t0 / t1 and dst overlap");
    const cudaStream_t s = pm_stream(stream);
    if (axis == 0) return pm_detect_pass_run<0>(src, nz, ny, nx, weights, lw, t0, t1, scale, dst, s);
    if (axis == 1) return pm_detect_pass_run<1>(src, nz, ny, nx, weights, lw, t0, t1, scale, dst, s);
    return pm_detect_pass_run<2>(src, nz, ny, nx, weights, lw, t0, t1, scale, dst, s);
}

// ---- Otsu threshold -----------------------------------------------------------------------------------------------
// Workspace: [0] min key, [1] max key (order-preserving uint32 images of the float32 values), then 256 uint64 counts.
constexpr int PM_DT_BINS = 256;

__device__ __forceinline__ unsigned pm_dt_fkey(float f) {
    const unsigned u = __float_as_uint(f);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float pm_dt_funkey(unsigned k) {
    return __uint_as_float((k & 0x80000000u) ? (k & 0x7fffffffu) : ~k);
}

__global__ void pm_detect_otsu_init_kernel(unsigned *mm, unsigned long long *counts) {
    if (threadIdx.x == 0) { mm[0] = 0xffffffffu; mm[1] = 0u; }
    counts[threadIdx.x] = 0ull;
}

__global__ void __launch_bounds__(256) pm_detect_minmax_kernel(const float *__restrict__ img, size_t n, unsigned *mm) {
    unsigned lo = 0xffffffffu, hi = 0u;
    for (size_t i = (size_t)blockIdx.x * 256 + threadIdx.x; i < n; i += (size_t)gridDim.x * 256) {
        const unsigned k = pm_dt_fkey(__ldg(img + i));
        lo = min(lo, k);
        hi = max(hi, k);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        lo = min(lo, __shfl_xor_sync(0xffffffffu, lo, o));
        hi = max(hi, __shfl_xor_sync(0xffffffffu, hi, o));
    }
    if ((threadIdx.x & 31) == 0) {
        atomicMin(mm, lo);
        atomicMax(mm + 1, hi);
    }
}

// edge i of np.linspace(first, last, 257) in float32: i * ((last - first) / 256) + first, the last edge = last
__device__ __forceinline__ float pm_dt_edge(int i, float first, float last, float step) {
    return i == PM_DT_BINS ? last : __fadd_rn(__fmul_rn((float)i, step), first);
}

// np.histogram(img, 256, range=(min, max)) for float32 data: the bin from ((v - first) / (last - first)) * 256 in
// float32, truncated, then corrected against the float32 edges exactly as numpy corrects it
__global__ void __launch_bounds__(256) pm_detect_hist_kernel(const float *__restrict__ img, size_t n,
                                                             const unsigned *mm, unsigned long long *counts) {
    __shared__ unsigned h[PM_DT_BINS];
    h[threadIdx.x] = 0u;
    __syncthreads();
    const float first = pm_dt_funkey(mm[0]), last = pm_dt_funkey(mm[1]);
    if (first < last) {                            // a constant image has no histogram (otsu returns its value)
        const float denom = __fsub_rn(last, first), step = __fdiv_rn(denom, (float)PM_DT_BINS);
        for (size_t i = (size_t)blockIdx.x * 256 + threadIdx.x; i < n; i += (size_t)gridDim.x * 256) {
            const float v = __ldg(img + i);
            if (!(v >= first && v <= last)) continue;
            int b = (int)__fmul_rn(__fdiv_rn(__fsub_rn(v, first), denom), (float)PM_DT_BINS);
            if (b == PM_DT_BINS) b -= 1;
            if (v < pm_dt_edge(b, first, last, step)) b -= 1;
            if (b != PM_DT_BINS - 1 && v >= pm_dt_edge(b + 1, first, last, step)) b += 1;
            atomicAdd(&h[b], 1u);
        }
    }
    __syncthreads();
    if (h[threadIdx.x]) atomicAdd(counts + threadIdx.x, (unsigned long long)h[threadIdx.x]);
}

// skimage.filters.threshold_otsu(nbins=256) on those counts, float64 in numpy's association, sequential cumulative
// sums, first maximum.  out[0] = otsu, out[1] = factor * otsu.
__global__ void pm_detect_otsu_final_kernel(const unsigned *mm, const unsigned long long *counts, double factor,
                                            double *out) {
    if (threadIdx.x != 0) return;
    const float first = pm_dt_funkey(mm[0]), last = pm_dt_funkey(mm[1]);
    double t = (double)first;
    if (first < last) {
        const float step = __fdiv_rn(__fsub_rn(last, first), (float)PM_DT_BINS);
        double c[PM_DT_BINS], m[PM_DT_BINS], w2[PM_DT_BINS], s2[PM_DT_BINS];
        for (int i = 0; i < PM_DT_BINS; ++i) {
            c[i] = (double)__fdiv_rn(__fadd_rn(pm_dt_edge(i, first, last, step), pm_dt_edge(i + 1, first, last, step)),
                                     2.0f);
            m[i] = (double)counts[i];
        }
        double a2 = 0.0, b2 = 0.0;
        for (int i = PM_DT_BINS - 1; i >= 0; --i) {
            a2 = i == PM_DT_BINS - 1 ? m[i] : a2 + m[i];
            b2 = i == PM_DT_BINS - 1 ? m[i] * c[i] : b2 + m[i] * c[i];
            w2[i] = a2;
            s2[i] = b2;
        }
        double w1 = 0.0, s1 = 0.0, best = 0.0;
        int arg = 0;
        for (int i = 0; i < PM_DT_BINS - 1; ++i) {
            w1 = i == 0 ? m[0] : w1 + m[i];
            s1 = i == 0 ? m[0] * c[0] : s1 + m[i] * c[i];
            const double d = s1 / w1 - s2[i + 1] / w2[i + 1];
            const double v = w1 * w2[i + 1] * (d * d);
            if (i == 0 || v > best) { best = v; arg = i; }
        }
        t = c[arg];
    }
    out[0] = t;
    out[1] = factor * t;
}

extern "C" size_t pm_detect_otsu_workspace_bytes(void) {
    return 2 * sizeof(unsigned long long) + PM_DT_BINS * sizeof(unsigned long long);
}

extern "C" int pm_detect_otsu(const float *img, size_t n, double factor, double *out, void *workspace,
                              size_t workspace_bytes, void *stream) {
    PM_REQUIRE(img && out && workspace, "null pointer");
    PM_REQUIRE(n >= 1, "the image must not be empty");
    if (workspace_bytes < pm_detect_otsu_workspace_bytes()) {
        pm_set_error("pm_detect_otsu: workspace of %zu bytes, %zu needed", workspace_bytes,
                     pm_detect_otsu_workspace_bytes());
        return PM_ERR_WORKSPACE;
    }
    const cudaStream_t s = pm_stream(stream);
    unsigned *mm = (unsigned *)workspace;
    unsigned long long *counts = (unsigned long long *)workspace + 2;
    const size_t want = (n + 255) / 256;
    const unsigned blocks = (unsigned)(want < 4096 ? want : 4096);
    pm_detect_otsu_init_kernel<<<1, PM_DT_BINS, 0, s>>>(mm, counts);
    pm_detect_minmax_kernel<<<blocks, 256, 0, s>>>(img, n, mm);
    pm_detect_hist_kernel<<<blocks, 256, 0, s>>>(img, n, mm, counts);
    pm_detect_otsu_final_kernel<<<1, 32, 0, s>>>(mm, counts, factor, out);
    PM_LAUNCH_CHECK_N(4);
    return PM_OK;
}

// ---- scale-space minima -------------------------------------------------------------------------------------------
// One thread per voxel of scale k.  (k, z, y, x) is a candidate when (L, linear index) is strictly smaller than the
// pair of each of its present 3x3x3x3 neighbours: smaller than an earlier neighbour, at most equal to a later one.
__global__ void __launch_bounds__(256) pm_detect_minima_kernel(const float *__restrict__ lp, const float *__restrict__ lc,
                                                               const float *__restrict__ ln, int nz, int ny, int nx,
                                                               int k, const double *__restrict__ thr,
                                                               unsigned long long cap, long long *keys, float *vals,
                                                               unsigned long long *count, unsigned tiles_x,
                                                               unsigned tiles_y) {
    const unsigned b = blockIdx.x, t2 = b / tiles_x;
    const int x = (int)((b - t2 * tiles_x) * 32 + (threadIdx.x & 31));
    const int y = (int)((t2 % tiles_y) * 8 + (threadIdx.x >> 5));
    const int z = (int)(t2 / tiles_y);
    if (x >= nx || y >= ny) return;
    const size_t plane = (size_t)ny * nx, i = (size_t)z * plane + (size_t)y * nx + x;
    const float v = lc[i];
    if (!(-(double)v > __ldg(thr + 1))) return;
    const float *vol[3] = {lp, lc, ln};
#pragma unroll
    for (int dk = 0; dk < 3; ++dk) {
        const float *L = vol[dk];
        if (!L) continue;
        for (int dz = -1; dz <= 1; ++dz) {
            const int zz = z + dz;
            if (zz < 0 || zz >= nz) continue;
            for (int dy = -1; dy <= 1; ++dy) {
                const int yy = y + dy;
                if (yy < 0 || yy >= ny) continue;
                const float *row = L + (size_t)zz * plane + (size_t)yy * nx;
#pragma unroll
                for (int dx = -1; dx <= 1; ++dx) {
                    const int xx = x + dx;
                    if (xx < 0 || xx >= nx || (dk == 1 && dz == 0 && dy == 0 && dx == 0)) continue;
                    const float u = __ldg(row + xx);
                    // neighbour later in (k, z, y, x) order: ties go to this voxel
                    const bool later = dk != 1 ? dk > 1 : dz != 0 ? dz > 0 : dy != 0 ? dy > 0 : dx > 0;
                    if (later ? !(v <= u) : !(v < u)) return;
                }
            }
        }
    }
    const unsigned long long pos = atomicAdd(count, 1ull);
    if (pos < cap) {
        keys[pos] = (long long)((size_t)k * nz * plane + i);
        vals[pos] = v;
    }
}

extern "C" int pm_detect_minima(const float *l_prev, const float *l_cur, const float *l_next, int nz, int ny, int nx,
                                int k, const double *threshold, long long capacity, long long *keys, float *values,
                                unsigned long long *count, void *stream) {
    PM_REQUIRE(l_cur && threshold && count, "null pointer");
    PM_REQUIRE(capacity >= 0 && (capacity == 0 || (keys && values)), "capacity must be >= 0 with keys and values");
    PM_REQUIRE(nz >= 1 && ny >= 1 && nx >= 1, "every extent must be >= 1");
    PM_REQUIRE(k >= 0, "k must be >= 0");
    const unsigned long long tiles_x = ((unsigned long long)nx + 31) / 32, tiles_y = ((unsigned long long)ny + 7) / 8;
    const unsigned long long tiles = tiles_x * tiles_y * (unsigned long long)nz;
    if (tiles > 0x7fffffffull) {
        pm_set_error("pm_detect_minima: volume of %d x %d x %d needs more than 2^31 - 1 CTAs", nz, ny, nx);
        return PM_ERR_UNSUPPORTED;
    }
    pm_detect_minima_kernel<<<(unsigned)tiles, 256, 0, pm_stream(stream)>>>(
        l_prev, l_cur, l_next, nz, ny, nx, k, threshold, (unsigned long long)capacity, keys, values, count,
        (unsigned)tiles_x, (unsigned)tiles_y);
    PM_LAUNCH_CHECK();
    return PM_OK;
}

// ---- greedy suppression -------------------------------------------------------------------------------------------
// Candidates arrive sorted by priority.  Each is a sphere at (z a, y, x) of radius radii[k]; candidate i is dropped
// when an earlier kept candidate j conflicts with it (lens volume > overlap x volume of the smaller sphere), else kept.
// Conflicting spheres are less than 2 max_radius apart, so a uniform grid of cells >= 2 max_radius holds every
// conflicting pair in adjacent cells.  One CTA decides 1024 consecutive candidates at a time: everything earlier is
// already decided, and inside the chunk the rule is iterated to its fixed point (a candidate is dropped as soon as an
// earlier conflicting one is kept, kept once all earlier conflicting ones are dropped), which is the sequential greedy
// after as many rounds as the longest chain of conflicts inside the chunk.
constexpr int PM_DT_MAX_CELLS = 1 << 22;
constexpr unsigned char PM_DT_UNDECIDED = 0, PM_DT_KEEP = 1, PM_DT_DROP = 2;

struct PmDtGrid {
    double cell;
    int g[3];
};

static PmDtGrid pm_dt_grid(int nz, int ny, int nx, double a, double max_radius) {
    PmDtGrid G;
    G.cell = 2.0 * max_radius;
    const double e[3] = {(double)(nz - 1) * a, (double)(ny - 1), (double)(nx - 1)};
    for (;;) {
        double cells = 1.0;
        for (int h = 0; h < 3; ++h) cells *= floor(e[h] / G.cell) + 1.0;
        if (cells <= PM_DT_MAX_CELLS) break;
        G.cell *= 2.0;
    }
    for (int h = 0; h < 3; ++h) G.g[h] = (int)floor(e[h] / G.cell) + 1;
    return G;
}

struct PmDtSphere {
    double c[3], r;
};

__device__ __forceinline__ PmDtSphere pm_dt_sphere(long long key, int nz, int ny, int nx, double a,
                                                   const double *radii) {
    const long long x = key % nx, t = key / nx, y = t % ny, t2 = t / ny, z = t2 % nz, k = t2 / nz;
    PmDtSphere s;
    s.c[0] = (double)z * a;
    s.c[1] = (double)y;
    s.c[2] = (double)x;
    s.r = __ldg(radii + k);
    return s;
}

__device__ __forceinline__ int pm_dt_cell(const PmDtSphere &s, double cell, int h, int g) {
    return min((int)floor(s.c[h] / cell), g - 1);
}

// the intersection volume of the two spheres > overlap x the smaller sphere's volume; same formula and association as
// ss_log.sphere_intersection (this file has no FMA contraction)
__device__ __forceinline__ bool pm_dt_conflict(const PmDtSphere &p, const PmDtSphere &q, double overlap) {
    const double dz = p.c[0] - q.c[0], dy = p.c[1] - q.c[1], dx = p.c[2] - q.c[2];
    const double d = sqrt(dz * dz + dy * dy + dx * dx);
    const double r1 = p.r > q.r ? p.r : q.r, r2 = p.r > q.r ? q.r : p.r, rs = r2;   // larger radius first
    const double vs = 4.0 / 3.0 * M_PI * rs * rs * rs;
    double inter;
    if (d >= r1 + r2) {
        inter = 0.0;
    } else if (d <= fabs(r1 - r2)) {
        inter = vs;
    } else {
        const double h = r1 + r2 - d;
        inter = M_PI * h * h * (d * d + 2.0 * d * r2 - 3.0 * r2 * r2 + 2.0 * d * r1 + 6.0 * r1 * r2 - 3.0 * r1 * r1) /
                (12.0 * d);
    }
    return inter > overlap * vs;
}

struct PmDtArgs {
    const long long *keys;
    const unsigned long long *count;
    unsigned long long cap;
    int nz, ny, nx;
    double a, overlap, cell;
    int g0, g1, g2;
    const double *radii;
    int *cell_of, *cell_start, *cursor, *members;
    unsigned char *state;
};

__device__ __forceinline__ unsigned long long pm_dt_n(const PmDtArgs &A) { return min(*A.count, A.cap); }

__global__ void pm_detect_cells_kernel(PmDtArgs A) {
    const unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= pm_dt_n(A)) return;
    const PmDtSphere s = pm_dt_sphere(A.keys[i], A.nz, A.ny, A.nx, A.a, A.radii);
    const int c = (pm_dt_cell(s, A.cell, 0, A.g0) * A.g1 + pm_dt_cell(s, A.cell, 1, A.g1)) * A.g2 +
                  pm_dt_cell(s, A.cell, 2, A.g2);
    A.cell_of[i] = c;
    A.state[i] = PM_DT_UNDECIDED;
    atomicAdd(A.cursor + c, 1);
}

// exclusive scan of the per-cell counts (held in cursor) into cell_start and cursor, one CTA of 1024 threads
__global__ void __launch_bounds__(1024) pm_detect_scan_kernel(PmDtArgs A, int cells) {
    __shared__ int warp_tot[32];
    __shared__ int carry;
    if (threadIdx.x == 0) carry = 0;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    for (int base = 0; base < cells; base += 1024) {
        const int c = base + threadIdx.x;
        const int v = c < cells ? A.cursor[c] : 0;
        int x = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int y = __shfl_up_sync(0xffffffffu, x, o);
            if (lane >= o) x += y;
        }
        __syncthreads();
        if (lane == 31) warp_tot[wid] = x;
        __syncthreads();
        if (wid == 0) {
            int t = warp_tot[lane];
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int y = __shfl_up_sync(0xffffffffu, t, o);
                if (lane >= o) t += y;
            }
            warp_tot[lane] = t;
        }
        __syncthreads();
        const int excl = carry + (wid ? warp_tot[wid - 1] : 0) + x - v;
        if (c < cells) {
            A.cell_start[c] = excl;
            A.cursor[c] = excl;
        }
        __syncthreads();
        if (threadIdx.x == 1023) carry = excl + v;
        __syncthreads();
    }
    if (threadIdx.x == 0) A.cell_start[cells] = carry;
}

__global__ void pm_detect_scatter_kernel(PmDtArgs A) {
    const unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= pm_dt_n(A)) return;
    A.members[atomicAdd(A.cursor + A.cell_of[i], 1)] = (int)i;
}

__global__ void __launch_bounds__(1024) pm_detect_resolve_kernel(PmDtArgs A) {
    const long long n = (long long)pm_dt_n(A);
    volatile unsigned char *state = A.state;
    for (long long b = 0; b < n; b += 1024) {
        const long long i = b + threadIdx.x;
        unsigned char st = i < n ? PM_DT_UNDECIDED : PM_DT_KEEP;
        PmDtSphere p;
        int c0 = 0, c1 = 0, c2 = 0;
        if (i < n) {
            p = pm_dt_sphere(A.keys[i], A.nz, A.ny, A.nx, A.a, A.radii);
            const int c = A.cell_of[i];
            c2 = c % A.g2;
            c1 = (c / A.g2) % A.g1;
            c0 = c / A.g2 / A.g1;
        }
        for (;;) {
            if (st == PM_DT_UNDECIDED) {
                bool kept = false, open = false;
                for (int z = max(c0 - 1, 0); z <= min(c0 + 1, A.g0 - 1) && !kept; ++z)
                    for (int y = max(c1 - 1, 0); y <= min(c1 + 1, A.g1 - 1) && !kept; ++y)
                        for (int x = max(c2 - 1, 0); x <= min(c2 + 1, A.g2 - 1) && !kept; ++x) {
                            const int c = (z * A.g1 + y) * A.g2 + x;
                            for (int m = A.cell_start[c]; m < A.cell_start[c + 1]; ++m) {
                                const int j = A.members[m];
                                if (j >= i) continue;
                                const unsigned char sj = state[j];
                                if (sj == PM_DT_DROP) continue;
                                if (!pm_dt_conflict(p, pm_dt_sphere(A.keys[j], A.nz, A.ny, A.nx, A.a, A.radii),
                                                    A.overlap))
                                    continue;
                                if (sj == PM_DT_KEEP) {
                                    kept = true;
                                    break;
                                }
                                open = true;
                            }
                        }
                if (kept || !open) {
                    st = kept ? PM_DT_DROP : PM_DT_KEEP;
                    state[i] = st;
                }
            }
            if (!__syncthreads_or(st == PM_DT_UNDECIDED)) break;
        }
    }
}

extern "C" size_t pm_detect_suppress_workspace_bytes(long long capacity, int nz, int ny, int nx, double max_radius,
                                                     double anisotropy) {
    if (capacity < 0 || nz < 1 || ny < 1 || nx < 1 || !(max_radius > 0.0) || !(anisotropy > 0.0)) return 0;
    const PmDtGrid G = pm_dt_grid(nz, ny, nx, anisotropy, max_radius);
    const size_t cells = (size_t)G.g[0] * G.g[1] * G.g[2];
    return (2 * cells + 1 + 2 * (size_t)capacity) * sizeof(int);
}

extern "C" int pm_detect_suppress(const long long *keys, const unsigned long long *count, long long capacity, int nz,
                                  int ny, int nx, const double *radii, double max_radius, double anisotropy,
                                  double overlap, unsigned char *state, void *workspace, size_t workspace_bytes,
                                  void *stream) {
    PM_REQUIRE(keys && count && radii && state && workspace, "null pointer");
    PM_REQUIRE(capacity >= 1 && capacity <= 0x7fffffffLL, "capacity must be in [1, 2^31 - 1]");
    PM_REQUIRE(nz >= 1 && ny >= 1 && nx >= 1, "every extent must be >= 1");
    PM_REQUIRE(max_radius > 0.0 && max_radius < 1e300, "max_radius must be > 0 and finite");
    PM_REQUIRE(anisotropy > 0.0 && anisotropy < 1e300, "anisotropy must be > 0 and finite");
    PM_REQUIRE(overlap >= 0.0 && overlap <= 1.0, "overlap must be in [0, 1]");
    const size_t need = pm_detect_suppress_workspace_bytes(capacity, nz, ny, nx, max_radius, anisotropy);
    if (workspace_bytes < need) {
        pm_set_error("pm_detect_suppress: workspace of %zu bytes, %zu needed", workspace_bytes, need);
        return PM_ERR_WORKSPACE;
    }
    const PmDtGrid G = pm_dt_grid(nz, ny, nx, anisotropy, max_radius);
    const int cells = G.g[0] * G.g[1] * G.g[2];
    PmDtArgs A;
    A.keys = keys;
    A.count = count;
    A.cap = (unsigned long long)capacity;
    A.nz = nz, A.ny = ny, A.nx = nx;
    A.a = anisotropy, A.overlap = overlap, A.cell = G.cell;
    A.g0 = G.g[0], A.g1 = G.g[1], A.g2 = G.g[2];
    A.radii = radii;
    int *ws = (int *)workspace;
    A.cursor = ws;
    A.cell_start = ws + cells;
    A.cell_of = ws + 2 * cells + 1;
    A.members = A.cell_of + capacity;
    A.state = state;
    const cudaStream_t s = pm_stream(stream);
    PM_CUDA_TRY(cudaMemsetAsync(A.cursor, 0, (size_t)cells * sizeof(int), s));
    const unsigned blocks = (unsigned)((capacity + 255) / 256);
    pm_detect_cells_kernel<<<blocks, 256, 0, s>>>(A);
    pm_detect_scan_kernel<<<1, 1024, 0, s>>>(A, cells);
    pm_detect_scatter_kernel<<<blocks, 256, 0, s>>>(A);
    pm_detect_resolve_kernel<<<1, 1024, 0, s>>>(A);
    PM_LAUNCH_CHECK_N(4);
    return PM_OK;
}
