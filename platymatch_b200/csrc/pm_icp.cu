// pm_icp.cu — K6: ICP refinement with affine (or similarity, perform_icp.py:19-20) re-fit.
//
// Reference: platymatch/estimate_transform/perform_icp.py:7-26.  Per iteration:
//   cost = distance_matrix(moving^T, fixed^T); i2 = argmin(cost, 1)          (:15-16, first min wins)
//   A_est = get_affine_transform(moving, fixed[:, i2])                        (:18, all N1 pairs)
//   moving = apply_affine_transform(moving, A_est)                            (:23)
//   residual = get_error(moving, fixed[:, i2])  (printed, :24; utils.py:77-88)
//   A_icp = A_est @ A_icp                                                      (:25)
// Always exactly `iterations` iterations, no convergence test, no outlier rejection.
//
// float64: brute-force tiled nearest neighbour (the N1 x N2 distance matrix is never materialised)
// fused with the per-CTA partial sums of the normal equations; one small CTA reduces the partials in
// a fixed order, solves the 4x4 system and composes; a third kernel applies the step and emits the
// residual partials.  Three launches per iteration, no host synchronisation inside the loop.
#include <stdlib.h>
#include <cooperative_groups.h>
#include "pm_common.cuh"

namespace cg = cooperative_groups;

#define PM_ICP_PTS 16      // moving points per CTA
#define PM_ICP_SLICES 16   // column slices per moving point (threads = 16 x 16)
#define PM_ICP_TILE 512    // fixed points staged per tile
#define PM_ICP_NSUM 22     // 10 (M M^T upper) + 12 (F M^T)

// normal-equation terms of one correspondence: 10 (M M^T upper) + 12 (F M^T).
// transform = PM_TRANSFORM_SIMILAR (perform_icp.py:19-20): Horn's fit needs the same sums (n, sum m, sum f,
// sum f m^T, sum |m|^2 = trace of the M M^T block) plus sum |f|^2, which takes the slot of the unused m_x m_y term
// (fixed coordinates shifted by fixed[0] for conditioning).
__device__ __forceinline__ void pm_icp_terms(double mx, double my, double mz, const double *__restrict__ shift,
                                             const double *__restrict__ fixed, int bj, int transform,
                                             double v[PM_ICP_NSUM]) {
    const double m[4] = {mx - shift[0], my - shift[1], mz - shift[2], 1.0};
    const double f[3] = {fixed[3 * (size_t)bj], fixed[3 * (size_t)bj + 1], fixed[3 * (size_t)bj + 2]};
    int q = 0;
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
        for (int b = a; b < 4; ++b) v[q++] = m[a] * m[b];
#pragma unroll
    for (int a = 0; a < 3; ++a)
#pragma unroll
        for (int b = 0; b < 4; ++b) v[q++] = f[a] * m[b];
    if (transform == PM_TRANSFORM_SIMILAR) {
        const double g0 = f[0] - fixed[0], g1 = f[1] - fixed[1], g2 = f[2] - fixed[2];
        v[1] = g0 * g0 + g1 * g1 + g2 * g2;
    }
}

// A_est (4x4, row-major) from the 22 summed terms: fixed_h @ pinv(moving_h) (rank-deficient clouds included), or
// Horn's similarity from the same sums
__device__ __noinline__ void pm_icp_solve_terms(const double *tot, const double *__restrict__ shift,
                                          const double *__restrict__ fixed, int transform, double A[16]) {
    if (transform == PM_TRANSFORM_SIMILAR) {
        // slots: (0,0)=0 (0,1)=1* (0,2)=2 (0,3)=3 (1,1)=4 (1,2)=5 (1,3)=6 (2,2)=7 (2,3)=8 (3,3)=9;  F M^T at 10 + 4 a + b
        const double n = tot[9];
        const double sm[3] = {tot[3], tot[6], tot[8]}, sf[3] = {tot[13], tot[17], tot[21]};
        double cp[3], cy[3], S[9];
        for (int a = 0; a < 3; ++a) { cp[a] = shift[a] + sm[a] / n; cy[a] = sf[a] / n; }
        for (int a = 0; a < 3; ++a)
            for (int b = 0; b < 3; ++b) S[a * 3 + b] = tot[10 + b * 4 + a] - sm[a] * sf[b] / n;
        const double spp = (tot[0] + tot[4] + tot[7]) - (sm[0] * sm[0] + sm[1] * sm[1] + sm[2] * sm[2]) / n;
        const double g[3] = {cy[0] - fixed[0], cy[1] - fixed[1], cy[2] - fixed[2]};
        const double syy = tot[1] - n * (g[0] * g[0] + g[1] * g[1] + g[2] * g[2]);
        pm_similar_from_moments(cp, cy, S, spp, syy, A);
        return;
    }
    double M[16];
    int k = 0;
    for (int a = 0; a < 4; ++a)
        for (int b = a; b < 4; ++b) { M[a * 4 + b] = tot[k]; M[b * 4 + a] = tot[k]; ++k; }
    const double sh[3] = {shift[0], shift[1], shift[2]};
    pm_affine_from_normal_eq(M, tot + 10, sh, 1e-14, A);   // rank-deficient clouds: pinv's minimum-norm answer
}

// cur: current moving positions [n1][3]; shift: 3 doubles subtracted from moving coordinates when
// forming the normal equations (conditioning); partial: [gridDim.x][PM_ICP_NSUM].
__global__ void __launch_bounds__(PM_ICP_PTS * PM_ICP_SLICES)
pm_icp_nn_kernel(const double *__restrict__ cur, int n1, const double *__restrict__ fixed, int n2,
                 const double *__restrict__ shift, int transform, int32_t *__restrict__ nn,
                 double *__restrict__ partial) {
    __shared__ __align__(16) double tile[2][PM_ICP_TILE * 3];      // double-buffered with cp.async
    __shared__ double best_d[PM_ICP_SLICES][PM_ICP_PTS];
    __shared__ int best_j[PM_ICP_SLICES][PM_ICP_PTS];
    __shared__ double sums[PM_ICP_PTS][PM_ICP_NSUM + 1];
    const int p = threadIdx.x % PM_ICP_PTS, s = threadIdx.x / PM_ICP_PTS;
    const int i = blockIdx.x * PM_ICP_PTS + p;
    const bool live = i < n1;
    double mx = 0, my = 0, mz = 0;
    if (live) { mx = cur[3 * i]; my = cur[3 * i + 1]; mz = cur[3 * i + 2]; }
    // The reference keeps the first strict minimum of sqrt(d2) in ascending j.  sqrt is monotone, so a new
    // minimum needs d2 < best d2: the hot loop compares squared distances and only on that (rare) branch
    // evaluates the square roots, which decide exactly like the reference (two different d2 can round to
    // the same distance, and then the earlier index must stay).
    double bd = INFINITY, bd2 = INFINITY;
    int bj = 0x7fffffff;
    auto stage = [&](int buf, int t0) {        // 8-byte cp.async copies of one tile of the fixed cloud
        const int tn = min(PM_ICP_TILE, n2 - t0);
        for (int q = threadIdx.x; q < tn * 3; q += blockDim.x) {
            const unsigned dst = (unsigned)__cvta_generic_to_shared(&tile[buf][q]);
            asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(dst), "l"(fixed + (size_t)t0 * 3 + q));
        }
        asm volatile("cp.async.commit_group;");
    };
    stage(0, 0);
    int buf = 0;
    for (int t0 = 0; t0 < n2; t0 += PM_ICP_TILE, buf ^= 1) {
        const int tn = min(PM_ICP_TILE, n2 - t0);
        if (t0 + PM_ICP_TILE < n2) {
            stage(buf ^ 1, t0 + PM_ICP_TILE);
            asm volatile("cp.async.wait_group 1;");
        } else {
            asm volatile("cp.async.wait_group 0;");
        }
        __syncthreads();
        const double *tl = tile[buf];
        int j = s;
        for (; j + PM_ICP_SLICES < tn; j += 2 * PM_ICP_SLICES) {   // two candidates per trip: independent chains
            const int ja = j, jb = j + PM_ICP_SLICES;
            const double a0 = tl[3 * ja] - mx, a1 = tl[3 * ja + 1] - my, a2 = tl[3 * ja + 2] - mz;
            const double b0 = tl[3 * jb] - mx, b1 = tl[3 * jb + 1] - my, b2 = tl[3 * jb + 2] - mz;
            const double qa = __dadd_rn(__dadd_rn(__dmul_rn(a0, a0), __dmul_rn(a1, a1)), __dmul_rn(a2, a2));
            const double qb = __dadd_rn(__dadd_rn(__dmul_rn(b0, b0), __dmul_rn(b1, b1)), __dmul_rn(b2, b2));
            if (qa < bd2) {                               // ascending j within a slice: first min kept
                const double d = sqrt(qa);
                if (d < bd) { bd = d; bd2 = qa; bj = t0 + ja; }
            }
            if (qb < bd2) {
                const double d = sqrt(qb);
                if (d < bd) { bd = d; bd2 = qb; bj = t0 + jb; }
            }
        }
        for (; j < tn; j += PM_ICP_SLICES) {
            const double d0 = tl[3 * j] - mx, d1 = tl[3 * j + 1] - my, d2 = tl[3 * j + 2] - mz;
            const double q2 = __dadd_rn(__dadd_rn(__dmul_rn(d0, d0), __dmul_rn(d1, d1)), __dmul_rn(d2, d2));
            if (q2 < bd2) {
                const double d = sqrt(q2);
                if (d < bd) { bd = d; bd2 = q2; bj = t0 + j; }
            }
        }
        __syncthreads();
    }
    best_d[s][p] = bd;
    best_j[s][p] = bj;
    __syncthreads();
    if (s == 0) {
        for (int q = 1; q < PM_ICP_SLICES; ++q) {
            const double od = best_d[q][p];
            const int oj = best_j[q][p];
            if (od < bd || (od == bd && oj < bj)) { bd = od; bj = oj; }   // first minimum overall
        }
        double v[PM_ICP_NSUM];
#pragma unroll
        for (int q = 0; q < PM_ICP_NSUM; ++q) v[q] = 0.0;
        if (live) {
            if (bj == 0x7fffffff) bj = 0;        // no finite distance at all: np.argmin of an all-NaN row
            nn[i] = bj;
            pm_icp_terms(mx, my, mz, shift, fixed, bj, transform, v);
        }
#pragma unroll
        for (int q = 0; q < PM_ICP_NSUM; ++q) sums[p][q] = v[q];
    }
    __syncthreads();
    if (threadIdx.x < PM_ICP_NSUM) {   // fixed-order sum over the 32 points of this CTA
        double acc = 0.0;
        for (int q = 0; q < PM_ICP_PTS; ++q) acc += sums[q][threadIdx.x];
        partial[(size_t)blockIdx.x * PM_ICP_NSUM + threadIdx.x] = acc;
    }
}

// ---- exact nearest neighbour through a uniform grid over the fixed cloud ------------------------------
// The fixed cloud does not move during ICP, so its points are bucketed once per call into a uniform grid
// (counting sort by cell); a query visits the cells ring by ring (Chebyshev distance 0, 1, 2, ... from its
// own cell) and stops as soon as the best distance found is smaller than the distance to everything outside
// the visited block.  Distances are evaluated exactly as in the brute-force kernel (numpy's association
// order, f64 sqrt) and the winner is the minimum of (distance, index), i.e. the reference's first minimum in
// ascending index - identical nearest-neighbour maps, ~100 instead of 8000 candidates per query.
struct PmIcpGrid {
    double lo[3];      // lower corner of the bounding box
    double h;          // cell edge
    int g[3];          // cells per axis
    int ncell;
};

__global__ void __launch_bounds__(1024) pm_icp_grid_setup_kernel(const double *__restrict__ fixed, int n2, int target,
                                                                 PmIcpGrid *__restrict__ G, int *__restrict__ cell_count,
                                                                 int max_cells) {
    __shared__ double s_lo[3][32], s_hi[3][32];
    double lo[3] = {INFINITY, INFINITY, INFINITY}, hi[3] = {-INFINITY, -INFINITY, -INFINITY};
    for (int j = threadIdx.x; j < n2; j += blockDim.x)
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            const double x = fixed[3 * (size_t)j + a];
            lo[a] = fmin(lo[a], x); hi[a] = fmax(hi[a], x);
        }
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int a = 0; a < 3; ++a) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            lo[a] = fmin(lo[a], __shfl_xor_sync(0xffffffffu, lo[a], o));
            hi[a] = fmax(hi[a], __shfl_xor_sync(0xffffffffu, hi[a], o));
        }
        if (lane == 0) { s_lo[a][warp] = lo[a]; s_hi[a][warp] = hi[a]; }
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        double ext = 0.0;
        for (int a = 0; a < 3; ++a) {
            double l = INFINITY, u = -INFINITY;
            for (int w = 0; w < (int)(blockDim.x >> 5); ++w) { l = fmin(l, s_lo[a][w]); u = fmax(u, s_hi[a][w]); }
            G->lo[a] = l;
            s_hi[a][0] = u - l;
            ext = fmax(ext, u - l);
        }
        double h = ext / (double)target;
        if (!(h > 0.0) || !isfinite(h)) h = 1.0;             // all points coincide (or non-finite input): one cell
        int ncell = 1;
        for (int a = 0; a < 3; ++a) {
            int g = (int)floor(s_hi[a][0] / h) + 1;
            if (!(g >= 1)) g = 1;
            if (g > target + 1) g = target + 1;
            G->g[a] = g;
            ncell *= g;
        }
        if (ncell > max_cells) { G->g[0] = G->g[1] = G->g[2] = 1; ncell = 1; h = INFINITY; }   // cannot happen: max_cells = (target+1)^3
        G->h = h;
        G->ncell = ncell;
    }
    __syncthreads();
    const int ncell = G->ncell;
    for (int c = threadIdx.x; c <= ncell; c += blockDim.x) cell_count[c] = 0;
}

__device__ __forceinline__ int pm_icp_cell_axis(double x, double lo, double h, int g) {
    const double t = floor((x - lo) / h);
    int c = (t >= (double)g) ? g - 1 : (t > 0.0 ? (int)t : 0);     // clamps queries outside the box; NaN -> 0
    return c;
}

__global__ void __launch_bounds__(256) pm_icp_cell_count_kernel(const double *__restrict__ fixed, int n2,
                                                                const PmIcpGrid *__restrict__ G, int *__restrict__ cell_of,
                                                                int *__restrict__ cell_count) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n2) return;
    const PmIcpGrid g = *G;
    const int cz = pm_icp_cell_axis(fixed[3 * (size_t)j], g.lo[0], g.h, g.g[0]);
    const int cy = pm_icp_cell_axis(fixed[3 * (size_t)j + 1], g.lo[1], g.h, g.g[1]);
    const int cx = pm_icp_cell_axis(fixed[3 * (size_t)j + 2], g.lo[2], g.h, g.g[2]);
    const int c = (cz * g.g[1] + cy) * g.g[2] + cx;
    cell_of[j] = c;
    atomicAdd(&cell_count[c], 1);
}

// one CTA: exclusive scan of the cell counts in place (cell_start[ncell] = n2); cursor = copy for the fill
__global__ void __launch_bounds__(1024) pm_icp_cell_scan_kernel(const PmIcpGrid *__restrict__ G, int *__restrict__ cell_start,
                                                                int *__restrict__ cursor) {
    __shared__ int s_scan[33];
    __shared__ int s_base;
    const int ncell = G->ncell, t = threadIdx.x, lane = t & 31, warp = t >> 5;
    if (t == 0) s_base = 0;
    __syncthreads();
    for (int b = 0; b <= ncell; b += 1024) {
        const int c = b + t;
        const int v = (c < ncell) ? cell_start[c] : 0;
        int incl = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int n = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += n;
        }
        if (lane == 31) s_scan[warp] = incl;
        __syncthreads();
        if (t == 0) {
            int a = s_base;
            for (int w = 0; w < 32; ++w) { const int x = s_scan[w]; s_scan[w] = a; a += x; }
            s_scan[32] = a;
        }
        __syncthreads();
        if (c <= ncell) {
            const int excl = s_scan[warp] + incl - v;
            cell_start[c] = excl;
            cursor[c] = excl;
        }
        __syncthreads();
        if (t == 0) s_base = s_scan[32];
        __syncthreads();
    }
}

__global__ void __launch_bounds__(256) pm_icp_cell_fill_kernel(const double *__restrict__ fixed, int n2,
                                                               const int *__restrict__ cell_of, int *__restrict__ cursor,
                                                               double *__restrict__ sorted_pts, int *__restrict__ sorted_idx) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n2) return;
    const int pos = atomicAdd(&cursor[cell_of[j]], 1);
    sorted_pts[3 * (size_t)pos] = fixed[3 * (size_t)j];
    sorted_pts[3 * (size_t)pos + 1] = fixed[3 * (size_t)j + 1];
    sorted_pts[3 * (size_t)pos + 2] = fixed[3 * (size_t)j + 2];
    sorted_idx[pos] = j;
}

#define PM_ICP_GPTS 128    // moving points per CTA of the grid kernel (one per thread)
#define PM_ICP_QPB 32      // persistent kernel: moving points per CTA ...
#define PM_ICP_LPQ 4       // ... and lanes that share the candidates of one point

// nearest fixed point of (mx, my, mz): ring-by-ring search of the grid, winner = min (distance, index)
// NSUB adjacent lanes share one query: each takes every NSUB-th candidate of a cell run and the partial
// winners are merged with shuffles after every ring (all NSUB lanes leave with the same result).
template <int NSUB>
__device__ __forceinline__ void pm_icp_grid_search(const PmIcpGrid &G, const int *__restrict__ cell_start,
                                                   const double *__restrict__ sorted_pts, const int *__restrict__ sorted_idx,
                                                   double mx, double my, double mz, double &bd, int &bj) {
    const int sub = (NSUB > 1) ? (threadIdx.x & (NSUB - 1)) : 0;
    // the lanes of one query run in lockstep, different queries of a warp do not: shuffle within the group only
    const unsigned gmask = (NSUB > 1) ? (((1u << NSUB) - 1u) << ((threadIdx.x & 31) & ~(NSUB - 1))) : 0u;
    double bd2 = INFINITY;
    bd = INFINITY;
    bj = 0x7fffffff;
        const double q[3] = {mx, my, mz};
        int c[3];
#pragma unroll
        for (int a = 0; a < 3; ++a) c[a] = pm_icp_cell_axis(q[a], G.lo[a], G.h, G.g[a]);
        const int rmax = max(G.g[0], max(G.g[1], G.g[2]));
        for (int r = 0; r <= rmax; ++r) {
            const int z0 = max(c[0] - r, 0), z1 = min(c[0] + r, G.g[0] - 1);
            const int y0 = max(c[1] - r, 0), y1 = min(c[1] + r, G.g[1] - 1);
            const int x0 = max(c[2] - r, 0), x1 = min(c[2] + r, G.g[2] - 1);
            for (int z = z0; z <= z1; ++z) {
                const bool zface = (z == c[0] - r) || (z == c[0] + r);
                for (int y = y0; y <= y1; ++y) {
                    const bool yface = zface || (y == c[1] - r) || (y == c[1] + r);
                    // on a face of the block the whole x-run belongs to ring r, otherwise only its two ends
                    const int row = (z * G.g[1] + y) * G.g[2];
                    auto scan_cells = [&](int xs, int xe) {     // contiguous cells -> contiguous sorted points
                        if (xs > xe) return;
                        const int p0 = __ldg(cell_start + row + xs), p1 = __ldg(cell_start + row + xe + 1);
                        for (int p = p0 + sub; p < p1; p += NSUB) {
                            const double d0 = __ldg(sorted_pts + 3 * (size_t)p) - mx, d1 = __ldg(sorted_pts + 3 * (size_t)p + 1) - my,
                                         d2 = __ldg(sorted_pts + 3 * (size_t)p + 2) - mz;
                            const double q2 = __dadd_rn(__dadd_rn(__dmul_rn(d0, d0), __dmul_rn(d1, d1)), __dmul_rn(d2, d2));
                            // candidates come in no particular index order, and two different q2 can round to the
                            // same distance: let everything within a few ulp of the best through and decide on
                            // (distance, index), which is the reference's first minimum in ascending index
                            if (q2 <= bd2 * (1.0 + 1e-15)) {
                                const double d = sqrt(q2);
                                const int j = __ldg(sorted_idx + p);
                                if (d < bd || (d == bd && j < bj)) { bd = d; bj = j; bd2 = q2; }
                            }
                        }
                    };
                    if (yface) scan_cells(x0, x1);
                    else {
                        if (c[2] - r >= 0) scan_cells(c[2] - r, c[2] - r);
                        if (r > 0 && c[2] + r <= G.g[2] - 1) scan_cells(c[2] + r, c[2] + r);
                    }
                }
            }
            if (NSUB > 1) {     // merge the lanes of this query: minimum of (distance, index)
#pragma unroll
                for (int o = 1; o < NSUB; o <<= 1) {
                    const double od = __shfl_xor_sync(gmask, bd, o), o2 = __shfl_xor_sync(gmask, bd2, o);
                    const int oj = __shfl_xor_sync(gmask, bj, o);
                    if (od < bd || (od == bd && oj < bj)) { bd = od; bj = oj; bd2 = o2; }
                }
            }
            // everything not visited yet lies outside the block of cells [c - r, c + r]: lower bound of its distance
            double bound = INFINITY;
#pragma unroll
            for (int a = 0; a < 3; ++a) {
                if (c[a] - r > 0) bound = fmin(bound, fmax(q[a] - (G.lo[a] + (double)(c[a] - r) * G.h), 0.0));
                if (c[a] + r < G.g[a] - 1) bound = fmin(bound, fmax((G.lo[a] + (double)(c[a] + r + 1) * G.h) - q[a], 0.0));
            }
            if (!(bound < INFINITY)) break;                        // the block covers the whole grid
            // strictly closer than anything outside, with slack for the rounding of the cell assignment
            if (bd < bound * (1.0 - 1e-12) - 1e-9 * G.h) break;
        }
}

__global__ void __launch_bounds__(PM_ICP_GPTS)
pm_icp_nn_grid_kernel(const double *__restrict__ cur, int n1, const double *__restrict__ fixed,
                      const PmIcpGrid *__restrict__ Gp, const int *__restrict__ cell_start,
                      const double *__restrict__ sorted_pts, const int *__restrict__ sorted_idx,
                      const double *__restrict__ shift, int transform, int32_t *__restrict__ nn,
                      double *__restrict__ partial) {
    __shared__ double sums[PM_ICP_GPTS][PM_ICP_NSUM + 1];
    const PmIcpGrid G = *Gp;
    const int i = blockIdx.x * PM_ICP_GPTS + threadIdx.x;
    const bool live = i < n1;
    double mx = 0, my = 0, mz = 0;
    if (live) { mx = cur[3 * (size_t)i]; my = cur[3 * (size_t)i + 1]; mz = cur[3 * (size_t)i + 2]; }
    double bd = INFINITY;
    int bj = 0x7fffffff;
    if (live) pm_icp_grid_search<1>(G, cell_start, sorted_pts, sorted_idx, mx, my, mz, bd, bj);
    double v[PM_ICP_NSUM];
#pragma unroll
    for (int q = 0; q < PM_ICP_NSUM; ++q) v[q] = 0.0;
    if (live) {
        if (bj == 0x7fffffff) bj = 0;            // no finite distance at all: np.argmin of an all-NaN row
        nn[i] = bj;
        pm_icp_terms(mx, my, mz, shift, fixed, bj, transform, v);
    }
#pragma unroll
    for (int q = 0; q < PM_ICP_NSUM; ++q) sums[threadIdx.x][q] = v[q];
    __syncthreads();
    if (threadIdx.x < PM_ICP_NSUM) {   // fixed-order sum over the points of this CTA
        double acc = 0.0;
        for (int q = 0; q < PM_ICP_GPTS; ++q) acc += sums[q][threadIdx.x];
        partial[(size_t)blockIdx.x * PM_ICP_NSUM + threadIdx.x] = acc;
    }
}

// ---- the whole ICP loop in ONE cooperative launch -------------------------------------------------------
// One thread per moving point keeps its point in registers for all iterations.  Per iteration: grid nearest
// neighbour + per-CTA partial sums of the 22 normal-equation terms -> ONE grid barrier -> every CTA reduces
// the partials in the same fixed order and solves the 4x4 system itself (redundantly: cheaper than a second
// barrier and a broadcast) -> apply, residual partials.  The partial sums ping-pong between two buffers, so
// a CTA that runs ahead into the next iteration cannot overwrite what a slower one still reads.
__global__ void __launch_bounds__(PM_ICP_QPB * PM_ICP_LPQ, 4)     // <= 128 registers: 4 CTAs per SM stay co-resident (20k clouds)
pm_icp_persistent_kernel(const double *__restrict__ moving, int n1, const double *__restrict__ fixed, int iterations,
                         int transform, const PmIcpGrid *__restrict__ Gp, const int *__restrict__ cell_start,
                         const double *__restrict__ sorted_pts, const int *__restrict__ sorted_idx,
                         int32_t *__restrict__ nn, double *__restrict__ partial /* [2][grid][NSUM] */,
                         double *__restrict__ res_partial /* [iterations][grid] */, double *__restrict__ a_icp_out) {
    cg::grid_group grid = cg::this_grid();
    __shared__ double sums[PM_ICP_QPB][PM_ICP_NSUM + 1];
    __shared__ double tot[PM_ICP_NSUM];
    __shared__ double s_a[16];
    __shared__ double red[32];
    const PmIcpGrid G = *Gp;
    const int nblk = gridDim.x;
    const int qi = threadIdx.x / PM_ICP_LPQ;                   // query slot of this thread; PM_ICP_LPQ lanes share it
    const bool lead = (threadIdx.x % PM_ICP_LPQ) == 0;
    const int i = blockIdx.x * PM_ICP_QPB + qi;
    const bool live = i < n1;
    const double shift[3] = {moving[0], moving[1], moving[2]};
    double mx = 0, my = 0, mz = 0;
    if (live) { mx = moving[3 * (size_t)i]; my = moving[3 * (size_t)i + 1]; mz = moving[3 * (size_t)i + 2]; }
    double a_icp[16];
#pragma unroll
    for (int e = 0; e < 16; ++e) a_icp[e] = (e % 5 == 0) ? 1.0 : 0.0;
    for (int it = 0; it < iterations; ++it) {
        double bd = INFINITY;
        int bj = 0;
        double v[PM_ICP_NSUM];
#pragma unroll
        for (int q = 0; q < PM_ICP_NSUM; ++q) v[q] = 0.0;
        // (a whole group of PM_ICP_LPQ lanes is live or not: the shuffles inside stay converged.  The padding groups of
        // the last CTA must NOT search: their query (0, 0, 0) lies far outside the cloud and walks the whole grid ring by
        // ring, ~3.5 ms per iteration while every other CTA waits at the grid barrier - 180-500 ms per call whenever
        // n1 is not a multiple of 32, found in round 2 with tools/icp_probe.py / tools/square_probe.py)
        if (live) pm_icp_grid_search<PM_ICP_LPQ>(G, cell_start, sorted_pts, sorted_idx, mx, my, mz, bd, bj);
        if (live) {
            if (bj == 0x7fffffff) bj = 0;        // no finite distance at all: np.argmin of an all-NaN row
            pm_icp_terms(mx, my, mz, shift, fixed, bj, transform, v);
        }
        if (lead) {
#pragma unroll
            for (int q = 0; q < PM_ICP_NSUM; ++q) sums[qi][q] = live ? v[q] : 0.0;
        }
        __syncthreads();
        double *pbuf = partial + (size_t)(it & 1) * nblk * PM_ICP_NSUM;
        if (threadIdx.x < PM_ICP_NSUM) {   // fixed-order sum over the points of this CTA
            double acc = 0.0;
            for (int q = 0; q < PM_ICP_QPB; ++q) acc += sums[q][threadIdx.x];
            pbuf[(size_t)blockIdx.x * PM_ICP_NSUM + threadIdx.x] = acc;
        }
        grid.sync();
        // every CTA: the same fixed-order reduction over all CTAs (5 chunks x 22 terms, then the chunks in order)
        if (threadIdx.x < 5 * PM_ICP_NSUM) {
            const int q = threadIdx.x % PM_ICP_NSUM, ch = threadIdx.x / PM_ICP_NSUM;
            const int per = (nblk + 4) / 5, b0 = ch * per, b1 = min(nblk, b0 + per);
            double acc = 0.0;
#pragma unroll 8
            for (int b = b0; b < b1; ++b) acc += __ldcg(pbuf + (size_t)b * PM_ICP_NSUM + q);
            sums[ch][q] = acc;             // (the per-point terms in `sums` were consumed before the grid barrier)
        }
        __syncthreads();
        if (threadIdx.x < PM_ICP_NSUM)
            tot[threadIdx.x] = (((sums[0][threadIdx.x] + sums[1][threadIdx.x]) + sums[2][threadIdx.x]) + sums[3][threadIdx.x]) +
                               sums[4][threadIdx.x];
        __syncthreads();
        if (threadIdx.x == 0) pm_icp_solve_terms(tot, shift, fixed, transform, s_a);
        __syncthreads();
        double r = 0.0;
        if (live) {     // apply (apply_transform.py:14-17), residual against this iteration's matches (utils.py:77-88)
            const double nx = ((s_a[0] * mx + s_a[1] * my) + s_a[2] * mz) + s_a[3];
            const double ny = ((s_a[4] * mx + s_a[5] * my) + s_a[6] * mz) + s_a[7];
            const double nz = ((s_a[8] * mx + s_a[9] * my) + s_a[10] * mz) + s_a[11];
            mx = nx; my = ny; mz = nz;
            const double e0 = nx - fixed[3 * (size_t)bj], e1 = ny - fixed[3 * (size_t)bj + 1], e2 = nz - fixed[3 * (size_t)bj + 2];
            r = lead ? sqrt(e0 * e0 + e1 * e1 + e2 * e2) : 0.0;
            if (lead && it == iterations - 1) nn[i] = bj;
        }
        r = pm_block_sum(r, red);
        if (threadIdx.x == 0) res_partial[(size_t)it * nblk + blockIdx.x] = r;
        if (blockIdx.x == 0 && threadIdx.x == 0) {      // A_icp <- A_est @ A_icp   (perform_icp.py:25)
            double c[16];
            for (int rr = 0; rr < 4; ++rr)
                for (int cc = 0; cc < 4; ++cc) {
                    double sacc = 0.0;
                    for (int kk = 0; kk < 4; ++kk) sacc += s_a[rr * 4 + kk] * a_icp[kk * 4 + cc];
                    c[rr * 4 + cc] = sacc;
                }
            for (int e = 0; e < 16; ++e) a_icp[e] = c[e];
        }
    }
    if (blockIdx.x == 0 && threadIdx.x == 0)
        for (int e = 0; e < 16; ++e) a_icp_out[e] = a_icp[e];
}

// One CTA: reduce partials, solve, compose.  A_est -> a_est[16]; a_icp <- A_est @ a_icp.
__global__ void __launch_bounds__(256) pm_icp_solve_kernel(const double *__restrict__ partial, int nblocks,
                                                           const double *__restrict__ shift,
                                                           const double *__restrict__ fixed, int transform,
                                                           double *__restrict__ a_est, double *__restrict__ a_icp) {
    __shared__ double tot[PM_ICP_NSUM];
    __shared__ double red[8][PM_ICP_NSUM];
    const int q = threadIdx.x % 32, g = threadIdx.x / 32;   // 8 groups x 32 lanes (22 used)
    if (q < PM_ICP_NSUM) {
        double acc = 0.0;
        for (int b = g; b < nblocks; b += 8) acc += partial[(size_t)b * PM_ICP_NSUM + q];
        red[g][q] = acc;
    }
    __syncthreads();
    if (threadIdx.x < PM_ICP_NSUM) {
        double acc = 0.0;
        for (int k = 0; k < 8; ++k) acc += red[k][threadIdx.x];
        tot[threadIdx.x] = acc;
    }
    __syncthreads();
    if (threadIdx.x != 0) return;
    double A[16];
    pm_icp_solve_terms(tot, shift, fixed, transform, A);
    double C[16];
    for (int r = 0; r < 4; ++r)
        for (int c = 0; c < 4; ++c) {
            double sacc = 0.0;
            for (int kk = 0; kk < 4; ++kk) sacc += A[r * 4 + kk] * a_icp[kk * 4 + c];
            C[r * 4 + c] = sacc;
        }
    for (int e = 0; e < 16; ++e) { a_est[e] = A[e]; a_icp[e] = C[e]; }
}

// cur <- A_est cur; residual partial per CTA (sum of ||cur' - fixed[nn]||).
__global__ void __launch_bounds__(256) pm_icp_apply_kernel(double *__restrict__ cur, int n1,
                                                           const double *__restrict__ fixed,
                                                           const int32_t *__restrict__ nn,
                                                           const double *__restrict__ a_est,
                                                           double *__restrict__ res_partial) {
    __shared__ double red[32];
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    double r = 0.0;
    if (i < n1) {
        const double x = cur[3 * i], y = cur[3 * i + 1], z = cur[3 * i + 2];
        const double nx = ((a_est[0] * x + a_est[1] * y) + a_est[2] * z) + a_est[3];
        const double ny = ((a_est[4] * x + a_est[5] * y) + a_est[6] * z) + a_est[7];
        const double nz = ((a_est[8] * x + a_est[9] * y) + a_est[10] * z) + a_est[11];
        cur[3 * i] = nx; cur[3 * i + 1] = ny; cur[3 * i + 2] = nz;
        const int j = nn[i];
        const double e0 = nx - fixed[3 * (size_t)j], e1 = ny - fixed[3 * (size_t)j + 1], e2 = nz - fixed[3 * (size_t)j + 2];
        r = sqrt(e0 * e0 + e1 * e1 + e2 * e2);
    }
    r = pm_block_sum(r, red);
    if (threadIdx.x == 0) res_partial[blockIdx.x] = r;
}

__global__ void __launch_bounds__(256) pm_icp_residual_kernel(const double *__restrict__ res_partial, int nblocks,
                                                              int n1, double *__restrict__ residuals) {
    __shared__ double red[32];
    const double *p = res_partial + (size_t)blockIdx.x * nblocks;
    double s = 0.0;
    for (int b = threadIdx.x; b < nblocks; b += blockDim.x) s += p[b];
    s = pm_block_sum(s, red);
    if (threadIdx.x == 0) residuals[blockIdx.x] = s / (double)n1;
}

__global__ void pm_icp_init_kernel(const double *__restrict__ moving, double *__restrict__ a_icp,
                                   double *__restrict__ shift) {
    if (threadIdx.x < 16) a_icp[threadIdx.x] = (threadIdx.x % 5 == 0) ? 1.0 : 0.0;
    if (threadIdx.x < 3) shift[threadIdx.x] = moving[threadIdx.x];
}

static inline size_t pm_align256(size_t x) { return (x + 255) & ~(size_t)255; }

static int pm_icp_grid_target(int n2) {      // cells along the longest axis: ~2 n2^(1/3), so occupied cells hold a few points
    int t = (int)ceil(2.0 * cbrt((double)(n2 > 1 ? n2 : 1)));
    if (t < 1) t = 1;
    if (t > 160) t = 160;
    return t;
}

static size_t pm_icp_max_cells(int n2) {
    const size_t t = (size_t)pm_icp_grid_target(n2) + 1;
    return t * t * t;
}

// byte offsets of the workspace of pm_icp, and its total size
struct PmIcpLayout {
    size_t cur, nn, partial, small, res_partial, grid, cell_start, cursor, cell_of, sorted_idx, sorted_pts, total;
};

static PmIcpLayout pm_icp_layout(int n1, int n2) {
    const size_t nb_nn = (size_t)(n1 + PM_ICP_PTS - 1) / PM_ICP_PTS;
    const size_t nb_res = (size_t)(n1 + PM_ICP_QPB - 1) / PM_ICP_QPB;
    const size_t max_cells = pm_icp_max_cells(n2);
    PmIcpLayout L;
    size_t o = 0;
    L.cur = o; o += pm_align256((size_t)n1 * 3 * sizeof(double));
    L.nn = o; o += pm_align256((size_t)n1 * sizeof(int32_t));
    L.partial = o; o += pm_align256((nb_nn + 2 * nb_res) * PM_ICP_NSUM * sizeof(double));   // ping-pong for the persistent kernel
    L.small = o; o += pm_align256(64 * sizeof(double));                                     // a_est, a_icp, shift
    L.res_partial = o; o += pm_align256(nb_res * sizeof(double) * 1024);                   // residual partials (<= 1024 iterations)
    // uniform grid over the fixed cloud
    L.grid = o; o += pm_align256(sizeof(PmIcpGrid));
    L.cell_start = o; o += pm_align256((max_cells + 1) * sizeof(int));
    L.cursor = o; o += pm_align256((max_cells + 1) * sizeof(int));
    L.cell_of = o; o += pm_align256((size_t)n2 * sizeof(int));
    L.sorted_idx = o; o += pm_align256((size_t)n2 * sizeof(int));
    L.sorted_pts = o; o += pm_align256((size_t)n2 * 3 * sizeof(double));
    L.total = o;
    return L;
}

extern "C" size_t pm_icp_workspace_bytes2(int n1, int n2) {
    if (n1 < 1 || n2 < 1) return 0;
    return pm_icp_layout(n1, n2).total;
}

extern "C" int pm_icp(const double *moving, int n1, const double *fixed, int n2, int iterations, int transform,
                      double *A_icp, double *residuals, int32_t *nn_out, void *workspace, size_t workspace_bytes,
                      void *stream) {
    PM_REQUIRE(moving && fixed && A_icp && workspace, "null pointer");
    PM_REQUIRE(n1 >= 1 && n2 >= 1, "need n1 >= 1 and n2 >= 1");
    PM_REQUIRE(transform == PM_TRANSFORM_AFFINE || transform == PM_TRANSFORM_SIMILAR, "unknown transform");
    PM_REQUIRE(iterations >= 0 && iterations <= 1024, "iterations must be 0..1024");
    const PmIcpLayout L = pm_icp_layout(n1, n2);
    if (workspace_bytes < L.total) {
        pm_set_error("pm_icp: workspace too small");
        return PM_ERR_WORKSPACE;
    }
    // the grid search pays off from a few hundred fixed points
    const bool use_grid = n2 >= 256 && !getenv("PM_ICP_BRUTE");
    cudaStream_t s = pm_stream(stream);
    const int nb_nn = (n1 + PM_ICP_PTS - 1) / PM_ICP_PTS, nb_ap = (n1 + 255) / 256;
    const int nb_pers = (n1 + PM_ICP_QPB - 1) / PM_ICP_QPB;
    char *w = (char *)workspace;
    double *cur = (double *)(w + L.cur);
    int32_t *nn = (int32_t *)(w + L.nn);
    double *partial = (double *)(w + L.partial);
    double *small = (double *)(w + L.small);
    double *res_partial = (double *)(w + L.res_partial);
    double *a_est = small, *a_icp = small + 16, *shift = small + 32;
    PmIcpGrid *grid = (PmIcpGrid *)(w + L.grid);
    int *cell_start = (int *)(w + L.cell_start), *cursor = (int *)(w + L.cursor);
    int *cell_of = (int *)(w + L.cell_of), *sorted_idx = (int *)(w + L.sorted_idx);
    double *sorted_pts = (double *)(w + L.sorted_pts);
    if (use_grid) {
        pm_icp_grid_setup_kernel<<<1, 1024, 0, s>>>(fixed, n2, pm_icp_grid_target(n2), grid, cell_start,
                                                    (int)pm_icp_max_cells(n2));
        pm_icp_cell_count_kernel<<<(n2 + 255) / 256, 256, 0, s>>>(fixed, n2, grid, cell_of, cell_start);
        pm_icp_cell_scan_kernel<<<1, 1024, 0, s>>>(grid, cell_start, cursor);
        pm_icp_cell_fill_kernel<<<(n2 + 255) / 256, 256, 0, s>>>(fixed, n2, cell_of, cursor, sorted_pts, sorted_idx);
        PM_LAUNCH_CHECK_N(4);
    }
    const int nb_grid = (n1 + PM_ICP_GPTS - 1) / PM_ICP_GPTS;
    if (use_grid && iterations > 0 && !getenv("PM_ICP_MULTI_LAUNCH")) {
        // whole loop in one cooperative launch when every CTA can be resident at once
        int dev = 0, sms = 0, per_sm = 0;
        PM_CUDA_TRY(cudaGetDevice(&dev));
        PM_CUDA_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
        PM_CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, pm_icp_persistent_kernel, PM_ICP_QPB * PM_ICP_LPQ, 0));
        if (nb_pers <= sms * per_sm) {
            double *a_out = a_icp;
            void *args[] = {(void *)&moving, (void *)&n1, (void *)&fixed, (void *)&iterations, (void *)&transform, (void *)&grid, (void *)&cell_start,
                            (void *)&sorted_pts, (void *)&sorted_idx, (void *)&nn, (void *)&partial, (void *)&res_partial,
                            (void *)&a_out};
            PM_CUDA_TRY(cudaLaunchCooperativeKernel((const void *)pm_icp_persistent_kernel, dim3(nb_pers),
                                                    dim3(PM_ICP_QPB * PM_ICP_LPQ), args, 0, s));
            PM_LAUNCH_CHECK();
            if (residuals) {
                pm_icp_residual_kernel<<<iterations, 256, 0, s>>>(res_partial, nb_pers, n1, residuals);
                PM_LAUNCH_CHECK();
            }
            PM_CUDA_TRY(cudaMemcpyAsync(A_icp, a_icp, 16 * sizeof(double), cudaMemcpyDeviceToDevice, s));
            if (nn_out) PM_CUDA_TRY(cudaMemcpyAsync(nn_out, nn, (size_t)n1 * sizeof(int32_t), cudaMemcpyDeviceToDevice, s));
            return PM_OK;
        }
    }
    PM_CUDA_TRY(cudaMemcpyAsync(cur, moving, (size_t)n1 * 3 * sizeof(double), cudaMemcpyDeviceToDevice, s));
    pm_icp_init_kernel<<<1, 32, 0, s>>>(moving, a_icp, shift);
    PM_LAUNCH_CHECK();
    for (int it = 0; it < iterations; ++it) {
        if (use_grid)
            pm_icp_nn_grid_kernel<<<nb_grid, PM_ICP_GPTS, 0, s>>>(cur, n1, fixed, grid, cell_start, sorted_pts, sorted_idx,
                                                                  shift, transform, nn, partial);
        else
            pm_icp_nn_kernel<<<nb_nn, PM_ICP_PTS * PM_ICP_SLICES, 0, s>>>(cur, n1, fixed, n2, shift, transform, nn, partial);
        pm_icp_solve_kernel<<<1, 256, 0, s>>>(partial, use_grid ? nb_grid : nb_nn, shift, fixed, transform, a_est, a_icp);
        pm_icp_apply_kernel<<<nb_ap, 256, 0, s>>>(cur, n1, fixed, nn, a_est, res_partial + (size_t)it * nb_ap);
    }
    PM_LAUNCH_CHECK_N(3 * iterations);
    if (residuals && iterations > 0) {
        pm_icp_residual_kernel<<<iterations, 256, 0, s>>>(res_partial, nb_ap, n1, residuals);
        PM_LAUNCH_CHECK();
    }
    PM_CUDA_TRY(cudaMemcpyAsync(A_icp, a_icp, 16 * sizeof(double), cudaMemcpyDeviceToDevice, s));
    if (nn_out && iterations > 0)
        PM_CUDA_TRY(cudaMemcpyAsync(nn_out, nn, (size_t)n1 * sizeof(int32_t), cudaMemcpyDeviceToDevice, s));
    return PM_OK;
}
