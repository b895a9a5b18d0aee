// pm_shape_context.cu — K2: 3D log-polar shape-context histograms for every nucleus, every
// orientation variant the reference tries, as a tiled O(N^2) kernel.
//
// Reference: platymatch/estimate_transform/shape_context.py:144-188 (get_unary: frames and the
// sc/sc2/sc3/sc4 variants), :61-84 (transform: neighbour coordinates in the local frame),
// :10-42 (get_shape_context: r, theta, phi) and :46-58 (get_bin_index: un-clamped linear bin).
//
// Layout / mapping
//   - one warp owns one query nucleus and a private 360-bin histogram per variant in shared memory;
//   - the point set is staged through shared memory in tiles (coalesced loads of the N x 3 float64
//     array), every lane bins one neighbour per step;
//   - lanes that hit the same bin are merged with __match_any_sync and the group leader adds the
//     group size (warp-aggregated update; the histogram is warp-private so no atomic is needed);
//   - bin DECISIONS are float64 with numpy's floor-division semantics, so the integer histograms are
//     comparable bit-for-bit with the reference; this file is compiled with -fmad=false so products
//     and sums round exactly as numpy's (no FMA contraction).
//   - r, theta are shared by all variants (the frames differ only by sign flips of x / y); phi is
//     re-evaluated per variant with the flipped signs, exactly as the reference does, so bin-edge
//     ties resolve identically instead of assuming the phi-bin permutation identity.
#include "pm_common.cuh"

#define PM_SC_WARPS 4
#define PM_SC_TILE 512

// numpy float64 `//` (npy_divmod): quotient from an exact fmod, snapped to the nearest integer.
__device__ __forceinline__ double pm_floor_divide(double a, double b) {
    const double mod = fmod(a, b);
    double div = (a - mod) / b;
    if (mod != 0.0) {
        if ((b < 0.0) != (mod < 0.0)) div -= 1.0;
    }
    if (div != 0.0) {
        double fl = floor(div);
        if (div - fl > 0.5) fl += 1.0;
        return fl;
    }
    return copysign(0.0, a / b);
}

__device__ __forceinline__ bool pm_near_edge(double v, double w) {
    const double mod = fmod(v, w);
    return fmin(mod, w - mod) <= 1.5e-14;
}

// Bin decision of one neighbour, the reference's way (float64 acos / atan2 / numpy floor-division,
// un-clamped index, NaN dropped): used for the few neighbours the fast classifier cannot decide.
template <int NVAR>
__device__ __noinline__ void pm_sc_exact_bins(double a, double b, double c, double mean_dist,
                                              const double *__restrict__ r_edges, int n_redges, int *bins,
                                              bool &tie) {
    const double w_bin = 3.14159265358979323846 / 6.0;        // np.pi / 6 == 2 * np.pi / 12
    const double two_pi = 2.0 * 3.14159265358979323846;
    const double r_ = sqrt(a * a + b * b + c * c);
    const double r = r_ / mean_dist;
    const double theta = acos(c / r_);
    const double ti = pm_floor_divide(theta, w_bin);
    int r_index = n_redges - 1;
    tie = pm_near_edge(theta, w_bin);
    for (int e = n_redges - 1; e >= 0; --e) {
        const double edge = r_edges[e];
        if (r < edge) r_index = e;
        tie |= fabs(r - edge) <= 1.5e-14 * edge;
    }
    const double base = (double)r_index * 72.0 + ti * 12.0;
#pragma unroll
    for (int v = 0; v < NVAR; ++v) {
        // sc (a,b)  sc2 (-a,-b)  sc3 (a,-b)  sc4 (-a,b)      (:170-185)
        const double av = (v == 1 || v == 3) ? -a : a;
        const double bv = (v == 1 || v == 2) ? -b : b;
        double phi = atan2(bv, av);
        if (phi < 0.0) phi = two_pi + phi;
        const double pi_ = pm_floor_divide(phi, w_bin);
        const double idx = base + pi_;
        bins[v] = (idx >= 0.0 && idx < (double)PM_NBINS) ? (int)idx : -1;   // NaN fails both -> dropped
        if (v == 0) tie |= pm_near_edge(phi, w_bin);
    }
}

// phi bin of variant v from the phi bin k of variant 0, valid strictly inside a sector:
// sc2 (-a,-b): phi + pi -> (k+6)%12;  sc3 (a,-b): 2pi - phi -> 11-k;  sc4 (-a,b): pi - phi -> (5-k)%12
__device__ __forceinline__ int pm_sc_variant_bin(int bin0, int v) {
    const int k = bin0 % 12, base = bin0 - k;
    const int kv = (v == 0) ? k : (v == 1) ? (k + 6) % 12 : (v == 2) ? 11 - k : (17 - k) % 12;
    return base + kv;
}

// Fast classifier.  Every bin boundary is a comparison of products (no sqrt, division or
// transcendental): ring: |n|^2 against (edge * mean_dist)^2; theta: c^2 against cos^2(k pi/6) |n|^2 and
// the sign of c; phi: |b| against tan(30 deg)|a| and tan(60 deg)|a| and the signs of a, b.  A neighbour
// closer than a relative 1e-11 to ANY boundary (rounding of the reference's float64 pipeline is ~1e-15)
// is not decided here but sent to pm_sc_exact_bins, so the histograms stay bit-identical to the
// reference, including its un-clamped overflow bins and NaN drops.
template <int NVAR>
__global__ void __launch_bounds__(PM_SC_WARPS * 32)
pm_shape_context_kernel(const double *__restrict__ pts, int n, const double *__restrict__ centroid,
                        const double *__restrict__ x0g, const double *__restrict__ mean_dist_p,
                        const double *__restrict__ r_edges, int n_redges, int row_begin, int row_end,
                        uint32_t *__restrict__ counts, uint32_t *__restrict__ dropped,
                        unsigned long long *__restrict__ edge_ties) {
    __shared__ uint32_t hist0[PM_SC_WARPS][PM_NBINS];            // fast-path neighbours, variant-0 bins
    __shared__ uint32_t histx[PM_SC_WARPS][NVAR][PM_NBINS];      // exact-path neighbours, per variant
    __shared__ double tile[PM_SC_TILE * 3];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int i = row_begin + blockIdx.x * PM_SC_WARPS + warp;      // query nucleus; output row i - row_begin
    const bool live = i < row_end;
    const int n_out = row_end - row_begin;
    const double mean_dist = mean_dist_p[0];
    const double BAND = 1e-11;
    // squared ring edges in absolute units with their undecided bands
    double e_lo[5], e_hi[5];
#pragma unroll
    for (int e = 0; e < 5; ++e) {
        const double edge = (e < n_redges) ? r_edges[e] * mean_dist : INFINITY;
        const double e2 = edge * edge;
        e_lo[e] = e2 * (1.0 - 4.0 * BAND);
        e_hi[e] = e2 * (1.0 + 4.0 * BAND);
    }

    for (int k = lane; k < PM_NBINS; k += 32) hist0[warp][k] = 0u;
    for (int k = lane; k < NVAR * PM_NBINS; k += 32) (&histx[warp][0][0])[k] = 0u;

    // local frame of the query nucleus (shape_context.py:169-175)
    double px = 0, py = 0, pz = 0, xv[3] = {0, 0, 0}, yv[3] = {0, 0, 0}, zv[3] = {0, 0, 0};
    if (live) {
        px = pts[3 * i]; py = pts[3 * i + 1]; pz = pts[3 * i + 2];
        const double d0 = px - centroid[0], d1 = py - centroid[1], d2 = pz - centroid[2];
        const double nz = sqrt(d0 * d0 + d1 * d1 + d2 * d2);
        zv[0] = d0 / nz; zv[1] = d1 / nz; zv[2] = d2 / nz;
        const double dot = x0g[0] * zv[0] + x0g[1] * zv[1] + x0g[2] * zv[2];
        xv[0] = x0g[0] - zv[0] * dot; xv[1] = x0g[1] - zv[1] * dot; xv[2] = x0g[2] - zv[2] * dot;
        const double nx = sqrt(xv[0] * xv[0] + xv[1] * xv[1] + xv[2] * xv[2]);
        xv[0] /= nx; xv[1] /= nx; xv[2] /= nx;
        yv[0] = zv[1] * xv[2] - zv[2] * xv[1];
        yv[1] = zv[2] * xv[0] - zv[0] * xv[2];
        yv[2] = zv[0] * xv[1] - zv[1] * xv[0];
        const double ny = sqrt(yv[0] * yv[0] + yv[1] * yv[1] + yv[2] * yv[2]);
        yv[0] /= ny; yv[1] /= ny; yv[2] /= ny;
    }
    // a frame with a non-finite axis (query at the centroid, ...) cannot be classified by products
    const bool frame_ok = isfinite(xv[0] + xv[1] + xv[2] + yv[0] + yv[1] + yv[2] + zv[0] + zv[1] + zv[2]);
    uint32_t drop[NVAR];
#pragma unroll
    for (int v = 0; v < NVAR; ++v) drop[v] = 0u;
    uint32_t ties = 0u;

    for (int t0 = 0; t0 < n; t0 += PM_SC_TILE) {
        const int tn = min(PM_SC_TILE, n - t0);
        __syncthreads();
        for (int k = threadIdx.x; k < tn * 3; k += blockDim.x) tile[k] = pts[(size_t)t0 * 3 + k];
        __syncthreads();
        if (!live) continue;
        for (int jb = 0; jb < tn; jb += 32) {
            const int jj = jb + lane;
            const bool valid = (jj < tn) && (t0 + jj != i);          // np.delete(detections, i) :168
            int bin0 = -1;
            bool exact = false;
            double a = 0, b = 0, c = 0;
            if (valid) {
                const double e0 = tile[3 * jj] - px, e1 = tile[3 * jj + 1] - py, e2 = tile[3 * jj + 2] - pz;
                a = e0 * xv[0] + e1 * xv[1] + e2 * xv[2];
                b = e0 * yv[0] + e1 * yv[1] + e2 * yv[2];
                c = e0 * zv[0] + e1 * zv[1] + e2 * zv[2];
                const double a2 = a * a, b2 = b * b, c2 = c * c;
                const double r2 = a2 + b2 + c2;
                bool ok = frame_ok && (r2 > 0.0) && (r2 < INFINITY);
                // ring: first edge with r < edge, else the last ring (open-ended)   (:49,53-56)
                int ring = n_redges - 1;
#pragma unroll
                for (int e = 4; e >= 0; --e) {
                    if (e < n_redges) {
                        if (r2 < e_lo[e]) ring = e;
                        else ok &= (r2 > e_hi[e]);
                    }
                }
                // theta = acos(c / |n|) // (pi/6): cos^2 thresholds 3/4, 1/4 and the sign of c
                const double q34 = 0.75 * r2, q14 = 0.25 * r2, qb = (2.0 * BAND) * r2;
                const bool big = c2 > q34 + qb, mid = c2 > q14 + qb;
                ok &= (big || c2 < q34 - qb) && (mid || c2 < q14 - qb) && (c2 > qb * BAND);   // c != 0 band
                ok &= !(c < 0.0 && c2 > r2 - qb);                                             // theta -> pi overflow
                const int tq = big ? 0 : mid ? 1 : 2;
                const int tbin = (c > 0.0) ? tq : 5 - tq;
                // phi = atan2(b, a) wrapped to [0, 2 pi) // (pi/6): 30-degree sectors
                const double fa = fabs(a), fb = fabs(b);
                const double t30 = 0.57735026918962576 * fa, t60 = 1.7320508075688772 * fa;
                const bool s60 = fb > t60 * (1.0 + BAND), s30 = fb > t30 * (1.0 + BAND);
                ok &= (s60 || fb < t60 * (1.0 - BAND)) && (s30 || fb < t30 * (1.0 - BAND));
                ok &= (fb > BAND * fa) && (fa > BAND * fb);                                   // on an axis
                const int pq = s60 ? 2 : s30 ? 1 : 0;
                const int pbin = (b > 0.0) ? ((a > 0.0) ? pq : 5 - pq) : ((a > 0.0) ? 11 - pq : 6 + pq);
                if (ok) bin0 = ring * 72 + tbin * 12 + pbin;
                else exact = true;
            }
            {   // fast-path neighbours: warp-aggregated update of the variant-0 histogram
                const unsigned voters = __ballot_sync(0xffffffffu, bin0 >= 0);
                if (bin0 >= 0) {
                    const unsigned peers = __match_any_sync(voters, bin0);
                    if (lane == __ffs(peers) - 1) hist0[warp][bin0] += __popc(peers);
                }
                __syncwarp();
            }
            if (__any_sync(0xffffffffu, exact)) {
                int bins[NVAR];
#pragma unroll
                for (int v = 0; v < NVAR; ++v) bins[v] = -1;
                if (exact) {
                    bool tie;
                    pm_sc_exact_bins<NVAR>(a, b, c, mean_dist, r_edges, n_redges, bins, tie);
                    ties += tie ? 1u : 0u;
#pragma unroll
                    for (int v = 0; v < NVAR; ++v)
                        if (bins[v] < 0) ++drop[v];
                }
#pragma unroll
                for (int v = 0; v < NVAR; ++v) {
                    const unsigned voters = __ballot_sync(0xffffffffu, bins[v] >= 0);
                    if (bins[v] >= 0) {
                        const unsigned peers = __match_any_sync(voters, bins[v]);
                        if (lane == __ffs(peers) - 1) histx[warp][v][bins[v]] += __popc(peers);
                    }
                    __syncwarp();
                }
            }
        }
    }
    __syncwarp();
    if (!live) return;
#pragma unroll
    for (int v = 0; v < NVAR; ++v) {
        uint32_t *dst = counts + ((size_t)v * n_out + (i - row_begin)) * PM_NBINS;
        // variant v of a fast-path neighbour sits in the phi-permuted bin (exactly, away from sector edges)
        for (int k = lane; k < PM_NBINS; k += 32) dst[pm_sc_variant_bin(k, v)] = hist0[warp][k];
        __syncwarp();
        for (int k = lane; k < PM_NBINS; k += 32)
            if (histx[warp][v][k]) dst[k] += histx[warp][v][k];
        uint32_t d = drop[v];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) d += __shfl_xor_sync(0xffffffffu, d, o);
        if (lane == 0 && dropped) dropped[(size_t)v * n_out + (i - row_begin)] = d;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) ties += __shfl_xor_sync(0xffffffffu, ties, o);
    if (lane == 0 && edge_ties && ties) atomicAdd(edge_ties, (unsigned long long)ties);
}

extern "C" int pm_shape_context_hist_rows(const double *pts, int n, const double *centroid, const double *x0,
                                          const double *mean_dist, const double *r_edges, int n_redges,
                                          int n_variants, int row_begin, int row_end, uint32_t *counts,
                                          uint32_t *dropped, unsigned long long *edge_ties, void *stream) {
    PM_REQUIRE(pts && centroid && x0 && mean_dist && r_edges && counts, "null pointer");
    PM_REQUIRE(n >= 2, "need at least 2 points");
    PM_REQUIRE(n_redges >= 1 && n_redges <= 5, "n_redges must be 1..5 (5 rings x 72 = 360 bins)");
    PM_REQUIRE(n_variants == 1 || n_variants == 2 || n_variants == 4, "n_variants must be 1, 2 or 4");
    PM_REQUIRE(row_begin >= 0 && row_begin <= row_end && row_end <= n, "need 0 <= row_begin <= row_end <= n");
    if (row_end == row_begin) return PM_OK;
    const int blocks = (row_end - row_begin + PM_SC_WARPS - 1) / PM_SC_WARPS;
    cudaStream_t s = pm_stream(stream);
    if (n_variants == 1)
        pm_shape_context_kernel<1><<<blocks, PM_SC_WARPS * 32, 0, s>>>(pts, n, centroid, x0, mean_dist, r_edges,
                                                                     n_redges, row_begin, row_end, counts, dropped, edge_ties);
    else if (n_variants == 2)
        pm_shape_context_kernel<2><<<blocks, PM_SC_WARPS * 32, 0, s>>>(pts, n, centroid, x0, mean_dist, r_edges,
                                                                     n_redges, row_begin, row_end, counts, dropped, edge_ties);
    else
        pm_shape_context_kernel<4><<<blocks, PM_SC_WARPS * 32, 0, s>>>(pts, n, centroid, x0, mean_dist, r_edges,
                                                                     n_redges, row_begin, row_end, counts, dropped, edge_ties);
    PM_LAUNCH_CHECK();
    return PM_OK;
}
