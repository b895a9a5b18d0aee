// pm_ransac.cu — K5: affine RANSAC hypothesis generation + scoring.
//
// Reference: platymatch/estimate_transform/shape_context.py:103-139 (do_ransac): per trial draw
// min_samples correspondences (:122), fit the affine on them (get_affine_transform,
// find_transform.py:4-17 = fixed_h @ pinv(moving_h)), apply it to all K moving points
// (apply_transform.py:3-17) and count ||fixed_k - predicted_k|| <= error (:131-135); keep the first
// strictly-better trial (:136-138).  A_best stays all-ones if no trial has an inlier (:120).
//
// float64 throughout (the 4x4 hypothesis feeds the final transform; inlier decisions are threshold
// tests on distances).  Three kernels: (1) one thread per trial solves the exact 4-point affine
// (Gauss-Jordan with partial pivoting; K > 4 samples go through the normal equations),
// (2) one warp per trial scores it against all correspondences staged through shared memory,
// (3) one CTA picks the maximum inlier count with the lowest trial index.
// Degenerate samples (numerically singular 4x4: coplanar points, flat 2-D data) get numpy's answer for them, the
// minimum-norm least-squares affine of pinv (pm_linalg.cuh), so planar clouds register like in the reference.
// transform = PM_TRANSFORM_SIMILAR fits Horn's similarity (get_similar_transform, find_transform.py:21-99) instead
// (shape_context.py:128-129).
#include "pm_common.cuh"

// ---- Philox4x32-10 counter RNG (device-side sampling when no index stream is given) ----
__device__ __forceinline__ void pm_philox_round(uint32_t &c0, uint32_t &c1, uint32_t &c2, uint32_t &c3, uint32_t k0,
                                                uint32_t k1) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
    c0 = hi1 ^ c1 ^ k0; c1 = lo1; c2 = hi0 ^ c3 ^ k1; c3 = lo0;
}
__device__ inline void pm_philox4(unsigned long long seed, uint32_t ctr0, uint32_t ctr1, uint32_t out[4]) {
    uint32_t c0 = ctr0, c1 = ctr1, c2 = 0x9E3779B9u, c3 = 0x85EBCA6Bu;
    uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        pm_philox_round(c0, c1, c2, c3, k0, k1);
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

#define PM_RANSAC_MAX_SAMPLES 16

// hyp[t][0:12] = rows 0..2 of A; hyp[t][12] = 1 if valid else 0
__global__ void pm_ransac_hypotheses(const double *__restrict__ moving, const double *__restrict__ fixed, int k,
                                     const int32_t *__restrict__ sample_idx, int trials, int min_samples,
                                     unsigned long long seed, int transform, double *__restrict__ hyp,
                                     int32_t *__restrict__ drawn_idx) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= trials) return;
    int idx[PM_RANSAC_MAX_SAMPLES];
    if (sample_idx) {
        for (int s = 0; s < min_samples; ++s) idx[s] = sample_idx[(size_t)t * min_samples + s];
    } else {
        uint32_t ctr = 0;
        for (int s = 0; s < min_samples;) {
            uint32_t r[4];
            pm_philox4(seed, (uint32_t)t, ctr++, r);
            for (int q = 0; q < 4 && s < min_samples; ++q) {
                const int cand = (int)(((unsigned long long)r[q] * (unsigned long long)k) >> 32);
                bool dup = false;
                for (int p = 0; p < s; ++p) dup |= (idx[p] == cand);
                if (!dup) idx[s++] = cand;
            }
        }
    }
    if (drawn_idx)
        for (int s = 0; s < min_samples; ++s) drawn_idx[(size_t)t * min_samples + s] = idx[s];
    double A[16];
    bool ok = true;
    for (int s = 0; s < min_samples; ++s) ok &= (idx[s] >= 0 && idx[s] < k);
    if (ok && transform == PM_TRANSFORM_SIMILAR) {
        // get_similar_transform (find_transform.py:21-99) on the sampled pairs: centroids, centred moments, Horn
        double cp[3] = {0.0, 0.0, 0.0}, cy[3] = {0.0, 0.0, 0.0};
        for (int s = 0; s < min_samples; ++s) {
            const double *m = moving + 3 * (size_t)idx[s], *f = fixed + 3 * (size_t)idx[s];
            for (int a = 0; a < 3; ++a) { cp[a] += m[a]; cy[a] += f[a]; }
        }
        for (int a = 0; a < 3; ++a) { cp[a] /= min_samples; cy[a] /= min_samples; }
        double S[9] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0}, spp = 0.0, syy = 0.0;
        for (int s = 0; s < min_samples; ++s) {
            const double *m = moving + 3 * (size_t)idx[s], *f = fixed + 3 * (size_t)idx[s];
            const double pc[3] = {m[0] - cp[0], m[1] - cp[1], m[2] - cp[2]};
            const double yc[3] = {f[0] - cy[0], f[1] - cy[1], f[2] - cy[2]};
            for (int a = 0; a < 3; ++a) {
                for (int b = 0; b < 3; ++b) S[a * 3 + b] += pc[a] * yc[b];
                spp += pc[a] * pc[a];
                syy += yc[a] * yc[a];
            }
        }
        pm_similar_from_moments(cp, cy, S, spp, syy, A);
    } else if (ok) {
        double M[16], R[12], X[12];
        bool solved = false;
        if (min_samples == 4) {
            // A M_h = F  with M_h columns = [m_s; 1]: exact solve
            for (int s = 0; s < 4; ++s) {
                const double *m = moving + 3 * (size_t)idx[s], *f = fixed + 3 * (size_t)idx[s];
                M[0 * 4 + s] = m[0]; M[1 * 4 + s] = m[1]; M[2 * 4 + s] = m[2]; M[3 * 4 + s] = 1.0;
                R[0 * 4 + s] = f[0]; R[1 * 4 + s] = f[1]; R[2 * 4 + s] = f[2];
            }
            solved = pm_solve_right_4x4(M, R, 3, X, 1e-13);
            if (solved) {
                for (int q = 0; q < 12; ++q) A[q] = X[q];
                A[12] = 0.0; A[13] = 0.0; A[14] = 0.0; A[15] = 1.0;
            }
        }
        if (!solved) {
            // more (or fewer) than 4 samples, or a degenerate (coplanar) 4-sample: least squares through the normal
            // equations, pinv's minimum-norm answer when they are singular (find_transform.py:17)
            const double *m0 = moving + 3 * (size_t)idx[0];
            const double shift[3] = {m0[0], m0[1], m0[2]};
            for (int q = 0; q < 16; ++q) M[q] = 0.0;
            for (int q = 0; q < 12; ++q) R[q] = 0.0;
            for (int s = 0; s < min_samples; ++s) {
                const double *m = moving + 3 * (size_t)idx[s], *f = fixed + 3 * (size_t)idx[s];
                const double mh[4] = {m[0] - shift[0], m[1] - shift[1], m[2] - shift[2], 1.0};
                for (int a = 0; a < 4; ++a)
                    for (int b = 0; b < 4; ++b) M[a * 4 + b] += mh[a] * mh[b];
                for (int a = 0; a < 3; ++a)
                    for (int b = 0; b < 4; ++b) R[a * 4 + b] += f[a] * mh[b];
            }
            pm_affine_from_normal_eq(M, R, shift, 1e-13, A);
        }
    }
    if (ok)
        for (int q = 0; q < 12; ++q) ok &= isfinite(A[q]);
    double *h = hyp + (size_t)t * 13;
    for (int q = 0; q < 12; ++q) h[q] = ok ? A[q] : 0.0;
    h[12] = ok ? 1.0 : 0.0;
}

#define PM_RANSAC_WARPS 8
#define PM_RANSAC_TILE 256

__global__ void __launch_bounds__(PM_RANSAC_WARPS * 32)
pm_ransac_score(const double *__restrict__ moving, const double *__restrict__ fixed, int k,
                const double *__restrict__ hyp, int trials, double error, int32_t *__restrict__ inliers) {
    __shared__ double sm[PM_RANSAC_TILE * 3], sf[PM_RANSAC_TILE * 3];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int t = blockIdx.x * PM_RANSAC_WARPS + warp;
    const bool live = t < trials;
    double a[12];
    bool valid = false;
    if (live) {
        const double *h = hyp + (size_t)t * 13;
#pragma unroll
        for (int q = 0; q < 12; ++q) a[q] = h[q];
        valid = h[12] != 0.0;
    }
    int cnt = 0;
    for (int p0 = 0; p0 < k; p0 += PM_RANSAC_TILE) {
        const int pn = min(PM_RANSAC_TILE, k - p0);
        __syncthreads();
        for (int q = threadIdx.x; q < pn * 3; q += blockDim.x) {
            sm[q] = moving[(size_t)p0 * 3 + q];
            sf[q] = fixed[(size_t)p0 * 3 + q];
        }
        __syncthreads();
        if (!valid) continue;
        for (int p = lane; p < pn; p += 32) {
            const double x = sm[3 * p], y = sm[3 * p + 1], z = sm[3 * p + 2];
            const double e0 = sf[3 * p] - (((a[0] * x + a[1] * y) + a[2] * z) + a[3]);
            const double e1 = sf[3 * p + 1] - (((a[4] * x + a[5] * y) + a[6] * z) + a[7]);
            const double e2 = sf[3 * p + 2] - (((a[8] * x + a[9] * y) + a[10] * z) + a[11]);
            const double d = sqrt(e0 * e0 + e1 * e1 + e2 * e2);
            cnt += (d <= error) ? 1 : 0;
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
    if (live && lane == 0) inliers[t] = cnt;
}

// first maximum (== first strictly-better trial); A = ones if the maximum is 0.
__global__ void __launch_bounds__(1024) pm_ransac_select(const int32_t *__restrict__ inliers,
                                                         const double *__restrict__ hyp, int trials,
                                                         double *__restrict__ best_A, int32_t *__restrict__ best_inliers,
                                                         int32_t *__restrict__ best_trial) {
    __shared__ long long red[32];
    // key: inliers in the high word, (INT_MAX - trial) in the low word -> max picks lowest trial
    long long key = -1;
    for (int t = threadIdx.x; t < trials; t += blockDim.x) {
        const long long kk = ((long long)inliers[t] << 32) | (long long)(0x7fffffff - t);
        key = kk > key ? kk : key;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const long long other = __shfl_xor_sync(0xffffffffu, key, o);
        key = other > key ? other : key;
    }
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = key;
    __syncthreads();
    if (threadIdx.x < 32) {
        key = red[threadIdx.x];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const long long other = __shfl_xor_sync(0xffffffffu, key, o);
            key = other > key ? other : key;
        }
        if (threadIdx.x == 0) {
            const int inl = (int)(key >> 32);
            const int t = 0x7fffffff - (int)(key & 0xffffffffLL);
            if (inl > 0) {
                const double *h = hyp + (size_t)t * 13;
                for (int q = 0; q < 12; ++q) best_A[q] = h[q];
                best_A[12] = 0.0; best_A[13] = 0.0; best_A[14] = 0.0; best_A[15] = 1.0;
                best_inliers[0] = inl;
                best_trial[0] = t;
            } else {
                for (int q = 0; q < 16; ++q) best_A[q] = 1.0;   // np.ones((4,4)) shape_context.py:120
                best_inliers[0] = 0;
                best_trial[0] = -1;
            }
        }
    }
}

extern "C" size_t pm_ransac_workspace_bytes(int trials) {
    if (trials < 1) return 0;
    return (size_t)trials * 13 * sizeof(double) + (size_t)trials * sizeof(int32_t) + 64;
}

extern "C" int pm_ransac(const double *moving, const double *fixed, int k, const int32_t *sample_idx, int trials,
                         int min_samples, double error, unsigned long long seed, int transform, double *best_A,
                         int32_t *best_inliers, int32_t *best_trial, int32_t *inliers_per_trial, void *workspace,
                         size_t workspace_bytes, void *stream) {
    PM_REQUIRE(moving && fixed && best_A && best_inliers && best_trial && workspace, "null pointer");
    PM_REQUIRE(trials >= 1, "need at least one trial");
    PM_REQUIRE(transform == PM_TRANSFORM_AFFINE || transform == PM_TRANSFORM_SIMILAR, "unknown transform");
    PM_REQUIRE(min_samples >= 1 && min_samples <= PM_RANSAC_MAX_SAMPLES, "min_samples must be 1..16");
    PM_REQUIRE(k >= min_samples, "fewer correspondences than samples");
    if (workspace_bytes < pm_ransac_workspace_bytes(trials)) {
        pm_set_error("pm_ransac: workspace too small");
        return PM_ERR_WORKSPACE;
    }
    cudaStream_t s = pm_stream(stream);
    double *hyp = (double *)workspace;
    int32_t *inl = inliers_per_trial ? inliers_per_trial : (int32_t *)(hyp + (size_t)trials * 13);
    pm_ransac_hypotheses<<<(trials + 127) / 128, 128, 0, s>>>(moving, fixed, k, sample_idx, trials, min_samples, seed,
                                                             transform, hyp, nullptr);
    PM_LAUNCH_CHECK();
    pm_ransac_score<<<(trials + PM_RANSAC_WARPS - 1) / PM_RANSAC_WARPS, PM_RANSAC_WARPS * 32, 0, s>>>(
        moving, fixed, k, hyp, trials, error, inl);
    PM_LAUNCH_CHECK();
    pm_ransac_select<<<1, 1024, 0, s>>>(inl, hyp, trials, best_A, best_inliers, best_trial);
    PM_LAUNCH_CHECK();
    return PM_OK;
}
