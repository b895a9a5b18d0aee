// pm_chi2.cu — K3: N1 x N2 chi^2 histogram-distance cost matrix, register-tiled packed FP32.
//
// Reference: platymatch/estimate_transform/shape_context.py:88-99 (get_unary_distance) evaluated for
// every (moving, fixed) pair by the double loops at platymatch/_dock_widget.py:547-602.
//   cost[i][j] = 0.5 * sum_k (a_ik - b_jk)^2 / (a_ik + b_jk),   bins with a == b skipped.
// The metric is not bilinear (one divide per bin pair), so it does not reduce to a dot product and
// there is no tensor-core formulation; it runs on the FP32 pipes + MUFU.RCP.
//
// Three things make it fast:
//  (1) structural zeros.  Shape-context histograms of shell-like clouds populate ~100 of the 360
//      bins each (r and theta are tied on a shell).  pm_chi2_operand records, per block of 16 and of
//      128 nuclei and per bin, whether any histogram of the block is non-empty (12 x u32 per block).
//      Each warp (16 rows x 128 columns of a CTA's tile) ORs / ANDs the masks of its 16 rows and of the
//      tile's 128 columns: bins empty on both sides are skipped (they contribute exactly 0), bins empty
//      on ONE side contribute the other side's value (a^2/a = a) and are folded into a per-row / per-column
//      sum, and only bins populated on both sides go through the full evaluation.
//  (2) two bins per reciprocal: t1/s1 + t2/s2 = (t1 s2 + t2 s1) / (s1 s2) halves the MUFU.RCP count
//      that bound the first version of this kernel (one MUFU per bin pair = 16/clk/SM).
//  (3) packed FP32 (FADD2/FMUL2/FFMA2, sm_100): two adjacent columns per instruction with the row
//      value as a scalar-broadcast operand -> 5 packed + 1 MUFU issue slots per 2 columns x 2 bins.
// Per (row, column, bin pair): 10 FP32 lane-operations + 1 MUFU, against 2 x 5 = 10 algorithmic FLOPs.
//
// Empty bins: both operands carry PM_CHI2_EPS (2^-60) instead of 0.  Then a == b == eps gives
// d = 0 exactly (contribution exactly 0, like the reference's "skip equal bins"), s = 2 eps and
// s1 * s2 >= 2^-118 stays a normal float, so the reciprocal is finite and no branch is needed;
// against a populated bin eps vanishes in the rounding (eps << ulp of any count / total).
// Identical histograms therefore give exactly 0.
#include <type_traits>
#include "pm_common.cuh"

#define PM_X2_TILE 128
#define PM_X2_KC 8           // bins per pipeline stage (4 pairs)
#define PM_X2_THREADS 256
#define PM_X2_NULL_BIN PM_NBINS   // operand row 360: all eps, pads the bin list to whole stages
#define PM_X2_MASK_WORDS 12
#define PM_X2_WROWS 16         // rows of one warp's tile = nuclei per fine mask block

typedef unsigned long long pm_f32x2;   // two floats in one 64-bit register pair: {lo, hi}

__device__ __forceinline__ pm_f32x2 pm_pack(float lo, float hi) {
    pm_f32x2 d;
    asm("mov.b64 %0, {%1, %2};" : "=l"(d) : "f"(lo), "f"(hi));
    return d;
}
__device__ __forceinline__ void pm_unpack(pm_f32x2 v, float &lo, float &hi) {
    asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ pm_f32x2 pm_add2(pm_f32x2 a, pm_f32x2 b) {
    pm_f32x2 d;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
    return d;
}
__device__ __forceinline__ pm_f32x2 pm_sub2(pm_f32x2 a, pm_f32x2 b) {
    pm_f32x2 d;
    asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
    return d;
}
__device__ __forceinline__ pm_f32x2 pm_mul2(pm_f32x2 a, pm_f32x2 b) {
    pm_f32x2 d;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
    return d;
}
__device__ __forceinline__ pm_f32x2 pm_fma2(pm_f32x2 a, pm_f32x2 b, pm_f32x2 c) {
    pm_f32x2 d;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
    return d;
}
__device__ __forceinline__ float pm_rcp(float x) {
    float r;
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
}
__device__ __forceinline__ pm_f32x2 pm_rcp2(pm_f32x2 p) {
    float lo, hi;
    pm_unpack(p, lo, hi);
    return pm_pack(pm_rcp(lo), pm_rcp(hi));
}

__device__ __forceinline__ void pm_cp_async16(void *smem, const void *gmem) {
    const unsigned s = (unsigned)__cvta_generic_to_shared(smem);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(s), "l"(gmem));
}
__device__ __forceinline__ void pm_cp_async16_l1(void *smem, const void *gmem) {   // through L1: read by 8 warps
    const unsigned s = (unsigned)__cvta_generic_to_shared(smem);
    asm volatile("cp.async.ca.shared.global [%0], [%1], 16;" ::"r"(s), "l"(gmem));
}
__device__ __forceinline__ void pm_cp_async_commit() { asm volatile("cp.async.commit_group;"); }
template <int N>
__device__ __forceinline__ void pm_cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N)); }

// ------------------------------------------------------------------------------------ operand
// counts [n][360] u32 -> out [361][ld] float32 bin-major (count / row total, empty -> eps, pad columns
// and the null row 360 -> eps), mask [ld/128][12] and fine [ld/16][12]: bit k of a block = some histogram
// of the block (128 / 16 nuclei) has a non-empty bin k.  grid (ld/128), block 256; coalesced through a
// shared-memory transpose.
// T = uint32_t: integer counts, normalised here by the row total; T = float: values used as given.
template <typename T>
__global__ void __launch_bounds__(256) pm_chi2_operand_kernel(const T *__restrict__ counts, int n,
                                                              float *__restrict__ out, int ld,
                                                              uint32_t *__restrict__ mask,
                                                              uint32_t *__restrict__ fine) {
    constexpr bool kCounts = sizeof(T) == sizeof(uint32_t) && !std::is_floating_point<T>::value;
    constexpr int kGroups = PM_X2_TILE / PM_X2_WROWS;
    __shared__ float tile[32][129];
    __shared__ float total[128];
    __shared__ uint32_t s_fine[kGroups][PM_X2_MASK_WORDS];
    const int i0 = blockIdx.x * 128;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;   // 8 warps
    if (threadIdx.x < kGroups * PM_X2_MASK_WORDS) (&s_fine[0][0])[threadIdx.x] = 0u;
    __syncthreads();
    for (int r = warp; r < 128 && kCounts; r += 8) {        // row totals: one warp per histogram
        const int i = i0 + r;
        uint32_t s = 0;
        if (i < n)
            for (int k = lane; k < PM_NBINS; k += 32) s += (uint32_t)counts[(size_t)i * PM_NBINS + k];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
        if (lane == 0) total[r] = (float)s;
    }
    __syncthreads();
    for (int k0 = 0; k0 < PM_NBINS; k0 += 32) {
        // load 128 histograms x 32 bins (lane = bin: 128-byte rows), mark non-empty bins
        for (int r = warp; r < 128; r += 8) {
            const int i = i0 + r, k = k0 + lane;
            float v = PM_CHI2_EPS;
            bool any = false;
            if (i < n && k < PM_NBINS) {
                const T c = counts[(size_t)i * PM_NBINS + k];
                if (c > (T)0) { v = kCounts ? (float)c / total[r] : (float)c; any = true; }   // count / total, one rounding
            }
            tile[lane][r] = v;
            const uint32_t word = __ballot_sync(0xffffffffu, any);   // bit = bin within this group of 32
            if (lane == 0 && word) atomicOr(&s_fine[r / PM_X2_WROWS][k0 >> 5], word);
        }
        __syncthreads();
        for (int kk = warp; kk < 32; kk += 8) {
            const int k = k0 + kk;
            if (k < PM_NBINS)
                for (int c = lane; c < 128; c += 32) out[(size_t)k * ld + i0 + c] = tile[kk][c];
        }
        __syncthreads();
    }
    for (int c = threadIdx.x; c < 128; c += 256) out[(size_t)PM_X2_NULL_BIN * ld + i0 + c] = PM_CHI2_EPS;
    if (threadIdx.x < kGroups * PM_X2_MASK_WORDS)
        fine[(size_t)blockIdx.x * kGroups * PM_X2_MASK_WORDS + threadIdx.x] = (&s_fine[0][0])[threadIdx.x];
    if (threadIdx.x < PM_X2_MASK_WORDS) {
        uint32_t m = 0u;
#pragma unroll
        for (int g = 0; g < kGroups; ++g) m |= s_fine[g][threadIdx.x];
        mask[(size_t)blockIdx.x * PM_X2_MASK_WORDS + threadIdx.x] = m;
    }
}

template <typename T>
static int pm_chi2_operand_launch(const T *counts, int n, float *out, int ld, uint32_t *mask, uint32_t *fine,
                                  void *stream) {
    pm_chi2_operand_kernel<T><<<ld / PM_X2_TILE, 256, 0, pm_stream(stream)>>>(counts, n, out, ld, mask, fine);
    PM_LAUNCH_CHECK();
    return PM_OK;
}

extern "C" int pm_chi2_operand(const uint32_t *counts, int n, float *out, int ld, uint32_t *mask, uint32_t *fine,
                               void *stream) {
    PM_REQUIRE(counts && out && mask && fine, "null pointer");
    PM_REQUIRE(n >= 1 && ld >= n && ld % PM_X2_TILE == 0, "need n >= 1 and ld = n rounded up to 128");
    return pm_chi2_operand_launch(counts, n, out, ld, mask, fine, stream);
}

extern "C" int pm_chi2_operand_f32(const float *hist, int n, float *out, int ld, uint32_t *mask, uint32_t *fine,
                                   void *stream) {
    PM_REQUIRE(hist && out && mask && fine, "null pointer");
    PM_REQUIRE(n >= 1 && ld >= n && ld % PM_X2_TILE == 0, "need n >= 1 and ld = n rounded up to 128");
    return pm_chi2_operand_launch(hist, n, out, ld, mask, fine, stream);
}

// ------------------------------------------------------------------------------------ cost
// Tiling: 128 x 128 outputs per CTA, 8 warps of 16 rows x 128 columns.  A thread holds an 8 x 8 register tile
// (rows ty*8..+7 of its warp's 16 with ty = lane / 16, columns tx*4..+3 and 64+tx*4..+3 with tx = lane % 16:
// LDS.128 operand reads without bank conflicts), accumulators as 8 x 4 packed column pairs.
// Each warp evaluates only the bins populated on both its own 16 rows (fine mask) and the tile's 128 columns
// (block mask), and stages their operand rows with 16-byte cp.async into a double-buffered ring of its own
// (8-bin stages): warps neither share a bin list nor wait for each other.  The 8 warps of a CTA read mostly the
// same column-side rows, so those copies go through L1.
#define PM_X2_WARPS (PM_X2_THREADS / 32)
#define PM_X2_WARP_FLOATS (2 * PM_X2_KC * (PM_X2_WROWS + PM_X2_TILE))
#define PM_X2_SMEM_BYTES (PM_X2_WARPS * PM_X2_WARP_FLOATS * (int)sizeof(float))

// Bins of a 360-bit mask whose words 0..11 are held by lanes 0..11 (0 in the other lanes), ascending, written to
// list by the whole warp; returns how many (all lanes).
__device__ __forceinline__ int pm_warp_bin_list(uint32_t word, unsigned short *list, int lane) {
    const int c = __popc(word);
    int incl = c;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += t;
    }
    for (int p = incl - c; word; word &= word - 1u) list[p++] = (unsigned short)(lane * 32 + __ffs(word) - 1);
    return __shfl_sync(0xffffffffu, incl, 31);
}

__global__ void __launch_bounds__(PM_X2_THREADS, 2)
pm_chi2_kernel(const float *__restrict__ a_t, int lda, const uint32_t *__restrict__ a_fine,
               const float *__restrict__ b_t, int ldb, const uint32_t *__restrict__ b_mask, int n2, int row_begin,
               int row_end, float *__restrict__ cost, int ldc) {
    extern __shared__ __align__(16) float x2_smem[];
    __shared__ unsigned short s_both[PM_X2_WARPS][PM_NBINS + PM_X2_KC], s_single[PM_X2_WARPS][PM_NBINS];
    __shared__ float s_rowsum[PM_X2_TILE], s_colsum[PM_X2_WARPS][PM_X2_TILE];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, tx = lane & 15, ty = lane >> 4;
    const int i0 = row_begin + blockIdx.y * PM_X2_TILE, j0 = blockIdx.x * PM_X2_TILE;
    const int r0 = i0 + warp * PM_X2_WROWS;                 // the warp's first operand row
    float(*As)[PM_X2_KC][PM_X2_WROWS] =
        reinterpret_cast<float(*)[PM_X2_KC][PM_X2_WROWS]>(x2_smem + warp * PM_X2_WARP_FLOATS);
    float(*Bs)[PM_X2_KC][PM_X2_TILE] = reinterpret_cast<float(*)[PM_X2_KC][PM_X2_TILE]>(
        x2_smem + warp * PM_X2_WARP_FLOATS + 2 * PM_X2_KC * PM_X2_WROWS);
    unsigned short *both = s_both[warp], *single = s_single[warp];

    // ordered bin lists: both sides populated / only the warp's rows / only the tile's columns
    uint32_t wa = 0u, wb = 0u;
    if (lane < PM_X2_MASK_WORDS) {
        wa = a_fine[(size_t)(r0 / PM_X2_WROWS) * PM_X2_MASK_WORDS + lane];
        wb = b_mask[(size_t)blockIdx.x * PM_X2_MASK_WORDS + lane];
    }
    const int n_both = pm_warp_bin_list(wa & wb, both, lane);
    const int n_aonly = pm_warp_bin_list(wa & ~wb, single, lane);
    const int n_bonly = pm_warp_bin_list(~wa & wb, single + n_aonly, lane);
    // two bins per reciprocal: an odd list ends with the null bin; the last stage is filled up with it, unevaluated
    const int n_eval = (n_both + 1) & ~1;
    const int n_stage = (n_eval + PM_X2_KC - 1) / PM_X2_KC;
    for (int q = n_both + lane; q < n_stage * PM_X2_KC; q += 32) both[q] = PM_X2_NULL_BIN;
    __syncwarp();

    // staging: a lane copies 4 of the 16 row-side values of bin lane / 4 and 4 column-side values of each bin
    const float *ag = a_t + r0 + (lane & 3) * 4;
    const float *bg = b_t + j0 + lane * 4;
    auto stage = [&](int st, int buf) {
        const unsigned short *ks = both + st * PM_X2_KC;
        pm_cp_async16(&As[buf][lane >> 2][(lane & 3) * 4], ag + (size_t)ks[lane >> 2] * lda);
#pragma unroll
        for (int e = 0; e < PM_X2_KC; ++e) pm_cp_async16_l1(&Bs[buf][e][lane * 4], bg + (size_t)ks[e] * ldb);
        pm_cp_async_commit();
    };
    if (n_stage > 0) stage(0, 0);

    // one-sided bins: (a - b)^2 / (a + b) with b empty is a; eps is taken off so that a == eps adds 0.
    // Row sums: lane tx sums row tx over every other bin; column sums: lane sums columns lane*4..+3.
    {
        float s = 0.0f;
        for (int q = ty; q < n_aonly; q += 2) s += a_t[(size_t)single[q] * lda + r0 + tx] - PM_CHI2_EPS;
        s += __shfl_xor_sync(0xffffffffu, s, 16);
        if (ty == 0) s_rowsum[warp * PM_X2_WROWS + tx] = s;
        float4 c = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
#pragma unroll 4
        for (int q = 0; q < n_bonly; ++q) {
            const float4 v = *reinterpret_cast<const float4 *>(bg + (size_t)single[n_aonly + q] * ldb);
            c.x += v.x - PM_CHI2_EPS;
            c.y += v.y - PM_CHI2_EPS;
            c.z += v.z - PM_CHI2_EPS;
            c.w += v.w - PM_CHI2_EPS;
        }
        *reinterpret_cast<float4 *>(&s_colsum[warp][lane * 4]) = c;
    }

    pm_f32x2 acc[8][4];
#pragma unroll
    for (int r = 0; r < 8; ++r)
#pragma unroll
        for (int c = 0; c < 4; ++c) acc[r][c] = 0ull;

    for (int st = 0; st < n_stage; ++st) {
        const int buf = st & 1;
        if (st + 1 < n_stage) {
            stage(st + 1, buf ^ 1);
            pm_cp_async_wait<1>();
        } else {
            pm_cp_async_wait<0>();
        }
        __syncwarp();
        const int n_here = n_eval - st * PM_X2_KC;   // bins of this stage to evaluate (< KC only in the last)
#pragma unroll
        for (int kp = 0; kp < PM_X2_KC; kp += 2) {
            if (kp >= n_here) break;
            const float4 a1_lo = *reinterpret_cast<const float4 *>(&As[buf][kp][ty * 8]);
            const float4 a1_hi = *reinterpret_cast<const float4 *>(&As[buf][kp][ty * 8 + 4]);
            const float4 a2_lo = *reinterpret_cast<const float4 *>(&As[buf][kp + 1][ty * 8]);
            const float4 a2_hi = *reinterpret_cast<const float4 *>(&As[buf][kp + 1][ty * 8 + 4]);
            const ulonglong2 b1_lo = *reinterpret_cast<const ulonglong2 *>(&Bs[buf][kp][tx * 4]);
            const ulonglong2 b1_hi = *reinterpret_cast<const ulonglong2 *>(&Bs[buf][kp][64 + tx * 4]);
            const ulonglong2 b2_lo = *reinterpret_cast<const ulonglong2 *>(&Bs[buf][kp + 1][tx * 4]);
            const ulonglong2 b2_hi = *reinterpret_cast<const ulonglong2 *>(&Bs[buf][kp + 1][64 + tx * 4]);
            const float a1[8] = {a1_lo.x, a1_lo.y, a1_lo.z, a1_lo.w, a1_hi.x, a1_hi.y, a1_hi.z, a1_hi.w};
            const float a2[8] = {a2_lo.x, a2_lo.y, a2_lo.z, a2_lo.w, a2_hi.x, a2_hi.y, a2_hi.z, a2_hi.w};
            const pm_f32x2 b1[4] = {b1_lo.x, b1_lo.y, b1_hi.x, b1_hi.y};
            const pm_f32x2 b2[4] = {b2_lo.x, b2_lo.y, b2_hi.x, b2_hi.y};
#pragma unroll
            for (int r = 0; r < 8; ++r) {
                const pm_f32x2 A1 = pm_pack(a1[r], a1[r]), A2 = pm_pack(a2[r], a2[r]);   // scalar-broadcast operand
#pragma unroll
                for (int c = 0; c < 4; ++c) {
                    const pm_f32x2 d1 = pm_sub2(A1, b1[c]), s1 = pm_add2(A1, b1[c]);
                    const pm_f32x2 d2 = pm_sub2(A2, b2[c]), s2 = pm_add2(A2, b2[c]);
                    const pm_f32x2 t1 = pm_mul2(d1, d1), t2 = pm_mul2(d2, d2);
                    const pm_f32x2 den = pm_mul2(s1, s2);
                    const pm_f32x2 num = pm_fma2(t2, s1, pm_mul2(t1, s2));
                    acc[r][c] = pm_fma2(num, pm_rcp2(den), acc[r][c]);
                }
            }
        }
        __syncwarp();
    }
    __syncwarp();   // s_rowsum / s_colsum of the warp visible

    const bool vec_ok = ((ldc & 3) == 0) && ((reinterpret_cast<size_t>(cost) & 15) == 0);
    float cs[8];
#pragma unroll
    for (int c = 0; c < 8; ++c) cs[c] = s_colsum[warp][(c < 4 ? 0 : 64) + tx * 4 + (c & 3)];
#pragma unroll
    for (int r = 0; r < 8; ++r) {
        const int lr = ty * 8 + r;
        const int i = r0 + lr;
        if (i >= row_end) continue;
        const float rs = s_rowsum[warp * PM_X2_WROWS + lr];
        float *crow = cost + (size_t)(i - row_begin) * ldc;
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            const int j = j0 + h * 64 + tx * 4;
            float v[4];
            pm_unpack(acc[r][h * 2 + 0], v[0], v[1]);
            pm_unpack(acc[r][h * 2 + 1], v[2], v[3]);
#pragma unroll
            for (int e = 0; e < 4; ++e) v[e] = 0.5f * (v[e] + (rs + cs[h * 4 + e]));
            if (vec_ok && j + 3 < n2) {
                *reinterpret_cast<float4 *>(crow + j) = make_float4(v[0], v[1], v[2], v[3]);
            } else {
#pragma unroll
                for (int e = 0; e < 4; ++e)
                    if (j + e < n2) crow[j + e] = v[e];
            }
        }
    }
}

extern "C" int pm_chi2_cost(const float *a_t, int lda, const uint32_t *a_fine, int n1, const float *b_t, int ldb,
                            const uint32_t *b_mask, int n2, int row_begin, int row_end, float *cost, int ldc,
                            void *stream) {
    PM_REQUIRE(a_t && b_t && a_fine && b_mask && cost, "null pointer");
    PM_REQUIRE(n1 >= 1 && n2 >= 1, "empty matrix");
    PM_REQUIRE(0 <= row_begin && row_begin <= row_end && row_end <= n1, "bad row range");
    PM_REQUIRE(ldc >= n2, "ldc < n2");
    // operand tiles are read without bounds checks: leading dimensions cover whole 128-blocks
    PM_REQUIRE(lda % PM_X2_TILE == 0 && ldb % PM_X2_TILE == 0 && lda >= n1 && ldb >= n2,
               "lda/ldb must be n1/n2 rounded up to 128 (pm_chi2_operand layout)");
    PM_REQUIRE((reinterpret_cast<size_t>(a_t) & 15) == 0 && (reinterpret_cast<size_t>(b_t) & 15) == 0,
               "operands must be 16-byte aligned");
    PM_REQUIRE(row_begin % PM_X2_TILE == 0, "row_begin must be a multiple of 128 (mask blocks)");
    const int rows = row_end - row_begin;
    if (rows == 0) return PM_OK;
    PM_CUDA_TRY(cudaFuncSetAttribute(pm_chi2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, PM_X2_SMEM_BYTES));
    const int tiles_y = (rows + PM_X2_TILE - 1) / PM_X2_TILE;
    dim3 grid((n2 + PM_X2_TILE - 1) / PM_X2_TILE, tiles_y);
    pm_chi2_kernel<<<grid, PM_X2_THREADS, PM_X2_SMEM_BYTES, pm_stream(stream)>>>(
        a_t, lda, a_fine, b_t, ldb, b_mask, n2, row_begin, row_end, cost, ldc);
    PM_LAUNCH_CHECK();
    return PM_OK;
}
