// pm_lap.cu — K4: exact rectangular linear sum assignment (min), nr <= nc, on the GPU.
//
// Replaces scipy.optimize.linear_sum_assignment at platymatch/_dock_widget.py:604-611 (third-party
// C++ in the reference: modified Jonker-Volgenant / Crouse 2016 shortest augmenting paths).
// Same optimum (equal total cost; identical assignment where the optimum is unique), different
// schedule, built for the GPU:
//
//  Phase 1 (default, "sparse asynchronous auction") — see the block comment above pm_ls_auction_kernel:
//    epsilon = 0 bidding over certified per-row candidate lists, 32 independent warps per matrix,
//    prices in shared memory, no barriers.
//  Phase 1 (fallback for column counts whose prices do not fit in shared memory, algorithm = 2) —
//    parallel bidding with epsilon = 0 (all SMs).  Every free row scans its cost row against
//    the column prices v and bids for its best column j1 with increment gamma = w2 - w1 (second best
//    minus best reduced value).  Per column the largest increment wins (ties: lowest row), the price
//    drops by gamma and the previous owner is released.  With epsilon = 0 every assigned edge stays
//    an exact arg-min of its row (prices only fall), so complementary slackness holds EXACTLY and
//    (u, v, matching) is a valid warm start for phase 2 at any time; rows whose bid would be a
//    zero-increment steal simply wait for phase 2 (this is where epsilon = 0 auctions stall).
//  Phase 2 — shortest augmenting paths for the remaining free rows (one CTA per matrix, float64
//    duals, Dijkstra over reduced costs).  Each thread owns 8 columns whose tentative distance d and
//    price v live in registers; one step = one coalesced cost-row load + one block arg-min.
//    Unassigned columns keep v = 0 (rectangular dual feasibility), exactly as in Crouse's algorithm.
//
// Costs are the float32 matrix produced by K3; duals, distances and the total are float64, so the
// result is optimal for the matrix given (up to float64 rounding, like scipy on the same values).
#include <limits.h>
#include <stdlib.h>
#include <cooperative_groups.h>
#include "pm_common.cuh"

namespace cg = cooperative_groups;

// squared (dummy rows + eps-scaling) when nc - nr <= this fraction of nc; measured crossover at 8k, profiles/r2_lap_slack.txt
#define PM_LAP_SQUARE_SLACK_DEFAULT 0.02
// eps-scaling schedule of a squared problem (DESIGN §4 K4): the first eps is this fraction of the matrix' cost scale,
// divided by PM_LAP_EPS_THETA from phase to phase, over PM_LAP_EPS_PHASES phases
#define PM_LAP_EPS0 (1.0 / 16.0)
#define PM_LAP_EPS_THETA 8.0
#define PM_LAP_EPS_PHASES 6
// an eps phase stops carrying displaced rows once this few warps are still bidding; measured, profiles/r2_lap_eps_truncation.txt
#define PM_LAP_EPS_STOP_LIVE 3
#define PM_LAP_BID_THREADS 1024
#define PM_LAP_CPT 8
#define PM_LAP_MAX_THREADS 1024

struct __align__(16) PmLsCell { double price; unsigned owner; unsigned pad; };

struct PmLapView {
    const float *cost;      // [nr][ldc]
    double *u, *v;          // [nr], [nc]
    int32_t *row4col;       // [nc]
    int32_t *col4row;       // [nr]  (workspace; rows >= nr_real are dummy rows; exported to the caller at the end)
    int32_t *col4row_out;   // [nr_real] caller's output buffer
    int32_t *bid_col;       // [nr]
    double *bid_gamma;      // [nr]
    unsigned long long *colbest;  // [nc] winning bid key of the round (0 = no bid)
    int32_t *free_lists;    // [3][nr] rotating free-row lists
    int32_t *counters;      // [0..2] list counts, [3] bid rounds run, [4] status
    int32_t *lcol;          // [nr][PM_LS_K] candidate columns (-1 = empty slot)
    float *lcost;           // [nr][PM_LS_K] their costs
    double *tau;            // [nr] every column outside the list has c - v >= tau, forever
    double *width;          // [nr] value range the list covered when it was built (refresh window)
    unsigned short *ring;   // [ring_cap] ring of displaced rows when it does not fit in shared memory (tail kernel)
    unsigned *ring32;       // [ring_cap] ring of displaced rows of the bulk kernel
    struct PmLsCell *cell;  // [nc] {price, owner} of the bulk kernel
    long long *stats;       // [PM_LAP_STATS] or null
    double *total;
};

static inline size_t pm_lap_align(size_t x) { return (x + 255) & ~(size_t)255; }

#define PM_LS_K 128          // candidate-list slots per row: 32 lanes x 4
// per-matrix int32 counters of the bulk auction kernel (PmLapView::counters)
#define PM_LS_CTR_FRESH 5
#define PM_LS_CTR_HEAD 6
#define PM_LS_CTR_TAIL 7
#define PM_LS_CTR_LIVE 8
#define PM_LS_CTR_BIDS 9
#define PM_LS_CTR_RETRIES 10
#define PM_LS_CTR_DROPPED 11
#define PM_LS_CTR_REFRESHES 12

struct PmLapLayout {
    size_t col4row, u, v, row4col, bid_col, bid_gamma, colbest, free_lists, counters, lcol, lcost, tau, width, ring, ring32, cell, per_item;
};

static unsigned pm_ls_ring_cap(int nr) {   // power of two >= nr: the ring can hold every row at once
    unsigned c = 1;
    while (c < (unsigned)nr) c <<= 1;
    return c;
}

static PmLapLayout pm_lap_layout(int nr, int nc) {
    PmLapLayout L;
    size_t o = 0;
    L.col4row = o; o += pm_lap_align((size_t)nr * 4);
    L.u = o; o += pm_lap_align((size_t)nr * 8);
    L.v = o; o += pm_lap_align((size_t)nc * 8);
    L.row4col = o; o += pm_lap_align((size_t)nc * 4);
    L.bid_col = o; o += pm_lap_align((size_t)nr * 4);
    L.bid_gamma = o; o += pm_lap_align((size_t)nr * 8);
    L.colbest = o; o += pm_lap_align((size_t)nc * 8);
    L.free_lists = o; o += pm_lap_align((size_t)nr * 4 * 3);
    L.counters = o; o += pm_lap_align(16 * 4);
    L.lcol = o; o += pm_lap_align((size_t)nr * PM_LS_K * 4);
    L.lcost = o; o += pm_lap_align((size_t)nr * PM_LS_K * 4);
    L.tau = o; o += pm_lap_align((size_t)nr * 8);
    L.width = o; o += pm_lap_align((size_t)nr * 8);
    L.ring = o; o += pm_lap_align((size_t)pm_ls_ring_cap(nr) * 2);
    L.ring32 = o; o += pm_lap_align((size_t)pm_ls_ring_cap(nr) * 4);
    L.cell = o; o += pm_lap_align((size_t)nc * 16);
    L.per_item = o;
    return L;
}

struct PmLapBatch {   // passed by value to kernels
    const float *cost; size_t cost_stride; int nr, nc, ncp, ldc;
    int nr_real;            // rows of the caller's matrix; rows nr_real..nr-1 are DUMMY rows (all costs 0) that make a
                            // problem with few slack columns square (nr == nc), see pm_lap_solve
    const float *zero_row;  // [ldc] zeros: the cost row of every dummy row
    char *ws; PmLapLayout L;
    int32_t *col4row; long long *stats; double *total;
    int32_t *progress;   // [2] assignments made in the current / previous bidding round
    long long max_bids;       // sparse auction: bid budget per warp of the bulk kernel
    long long max_bids_tail;  // ... and of the tail kernel
    int stop_live;       // sparse auction: stop carrying displaced rows once this few warps are still bidding
    int bulk_stop_live;  // bulk kernel: stop once this few warps (of bulk_warps) are still bidding
    int bulk_warps;
    int bulk_patience;   // bulk kernel: polls (200 ns apart) a warp waits for its ring slot before it leaves
    unsigned ring_cap;   // sparse auction: ticket ring capacity (power of two >= nr)
    int ring_in_smem;
    // eps-scaling phases (problems without slack columns): increment = certified gap + eps, eps = eps_factor x the
    // matrix' own cost scale (mean candidate-list width, accumulated by pm_ls_build_lists into scale[0..1] per matrix)
    double eps_factor;   // 0 = exact phase (eps = 0)
    double *scale;       // [batch][2]: sum of list widths, number of rows that contributed
    int path;            // PM_LAP_PATH_* bits of this solve, reported by the finishing kernel as PM_LAP_STAT_PATH
};

// cost row of row i (dummy rows share one row of zeros)
__device__ __forceinline__ const float *pm_lap_row(const float *cost, const PmLapBatch &B, int i) {
    return i < B.nr_real ? cost + (size_t)i * B.ldc : B.zero_row;
}

__device__ __forceinline__ PmLapView pm_lap_view(const PmLapBatch &B, int b) {
    PmLapView V;
    char *w = B.ws + (size_t)b * B.L.per_item;
    V.cost = B.cost + (size_t)b * B.cost_stride;
    V.u = (double *)(w + B.L.u); V.v = (double *)(w + B.L.v);
    V.row4col = (int32_t *)(w + B.L.row4col);
    V.col4row = (int32_t *)(w + B.L.col4row);
    V.col4row_out = B.col4row + (size_t)b * B.nr_real;
    V.bid_col = (int32_t *)(w + B.L.bid_col); V.bid_gamma = (double *)(w + B.L.bid_gamma);
    V.colbest = (unsigned long long *)(w + B.L.colbest);
    V.free_lists = (int32_t *)(w + B.L.free_lists);
    V.counters = (int32_t *)(w + B.L.counters);
    V.lcol = (int32_t *)(w + B.L.lcol); V.lcost = (float *)(w + B.L.lcost); V.tau = (double *)(w + B.L.tau);
    V.width = (double *)(w + B.L.width); V.ring = (unsigned short *)(w + B.L.ring);
    V.ring32 = (unsigned *)(w + B.L.ring32); V.cell = (PmLsCell *)(w + B.L.cell);
    V.stats = B.stats ? B.stats + (size_t)b * PM_LAP_STATS : nullptr;
    V.total = B.total + b;
    return V;
}

// ------------------------------------------------------------------------------------- init
__global__ void pm_lap_init_kernel(PmLapBatch B) {
    const PmLapView V = pm_lap_view(B, blockIdx.y);
    const int t = blockIdx.x * blockDim.x + threadIdx.x, stride = gridDim.x * blockDim.x;
    for (int i = t; i < B.nr; i += stride) { V.u[i] = 0.0; V.col4row[i] = -1; V.free_lists[i] = i; V.bid_col[i] = -1; }
    for (int j = t; j < B.ncp; j += stride) {
        V.v[j] = 0.0; V.row4col[j] = -1; V.colbest[j] = 0ull;
        V.cell[j].price = 0.0; V.cell[j].owner = 0xFFFFFFFFu; V.cell[j].pad = 0u;
    }
    for (unsigned q = t; q < B.ring_cap; q += stride) V.ring32[q] = 0xFFFFFFFFu;
    if (blockIdx.y == 0)
        for (int j = t; j < B.ncp + 32; j += stride) const_cast<float *>(B.zero_row)[j] = 0.0f;
    if (t == 0) {
        V.counters[0] = B.nr; V.counters[1] = 0; V.counters[2] = 0; V.counters[3] = 0; V.counters[4] = 0;
        for (int k = 5; k < 16; ++k) V.counters[k] = 0;
        V.counters[PM_LS_CTR_LIVE] = B.bulk_warps;
        B.progress[0] = 0; B.progress[1] = 0;
        B.scale[2 * blockIdx.y] = 0.0; B.scale[2 * blockIdx.y + 1] = 0.0;
        if (V.stats) for (int k = 0; k < PM_LAP_STATS; ++k) V.stats[k] = 0;
    }
}

// ------------------------------------------------------------------------------------- phase 1
struct PmBid { double w1, w2; int j1; };

__device__ __forceinline__ void pm_bid_push(PmBid &a, double w, int j) {
    if (w < a.w1) { a.w2 = a.w1; a.w1 = w; a.j1 = j; }
    else if (w < a.w2) a.w2 = w;
}
__device__ __forceinline__ void pm_bid_merge(PmBid &a, double w1, double w2, int j1) {
    if (w1 < a.w1 || (w1 == a.w1 && j1 < a.j1)) { a.w2 = fmin(a.w1, w2); a.w1 = w1; a.j1 = j1; }
    else a.w2 = fmin(a.w2, w1);
}

// Winner selection key of a bid: float32 image of the increment (monotone in gamma) in the high
// word, ~row in the low word -> atomicMax picks the largest increment, ties to the lowest row.
// ANY bidder may win without hurting exactness: the winner lowers the price by its OWN float64
// gamma, which makes its edge tight against its own second-best column.
__device__ __forceinline__ unsigned long long pm_bid_key(double gamma, int row) {
    return ((unsigned long long)__float_as_uint(__double2float_rd(gamma)) << 32) |
           (unsigned long long)(0xffffffffu - (unsigned)row);
}

// Persistent cooperative kernel: all rounds of the parallel bidding for all matrices of the batch.
// Per round: (A) every free row is scanned by one CTA and bids; grid barrier; (B) winners take
// their columns, everybody else goes to the next free list; grid barrier.  Three rotating list
// counters (current / next / stale-to-zero) avoid any reset race.  Stops when no row is free, when a
// round assigns nothing (only zero-increment steals left), or after max_rounds.
__global__ void __launch_bounds__(PM_LAP_BID_THREADS) pm_lap_bid_persistent(PmLapBatch B, int batch, int max_rounds) {
    cg::grid_group grid = cg::this_grid();
    __shared__ double s_w1[PM_LAP_BID_THREADS / 32], s_w2[PM_LAP_BID_THREADS / 32];
    __shared__ int s_j1[PM_LAP_BID_THREADS / 32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int gtid = blockIdx.x * blockDim.x + threadIdx.x, gthreads = gridDim.x * blockDim.x;
    int round = 0;
    for (; round < max_rounds; ++round) {
        const int cur = round % 3, nxt = (round + 1) % 3, old = (round + 2) % 3;
        // ---- phase A: bids.  Work item = (matrix b, position idx in its free list)
        int total_free = 0;
        for (int b = 0; b < batch; ++b) {
            const PmLapView V = pm_lap_view(B, b);
            const int nfree = __ldcg(&V.counters[cur]);
            const int32_t *list = V.free_lists + (size_t)cur * B.nr;
            // CTA c takes items (c - total_free) mod gridDim of this matrix, so matrices interleave over CTAs
            int first = (int)blockIdx.x - (total_free % (int)gridDim.x);
            if (first < 0) first += gridDim.x;
            for (int idx = first; idx < nfree; idx += gridDim.x) {
                const int i = __ldcg(&list[idx]);
                const float *ci = pm_lap_row(V.cost, B, i);
                PmBid bid = {INFINITY, INFINITY, INT_MAX};
                // two float4 sweeps per trip so that all loads of a thread are in flight together
                for (int j0 = threadIdx.x * 4; j0 < B.nc; j0 += PM_LAP_BID_THREADS * 8) {
                    const int j1 = j0 + PM_LAP_BID_THREADS * 4;
                    const bool second = j1 < B.nc;
                    const float4 c4 = *reinterpret_cast<const float4 *>(ci + j0);   // ldc % 4 == 0, pad readable
                    const double2 va = __ldcg(reinterpret_cast<const double2 *>(V.v + j0));
                    const double2 vb = __ldcg(reinterpret_cast<const double2 *>(V.v + j0 + 2));
                    float4 d4 = make_float4(0.f, 0.f, 0.f, 0.f);
                    double2 wa = make_double2(0.0, 0.0), wb = make_double2(0.0, 0.0);
                    if (second) {
                        d4 = *reinterpret_cast<const float4 *>(ci + j1);
                        wa = __ldcg(reinterpret_cast<const double2 *>(V.v + j1));
                        wb = __ldcg(reinterpret_cast<const double2 *>(V.v + j1 + 2));
                    }
                    if (j0 + 0 < B.nc) pm_bid_push(bid, (double)c4.x - va.x, j0 + 0);
                    if (j0 + 1 < B.nc) pm_bid_push(bid, (double)c4.y - va.y, j0 + 1);
                    if (j0 + 2 < B.nc) pm_bid_push(bid, (double)c4.z - vb.x, j0 + 2);
                    if (j0 + 3 < B.nc) pm_bid_push(bid, (double)c4.w - vb.y, j0 + 3);
                    if (second) {
                        if (j1 + 0 < B.nc) pm_bid_push(bid, (double)d4.x - wa.x, j1 + 0);
                        if (j1 + 1 < B.nc) pm_bid_push(bid, (double)d4.y - wa.y, j1 + 1);
                        if (j1 + 2 < B.nc) pm_bid_push(bid, (double)d4.z - wb.x, j1 + 2);
                        if (j1 + 3 < B.nc) pm_bid_push(bid, (double)d4.w - wb.y, j1 + 3);
                    }
                }
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) {
                    const double ow1 = __shfl_xor_sync(0xffffffffu, bid.w1, o), ow2 = __shfl_xor_sync(0xffffffffu, bid.w2, o);
                    const int oj = __shfl_xor_sync(0xffffffffu, bid.j1, o);
                    pm_bid_merge(bid, ow1, ow2, oj);
                }
                __syncthreads();
                if (lane == 0) { s_w1[warp] = bid.w1; s_w2[warp] = bid.w2; s_j1[warp] = bid.j1; }
                __syncthreads();
                if (threadIdx.x == 0) {
                    PmBid tot = {s_w1[0], s_w2[0], s_j1[0]};
                    for (int w = 1; w < PM_LAP_BID_THREADS / 32; ++w) pm_bid_merge(tot, s_w1[w], s_w2[w], s_j1[w]);
                    // nc == 1: no second best; an unowned single column is simply taken with gamma 0
                    double gamma = (tot.w2 == INFINITY) ? 0.0 : tot.w2 - tot.w1;
                    if (!(gamma > 0.0)) gamma = 0.0;
                    int j1 = tot.j1;
                    if (j1 == INT_MAX || tot.w1 == INFINITY) j1 = -1;                    // all-inf row: phase 2 reports it
                    else if (gamma == 0.0 && __ldcg(&V.row4col[j1]) >= 0) j1 = -1;       // zero-increment steal: wait
                    V.bid_col[i] = j1;
                    V.bid_gamma[i] = gamma;
                    if (j1 >= 0) atomicMax(&V.colbest[j1], pm_bid_key(gamma, i));
                }
            }
            total_free += nfree;
            if (gtid == 0) V.counters[old] = 0;        // consumed in the previous round
        }
        if (gtid == 0) B.progress[round & 1] = 0;
        if (total_free == 0) break;                    // uniform: every CTA read the same counters
        grid.sync();
        // ---- phase B: winners take their columns; everybody else (and displaced owners) -> next list
        for (int b = 0; b < batch; ++b) {
            const PmLapView V = pm_lap_view(B, b);
            const int nfree = __ldcg(&V.counters[cur]);
            const int32_t *list = V.free_lists + (size_t)cur * B.nr;
            int32_t *next = V.free_lists + (size_t)nxt * B.nr;
            int32_t *next_count = &V.counters[nxt];
            for (int idx = gtid; idx < nfree; idx += gthreads) {
                const int i = __ldcg(&list[idx]), j = __ldcg(&V.bid_col[i]);
                bool won = false;
                if (j >= 0) {
                    const double gamma = __ldcg(&V.bid_gamma[i]);
                    won = __ldcg(&V.colbest[j]) == pm_bid_key(gamma, i);
                    if (won) {
                        const int prev = __ldcg(&V.row4col[j]);
                        const double vj = __ldcg(&V.v[j]) - gamma;
                        V.v[j] = vj;
                        V.u[i] = (double)pm_lap_row(V.cost, B, i)[j] - vj;
                        V.row4col[j] = i;
                        V.col4row[i] = j;
                        V.colbest[j] = 0ull;
                        if (prev >= 0) { V.col4row[prev] = -1; next[atomicAdd(next_count, 1)] = prev; }
                        atomicAdd(&B.progress[round & 1], 1);
                    }
                }
                if (!won) next[atomicAdd(next_count, 1)] = i;
            }
        }
        grid.sync();
        // every bid-on column has exactly one winner, which cleared its key above: nothing left to reset
        if (__ldcg(&B.progress[round & 1]) == 0) { ++round; break; }     // stalled: only zero-increment steals left
    }
    if (gtid == 0)
        for (int b = 0; b < batch; ++b) pm_lap_view(B, b).counters[3] = round;
}

// ------------------------------------------------------------------------------------- phase 1 (sparse, asynchronous)
// Exact epsilon = 0 auction over *certified candidate lists*.
//
// Lists.  For every row i a warp scans the dense cost row once; each lane keeps the 5 smallest
// reduced values c_ij - v_j of the columns it visited.  tau_i = the smallest "5th value" over the 32
// lanes; the list L_i = the (<= 128) kept entries with value <= tau_i, stored in the lane's own 4
// slots (no compaction, no overflow).  Every column outside L_i then has c_ij - v_j >= tau_i, and
// because prices only ever FALL in this algorithm that stays true forever:
//        c_ij - v_j >= tau_i   for all j not in L_i.                                        (*)
// (*) turns the list into an exact oracle for the dense row: if the best list value w1 is below
// tau_i, it is the best over ALL columns, and min(w2, tau_i) is a lower bound of the true second
// best, so bidding the increment gamma = min(w2, tau_i) - w1 keeps the new edge an exact arg-min of
// its row (complementary slackness holds exactly; a smaller-than-possible increment is always valid).
// If w1 >= tau_i the list is exhausted and the warp rebuilds it from the dense row at current prices:
// one sweep that collects every column with c - v < tau_i + width_i (width_i = the value range the
// previous list covered) into the 128 slots; columns that do not fit lower the new tau instead.
//
// Schedule.  ONE 1024-thread CTA per matrix: prices (f64) and the column owners (u16) live in shared
// memory, the lists in global memory (L2 resident).  The 32 warps run independently, without any
// barrier.  Rows are served first-in first-out: fresh rows 0..nr-1 from a counter, then displaced
// owners through a ticket ring (FIFO order needs ~40 % fewer bids than following the displaced row
// depth-first).  Per bid: 4 list entries per lane against the current prices, warp arg-min and
// second-min with REDUX on order-preserving integer keys, and the lane that holds the winning column
// commits under a per-column lock (the owner word, CAS to a sentinel): the price must still be the one
// the bid was computed from, otherwise the bid is recomputed.  Other prices may have fallen in the
// meantime, which only makes the true second-best larger, i.e. the committed increment smaller than
// allowed: still exact.  A row whose bid would be a zero-increment steal is parked for phase 2 (this
// is where epsilon = 0 auctions stall); at 8k that is 0-15 rows per matrix.
#define PM_LS_NONE 0xFFFFu
#define PM_LS_LOCKED 0xFFFEu
#define PM_LS_MAX_ROWS 0xFFFDu
#define PM_LS_EMPTY 0xFFFFu

struct PmLsTop {           // the five smallest reduced values a lane has seen, ascending
    double w[5];
    int j[5];
    float c[5];
};

__device__ __forceinline__ void pm_ls_top_init(PmLsTop &t) {
#pragma unroll
    for (int m = 0; m < 5; ++m) { t.w[m] = INFINITY; t.j[m] = -1; t.c[m] = 0.0f; }
}

__device__ __forceinline__ void pm_ls_top_push(PmLsTop &t, double w, int j, float c) {
    if (w < t.w[4]) {      // strict: among equal values the earlier (lower) column stays in front
        t.w[4] = w; t.j[4] = j; t.c[4] = c;
#pragma unroll
        for (int m = 4; m > 0; --m) {
            if (t.w[m] < t.w[m - 1]) {
                const double tw = t.w[m]; t.w[m] = t.w[m - 1]; t.w[m - 1] = tw;
                const int tj = t.j[m]; t.j[m] = t.j[m - 1]; t.j[m - 1] = tj;
                const float tc = t.c[m]; t.c[m] = t.c[m - 1]; t.c[m - 1] = tc;
            }
        }
    }
}

// Candidate lists of all rows at once: one warp per row, all SMs (float4 sweeps, ldc % 4 == 0).
// AT_PRICES = false: the initial lists at zero prices; also accumulates the matrix' cost scale (mean list width).
// AT_PRICES = true: lists at the prices the eps-scaling phases ended with (cells), plus the TIGHT FILTER that turns
// the eps-optimal assignment into an exact warm start: a row keeps its column only if that column is an exact
// arg-min of its row at these prices (complementary slackness with epsilon = 0); every other row is set free and
// its column released.  (An eps-auction leaves the winning edge eps ABOVE the row's second best, so roughly half
// of the rows are released; the exact phase re-seats them with ~1.3 bids each.)
template <bool AT_PRICES>
__global__ void __launch_bounds__(256) pm_ls_build_lists(PmLapBatch B) {
    const PmLapView V = pm_lap_view(B, blockIdx.y);
    const int lane = threadIdx.x & 31;
    const int warp = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), nwarps = gridDim.x * (blockDim.x >> 5);
    const double *prices = reinterpret_cast<const double *>(V.cell);      // first double of every 16-byte cell
    for (int i = warp; i < B.nr; i += nwarps) {
        const float *ci = pm_lap_row(V.cost, B, i);
        PmLsTop t;
        pm_ls_top_init(t);
#pragma unroll 4
        for (int j0 = lane * 4; j0 < B.nc; j0 += 128) {
            const float4 c4 = *reinterpret_cast<const float4 *>(ci + j0);
            const float cc[4] = {c4.x, c4.y, c4.z, c4.w};
#pragma unroll
            for (int e = 0; e < 4; ++e)
                if (j0 + e < B.nc) {
                    const double w = AT_PRICES ? (double)cc[e] - __ldcg(prices + 2 * (size_t)(j0 + e)) : (double)cc[e];
                    pm_ls_top_push(t, w, j0 + e, cc[e]);
                }
        }
        double tmin = t.w[4], wmin = t.w[0];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            tmin = fmin(tmin, __shfl_xor_sync(0xffffffffu, tmin, o));
            wmin = fmin(wmin, __shfl_xor_sync(0xffffffffu, wmin, o));
        }
        reinterpret_cast<int4 *>(V.lcol + (size_t)i * PM_LS_K)[lane] =
            make_int4(t.w[0] <= tmin ? t.j[0] : -1, t.w[1] <= tmin ? t.j[1] : -1, t.w[2] <= tmin ? t.j[2] : -1,
                      t.w[3] <= tmin ? t.j[3] : -1);
        reinterpret_cast<float4 *>(V.lcost + (size_t)i * PM_LS_K)[lane] = make_float4(t.c[0], t.c[1], t.c[2], t.c[3]);
        if (lane == 0) {
            const double width = (tmin < INFINITY && wmin < INFINITY) ? tmin - wmin : INFINITY;
            V.tau[i] = tmin;
            V.width[i] = width;
            if (!AT_PRICES && width < INFINITY && B.scale && i < B.nr_real) {     // (dummy rows have no cost scale)
                atomicAdd(B.scale + 2 * blockIdx.y, width);
                atomicAdd(B.scale + 2 * blockIdx.y + 1, 1.0);
            }
            if (AT_PRICES) {
                const int a = V.col4row[i];
                if (a >= 0) {
                    const double wa = (double)ci[a] - __ldcg(prices + 2 * (size_t)a);
                    if (!(wa <= wmin)) {                  // not an exact arg-min: release (each column has one owner)
                        V.col4row[i] = -1;
                        V.cell[a].owner = 0xFFFFFFFFu;
                    }
                }
            }
        }
    }
}

// start of an eps-scaling phase: every row free again, prices kept (cells), queues empty
__global__ void pm_ls_phase_reset_kernel(PmLapBatch B) {
    const PmLapView V = pm_lap_view(B, blockIdx.y);
    const int t = blockIdx.x * blockDim.x + threadIdx.x, stride = gridDim.x * blockDim.x;
    for (int j = t; j < B.ncp; j += stride) V.cell[j].owner = 0xFFFFFFFFu;
    for (int i = t; i < B.nr; i += stride) V.col4row[i] = -1;
    for (unsigned q = t; q < B.ring_cap; q += stride) V.ring32[q] = 0xFFFFFFFFu;
    if (t == 0) {
        V.counters[PM_LS_CTR_FRESH] = 0; V.counters[PM_LS_CTR_HEAD] = 0; V.counters[PM_LS_CTR_TAIL] = 0;
        V.counters[PM_LS_CTR_LIVE] = B.bulk_warps;
    }
}

// After the last eps-scaling phase of a problem that was made square with dummy rows: make the dummies EXACTLY
// tight before the exact phase.  A dummy (all costs zero) is indifferent between columns of equal price and tight on
// its column only if no column is more expensive.  lambda = the lowest price among the dummy-held columns; every
// column priced above lambda is lowered to lambda (prices only ever fall, so the candidate lists stay certified);
// a real row that held such a column is released (its edge is no longer tight) and re-seated by the exact phase.
// Afterwards all dummy-held columns cost lambda = the maximum price: complementary slackness holds exactly for them.
__global__ void __launch_bounds__(1024) pm_ls_equalise_dummies_kernel(PmLapBatch B) {
    const PmLapView V = pm_lap_view(B, blockIdx.x);
    __shared__ double red[32];
    __shared__ double s_lambda;
    double lam = INFINITY;
    for (int d = B.nr_real + threadIdx.x; d < B.nr; d += blockDim.x) {
        const int j = V.col4row[d];
        if (j >= 0) lam = fmin(lam, V.cell[j].price);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) lam = fmin(lam, __shfl_xor_sync(0xffffffffu, lam, o));
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = lam;
    __syncthreads();
    if (threadIdx.x < 32) {
        lam = red[threadIdx.x];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) lam = fmin(lam, __shfl_xor_sync(0xffffffffu, lam, o));
        if (threadIdx.x == 0) s_lambda = lam;
    }
    __syncthreads();
    lam = s_lambda;
    if (!(lam < INFINITY)) return;              // no dummy is seated (phase cut short): nothing to equalise
    for (int j = threadIdx.x; j < B.nc; j += blockDim.x) {
        if (V.cell[j].price > lam) {
            V.cell[j].price = lam;
            const unsigned r = V.cell[j].owner;
            if (r != 0xFFFFFFFFu && (int)r < B.nr_real) {
                V.cell[j].owner = 0xFFFFFFFFu;
                V.col4row[r] = -1;
            }
        }
    }
}

// eps of this launch for one matrix (0 in the exact phases)
__device__ __forceinline__ double pm_ls_eps(const PmLapBatch &B, int b) {
    if (!(B.eps_factor > 0.0)) return 0.0;
    const double sum = __ldcg(B.scale + 2 * b), cnt = __ldcg(B.scale + 2 * b + 1);
    const double scale = cnt > 0.0 ? sum / cnt : 0.0;
    return (scale > 0.0 && scale < INFINITY) ? B.eps_factor * scale : 0.0;
}

// order-preserving 64-bit integer image of a double (so that REDUX.MIN on two 32-bit halves finds the minimum)
__device__ __forceinline__ unsigned long long pm_ordkey(double x) {
    const long long b = __double_as_longlong(x);
    return (unsigned long long)(b ^ ((b >> 63) | (long long)0x8000000000000000LL));
}
__device__ __forceinline__ double pm_ordval(unsigned long long k) {
    const long long b = (k & 0x8000000000000000ULL) ? (long long)(k ^ 0x8000000000000000ULL) : (long long)~k;
    return __longlong_as_double(b);
}
__device__ __forceinline__ unsigned long long pm_warp_min_u64(unsigned long long k) {
    const unsigned hi = (unsigned)(k >> 32), lo = (unsigned)k;
    const unsigned mh = __reduce_min_sync(0xffffffffu, hi);
    const unsigned ml = __reduce_min_sync(0xffffffffu, hi == mh ? lo : 0xffffffffu);
    return ((unsigned long long)mh << 32) | ml;
}

// Rebuild the list of one row at current prices (one warp): every column with c - v < limit goes into
// the row's 128 slots in column order; what does not fit lowers tau.  Returns the number of entries
// (uniform); the lane's own slots and the new tau / width come back in registers.
// CELLS: prices are the first double of the bulk kernel's 16-byte global cells (read through L2);
// otherwise a plain (shared-memory) array.  A stale price only makes the certificate more conservative.
template <bool CELLS>
__device__ __forceinline__ int pm_ls_refresh_row(const PmLapView &V, int row, const float *__restrict__ ci,
                                                 const double *v, int nc, int lane, double limit, int4 &cj,
                                                 float4 &cc, double &tau, double &wmin_out) {
    int32_t *lcol = V.lcol + (size_t)row * PM_LS_K;
    float *lcost = V.lcost + (size_t)row * PM_LS_K;
    reinterpret_cast<int4 *>(lcol)[lane] = make_int4(-1, -1, -1, -1);
    __syncwarp();
    int count = 0;
    double dropped = INFINITY, wmin = INFINITY;
    for (int base = 0; base < nc; base += 512) {       // 4 sweeps per trip: the four row loads are in flight together
        float4 c4[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int j0 = base + u * 128 + lane * 4;
            c4[u] = make_float4(0.f, 0.f, 0.f, 0.f);
            if (j0 < nc) c4[u] = *reinterpret_cast<const float4 *>(ci + j0);
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int j0 = base + u * 128 + lane * 4;
            const float cs[4] = {c4[u].x, c4[u].y, c4[u].z, c4[u].w};
            double w[4];
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const int j = j0 + e;
                w[e] = INFINITY;
                if (j < nc) w[e] = (double)cs[e] - (CELLS ? __ldcg(v + 2 * (size_t)j) : v[j]);
                wmin = fmin(wmin, w[e]);
            }
            const bool any = (w[0] < limit) || (w[1] < limit) || (w[2] < limit) || (w[3] < limit);
            if (__any_sync(0xffffffffu, any)) {
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    const bool hit = w[e] < limit;
                    const unsigned hits = __ballot_sync(0xffffffffu, hit);
                    if (hits) {
                        const int pos = count + __popc(hits & ((1u << lane) - 1u));
                        if (hit) {
                            if (pos < PM_LS_K) { lcol[pos] = j0 + e; lcost[pos] = cs[e]; }
                            else dropped = fmin(dropped, w[e]);
                        }
                        count += __popc(hits);
                    }
                }
            }
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        dropped = fmin(dropped, __shfl_xor_sync(0xffffffffu, dropped, o));
        wmin = fmin(wmin, __shfl_xor_sync(0xffffffffu, wmin, o));
    }
    tau = fmin(limit, dropped);
    wmin_out = wmin;
    __syncwarp();
    cj = __ldcg(reinterpret_cast<const int4 *>(lcol) + lane);
    cc = __ldcg(reinterpret_cast<const float4 *>(lcost) + lane);
    return count;          // columns below the limit (more than PM_LS_K: the surplus was dropped and lowered tau)
}

// Rebuild a row's list so that it CERTIFIES its own best entry again (one warp).  First the window the previous list
// covered above the old bound; if that catches fewer than 8 columns (prices moved a lot) a 4x wider one centred on the
// row minimum.  The slots fill in COLUMN order, so when more than PM_LS_K columns lie below the limit the row minimum
// itself can be among the dropped ones: then tau <= wmin, the list certifies nothing, and repeating the same two
// windows would never end (a matrix of ones with one zero per row after a price drop; the near-ties of an
// eps-equilibrium).  The window above the minimum therefore shrinks by the overflow ratio until the minimum is inside
// (at most PM_LS_K columns below the limit, or only exact ties at the minimum left: tau == wmin, a zero increment).
template <bool CELLS>
__device__ __forceinline__ void pm_ls_refresh_certified(const PmLapView &V, const PmLapBatch &B, int row, const double *prices,
                                                        int nc, int lane, int4 &cj, float4 &cc, double &tau) {
    double width = __ldcg(V.width + row), wmin;
    if (!(width > 0.0) || !(width < INFINITY)) width = fabs(tau) * 1e-3 + 1e-300;
    const float *ci = pm_lap_row(V.cost, B, row);
    double limit = tau + width;
    int n = pm_ls_refresh_row<CELLS>(V, row, ci, prices, nc, lane, limit, cj, cc, tau, wmin);
    if (n < 8 && wmin < INFINITY) {            // window too narrow (prices moved a lot): centre it on the minimum
        width *= 4.0;
        limit = wmin + width;
        if (!(limit > wmin)) limit = nextafter(wmin, (double)INFINITY);
        n = pm_ls_refresh_row<CELLS>(V, row, ci, prices, nc, lane, limit, cj, cc, tau, wmin);
    } else if (n >= PM_LS_K) {
        width *= 0.5;
    }
    for (int guard = 0; n > PM_LS_K && !(wmin < tau) && wmin < INFINITY && guard < 128; ++guard) {
        double span = limit - wmin, next;
        if (span > 0.0 && span < INFINITY) {
            next = wmin + span * (0.5 * (double)PM_LS_K / (double)n);
            if (!(next > wmin)) next = nextafter(wmin, (double)INFINITY);
            if (!(next < limit)) break;                               // only exact ties at the minimum are left
        } else {
            next = wmin + width;                                      // (prices fell meanwhile: the minimum moved past the limit)
            if (!(next > wmin)) next = nextafter(wmin, (double)INFINITY);
        }
        limit = next;
        n = pm_ls_refresh_row<CELLS>(V, row, ci, prices, nc, lane, limit, cj, cc, tau, wmin);
        if (limit - wmin > 0.0) width = limit - wmin;
    }
    if (lane == 0) { V.tau[row] = tau; V.width[row] = width; }
}


enum { PM_LS_WON = 0, PM_LS_PARK = 1, PM_LS_RETRY = 2 };
#define PM_LS_MAX_SPINS 4096   // recomputations (lost races, list rebuilds) of ONE bid before the row is left to phase 2

// ---- bulk phase: the same certified bids, spread over many SMs --------------------------------------
// While thousands of rows are free the auction is throughput-bound, so the bulk of the bids runs on
// `bulk_warps` warps per matrix all over the GPU.  Prices and owners live in global memory as 16-byte
// cells {price, owner}; a bid is committed with ONE 128-bit compare-and-swap on the cell (expected =
// the price the bid was computed from and the owner just read), so price and owner always change
// together and no lock is needed.  Rows whose list is exhausted, zero-increment steals, and whatever
// is still queued when the parallelism has collapsed are simply left free: the tail kernel below
// (shared-memory prices, one CTA) picks them up.
__device__ __forceinline__ bool pm_ls_cas128(PmLsCell *addr, double exp_price, unsigned exp_owner, double new_price,
                                             unsigned new_owner) {
    unsigned long long elo = (unsigned long long)__double_as_longlong(exp_price), ehi = (unsigned long long)exp_owner;
    unsigned long long dlo = (unsigned long long)__double_as_longlong(new_price), dhi = (unsigned long long)new_owner;
    unsigned long long rlo, rhi;
    asm volatile(
        "{\n\t.reg .b128 e, d, r;\n\tmov.b128 e, {%2, %3};\n\tmov.b128 d, {%4, %5};\n\t"
        "atom.acq_rel.gpu.global.cas.b128 r, [%6], e, d;\n\tmov.b128 {%0, %1}, r;\n\t}"
        : "=l"(rlo), "=l"(rhi)
        : "l"(elo), "l"(ehi), "l"(dlo), "l"(dhi), "l"(addr)
        : "memory");
    return rlo == elo && rhi == ehi;
}

__global__ void __launch_bounds__(256) pm_ls_bulk_kernel(PmLapBatch B, int ctas_per_matrix) {
    const PmLapView V = pm_lap_view(B, blockIdx.x / ctas_per_matrix);
    const int nr = B.nr_real, nc = B.nc, lane = threadIdx.x & 31;
    PmLsCell *cell = V.cell;
    volatile unsigned *ring = V.ring32;
    const unsigned ring_mask = B.ring_cap - 1;
    volatile int *ctr = V.counters;
    const double eps = pm_ls_eps(B, blockIdx.x / ctas_per_matrix);
    int bids = 0, retries = 0, dropped = 0, refreshes = 0;
    int carry = -1;
    while (bids < B.max_bids) {
        int row = carry;
        carry = -1;
        if (row >= 0 && ctr[PM_LS_CTR_LIVE] <= B.bulk_stop_live) break;    // few chains left: tail kernel
        if (row < 0) {
            if (lane == 0) {
                if (ctr[PM_LS_CTR_FRESH] < nr) {
                    const int r = atomicAdd(&V.counters[PM_LS_CTR_FRESH], 1);
                    if (r < nr) row = r;
                }
                if (row < 0 && ctr[PM_LS_CTR_LIVE] > B.bulk_stop_live &&
                    (int)((unsigned)ctr[PM_LS_CTR_TAIL] - (unsigned)ctr[PM_LS_CTR_HEAD]) > 0) {
                    // ticket pop: slots fill in ticket order; a warp whose ticket overshot the queue waits a
                    // little for the next push and then leaves - a row that later lands in an abandoned
                    // slot simply stays free for the tail kernel
                    const unsigned ticket = atomicAdd((unsigned *)&V.counters[PM_LS_CTR_HEAD], 1u);
                    for (int spin = 0; spin < B.bulk_patience; ++spin) {
                        const unsigned x = ring[ticket & ring_mask];
                        if (x != 0xFFFFFFFFu) { ring[ticket & ring_mask] = 0xFFFFFFFFu; row = (int)x; break; }
                        if (ctr[PM_LS_CTR_LIVE] <= B.bulk_stop_live) break;
                        __nanosleep(200);
                    }
                }
            }
            row = __shfl_sync(0xffffffffu, row, 0);
            if (row < 0) break;
        }
        // (DUMMY rows, row >= nr_real, present when a problem with few slack columns was made square, never bid here:
        // a dummy's bid is a sweep over all prices, cheap in the tail kernel's shared memory and ~40 us through L2;
        // a displaced dummy is simply left free and the tail kernel seats it)
        int4 cj = __ldcg(reinterpret_cast<const int4 *>(V.lcol + (size_t)row * PM_LS_K) + lane);
        float4 cc = __ldcg(reinterpret_cast<const float4 *>(V.lcost + (size_t)row * PM_LS_K) + lane);
        double tau = __ldcg(V.tau + row);
        bool fresh = false, won = false;
        int spins = 0;
        while (true) {
            if (++spins > PM_LS_MAX_SPINS) break;           // watchdog: the row stays free for the augmenting paths
            double w1, w2, v1 = 0.0;        // lane-local: best and second-best reduced value, price / owner of the best
            int bj = -1;
            unsigned own = 0xFFFFFFFFu;
            {
                const int js[4] = {cj.x, cj.y, cj.z, cj.w};
                const float cs[4] = {cc.x, cc.y, cc.z, cc.w};
                double vs[4], ws[4];
                unsigned os[4];
#pragma unroll
                for (int e = 0; e < 4; ++e) {       // {price, owner} of the cell in one 16-byte load
                    const ulonglong2 c = __ldcv(reinterpret_cast<const ulonglong2 *>(&cell[js[e] < 0 ? 0 : js[e]]));
                    vs[e] = __longlong_as_double((long long)c.x);
                    os[e] = (unsigned)c.y;
                    const double w = (double)cs[e] - vs[e];
                    ws[e] = js[e] < 0 ? INFINITY : w;
                }
                const double lo01 = fmin(ws[0], ws[1]), hi01 = fmax(ws[0], ws[1]);
                const double lo23 = fmin(ws[2], ws[3]), hi23 = fmax(ws[2], ws[3]);
                w1 = fmin(lo01, lo23);
                w2 = fmin(fmax(lo01, lo23), fmin(hi01, hi23));
                const bool m0 = ws[0] == w1, m1 = ws[1] == w1, m2 = ws[2] == w1;
                bj = m0 ? js[0] : m1 ? js[1] : m2 ? js[2] : js[3];
                v1 = m0 ? vs[0] : m1 ? vs[1] : m2 ? vs[2] : vs[3];
                own = m0 ? os[0] : m1 ? os[1] : m2 ? os[2] : os[3];
            }
            const unsigned long long k1 = pm_ordkey(w1);
            const unsigned long long kb = pm_warp_min_u64(k1);
            const int hl = __ffs(__ballot_sync(0xffffffffu, k1 == kb)) - 1;
            const bool holder = lane == hl;
            const double bw = pm_ordval(kb);
            const double sw = pm_ordval(pm_warp_min_u64(pm_ordkey(holder ? w2 : w1)));
            if (!(bw < INFINITY)) break;                    // no finite entry: phase 2 reports it
            if (!(bw < tau) && !(fresh && bw <= tau)) {     // list exhausted: rebuild from the dense row
                pm_ls_refresh_certified<true>(V, B, row, reinterpret_cast<const double *>(cell), nc, lane, cj, cc, tau);
                __threadfence();                            // the next warp that serves this row may sit on another SM
                fresh = true;
                ++refreshes;
                continue;
            }
            double gamma = fmin(sw, tau) - bw;
            if (!(gamma > 0.0)) gamma = 0.0;
            gamma += eps;                                   // (eps-scaling phases; 0 in the exact phases)
            int result = PM_LS_RETRY;
            unsigned prev = 0xFFFFFFFFu;
            if (holder) {
                if (v1 - gamma == v1 && own != 0xFFFFFFFFu) result = PM_LS_PARK;        // zero-increment steal (or an increment below the price's resolution)
                else if (pm_ls_cas128(&cell[bj], v1, own, v1 - gamma, (unsigned)row)) {
                    result = PM_LS_WON;
                    if (own != 0xFFFFFFFFu && (int)own < nr) {
                        // displaced owner: behind everything that is queued, or carried on by this warp
                        const bool queued = ctr[PM_LS_CTR_FRESH] < nr ||
                                            (int)((unsigned)ctr[PM_LS_CTR_TAIL] - (unsigned)ctr[PM_LS_CTR_HEAD]) > 0;
                        if (queued) {
                            const unsigned pos = atomicAdd((unsigned *)&V.counters[PM_LS_CTR_TAIL], 1u);
                            ring[pos & ring_mask] = own;
                        } else {
                            prev = own;
                        }
                    }
                }
            }
            result = __shfl_sync(0xffffffffu, result, hl);
            prev = __shfl_sync(0xffffffffu, prev, hl);
            if (result == PM_LS_WON) { won = true; if (prev != 0xFFFFFFFFu) carry = (int)prev; break; }
            if (result == PM_LS_PARK) break;
            ++retries;
        }
        ++bids;
        if (!won) ++dropped;
    }
    if (lane == 0) {
        atomicSub(&V.counters[PM_LS_CTR_LIVE], 1);
        atomicAdd(&V.counters[PM_LS_CTR_BIDS], bids);
        atomicAdd(&V.counters[PM_LS_CTR_RETRIES], retries);
        atomicAdd(&V.counters[PM_LS_CTR_DROPPED], dropped);
        atomicAdd(&V.counters[PM_LS_CTR_REFRESHES], refreshes);
    }
}

struct PmLsShared {
    int fresh;              // next fresh row
    unsigned head, tail;    // ring of displaced rows
    int live;               // warps still bidding
    int dummy_token;        // held by the one warp that bids for a dummy row (see the tail kernel)
    unsigned long long stat[6];   // bids, refreshes, retries, parked, refresh cycles, (max) busy cycles
    unsigned long long maxbids;
};

// dynamic shared memory: v f64[ncp] | owner u16[ncp] | ring u16[ring_cap] (ring_cap = 0: ring in global memory)
__global__ void __launch_bounds__(1024, 1) pm_ls_auction_kernel(PmLapBatch B) {
    extern __shared__ __align__(16) unsigned char pm_ls_smem[];
    const PmLapView V = pm_lap_view(B, blockIdx.x);
    const int nr = B.nr, nc = B.nc, ncp = B.ncp;
    double *v = reinterpret_cast<double *>(pm_ls_smem);
    unsigned short *owner = reinterpret_cast<unsigned short *>(v + ncp);
    volatile unsigned short *ring = B.ring_in_smem ? (owner + ncp) : V.ring;
    const unsigned ring_mask = B.ring_cap - 1;
    __shared__ PmLsShared S;
    const int t = threadIdx.x, lane = t & 31;

    // state left by the bulk kernel: prices / owners from the cells, free rows (ascending) into the ring
    __shared__ int s_scan[33];
    for (int j = t; j < ncp; j += blockDim.x) {
        const PmLsCell c = V.cell[j];
        v[j] = (j < nc) ? c.price : 0.0;
        owner[j] = (j < nc && c.owner != 0xFFFFFFFFu) ? (unsigned short)c.owner : (unsigned short)PM_LS_NONE;
    }
    for (unsigned q = t; q < B.ring_cap; q += blockDim.x) ring[q] = PM_LS_EMPTY;
    for (int i = t; i < nr; i += blockDim.x) { V.col4row[i] = -1; V.u[i] = 0.0; }
    if (t == 0) {
        S.fresh = nr; S.head = 0; S.tail = 0; S.maxbids = 0; S.live = blockDim.x >> 5; S.dummy_token = 0;
        for (int k = 0; k < 6; ++k) S.stat[k] = 0;
    }
    __syncthreads();
    for (int j = t; j < nc; j += blockDim.x)
        if (owner[j] != PM_LS_NONE) V.col4row[owner[j]] = j;
    __syncthreads();
    for (int base = 0; base < nr; base += blockDim.x) {
        const int i = base + t;
        const bool is_free = (i < nr) && (V.col4row[i] < 0);
        const unsigned bal = __ballot_sync(0xffffffffu, is_free);
        if (lane == 0) s_scan[t >> 5] = __popc(bal);
        __syncthreads();
        if (t == 0) {
            int acc = (int)S.tail;
            for (int w = 0; w < (int)(blockDim.x >> 5); ++w) { const int c = s_scan[w]; s_scan[w] = acc; acc += c; }
            s_scan[32] = acc;
        }
        __syncthreads();
        if (is_free) ring[(s_scan[t >> 5] + __popc(bal & ((1u << lane) - 1u))) & ring_mask] = (unsigned short)i;
        __syncthreads();
        if (t == 0) S.tail = (unsigned)s_scan[32];
        __syncthreads();
    }
    const double eps = pm_ls_eps(B, blockIdx.x);
    long long bids = 0, refreshes = 0, retries = 0, parked = 0, refresh_cycles = 0;
    int requeues = 0;
    const long long t_begin = clock64();
    int carry = -1;          // displaced owner this warp continues with (only when nothing is queued)
    while (bids < B.max_bids_tail) {
        // ---- next row: fresh rows first, then displaced owners in FIFO order
        int row = carry;
        carry = -1;
        // few chains left: the tail of an epsilon = 0 auction is a sequential price war that one
        // shortest-augmenting-path search settles at once -> leave the carried row to phase 2
        if (row >= 0 && *(volatile int *)&S.live <= B.stop_live) break;
        if (row < 0) {
            if (lane == 0) {
                if (*(volatile int *)&S.fresh < nr) {
                    const int r = atomicAdd(&S.fresh, 1);
                    if (r < nr) row = r;
                }
                while (row < 0) {
                    const unsigned h = *(volatile unsigned *)&S.head, tl = *(volatile unsigned *)&S.tail;
                    if ((int)(tl - h) <= 0) break;                       // nothing queued: this warp is done
                    if (atomicCAS(&S.head, h, h + 1u) != h) continue;
                    unsigned short x;
                    do { x = ring[h & ring_mask]; } while (x == PM_LS_EMPTY);   // slot reserved, value in flight
                    ring[h & ring_mask] = PM_LS_EMPTY;
                    row = x;
                }
            }
            row = __shfl_sync(0xffffffffu, row, 0);
            if (row < 0) break;
        }
        // A DUMMY row (row >= nr_real: all costs zero, present when a problem with few slack columns was made square) has
        // no use for a candidate list: its reduced values are just the negated prices, so it bids from one sweep over the
        // prices (exact best / second best, no certificate needed).  All dummies want the same column, the most expensive
        // one: bidding for them concurrently means that every commit invalidates the sweeps of all the others.  ONE warp
        // at a time bids for a dummy; the others put theirs back in the queue.  (The large cost of the dummies, 2.3 ms each
        // per solve, was the chain of individual bids, see the class rule below; the token alone did not change it.)
        const bool dummy = row >= B.nr_real;
        if (dummy) {
            int got = 0;
            if (lane == 0) {
                got = atomicCAS(&S.dummy_token, 0, 1) == 0;
                if (!got) {
                    const unsigned pos = atomicAdd(&S.tail, 1u);
                    ring[pos & ring_mask] = (unsigned short)row;
                }
            }
            got = __shfl_sync(0xffffffffu, got, 0);
            if (!got) {
                if (++requeues > (1 << 22)) break;       // (watchdog; the token holder always finishes its bid)
                __nanosleep(400);
                continue;
            }
        }
        int4 cj = make_int4(-1, -1, -1, -1);
        float4 cc = make_float4(0.f, 0.f, 0.f, 0.f);
        double tau = INFINITY;
        if (!dummy) {
            cj = __ldcg(reinterpret_cast<const int4 *>(V.lcol + (size_t)row * PM_LS_K) + lane);
            cc = __ldcg(reinterpret_cast<const float4 *>(V.lcost + (size_t)row * PM_LS_K) + lane);
            tau = __ldcg(V.tau + row);
        }
        bool fresh = false;
        int result, prev = PM_LS_NONE, spins = 0;
        while (true) {
            if (++spins > PM_LS_MAX_SPINS) { result = PM_LS_PARK; break; }        // watchdog: left to the augmenting paths
            double w1, w2, v1 = 0.0;        // lane-local: best and second-best reduced value, price of the best
            int bj = -1;
            if (dummy) {
                // eps-scaling phases: the dummies bid as ONE class of similar persons (Bertsekas & Castanon): a dummy
                // looks only at columns that no other dummy holds.  Bidding individually, a displaced dummy takes the
                // most expensive column from the next dummy, which takes the next one ... a chain through all
                // nc - nr dummies for every column a real row takes from them (measured: 2.3 ms per dummy and solve
                // at 8k).  The class keeps eps-complementary-slackness as a whole (every column outside it costs at
                // most the cheapest dummy-held column + eps).  The exact phase (eps = 0) bids individually: there the
                // dummies sit on equal prices (pm_ls_equalise_dummies_kernel) and a displaced one parks at once.
                w1 = INFINITY; w2 = INFINITY;
                // two columns per lane and trip (one 16-byte and one 4-byte shared load), four trips in flight
                const unsigned v_s = (unsigned)__cvta_generic_to_shared(v), o_s = (unsigned)__cvta_generic_to_shared(owner);
#pragma unroll 4
                for (int j = 2 * lane; j < nc; j += 64) {
                    double va, vb;
                    unsigned oo;
                    asm volatile("ld.volatile.shared.v2.f64 {%0, %1}, [%2];" : "=d"(va), "=d"(vb) : "r"(v_s + 8u * (unsigned)j));
                    asm volatile("ld.volatile.shared.u32 %0, [%1];" : "=r"(oo) : "r"(o_s + 2u * (unsigned)j));
                    const unsigned oa = oo & 0xffffu, ob = oo >> 16;
                    const bool skip_a = eps > 0.0 && oa < PM_LS_LOCKED && (int)oa >= B.nr_real;
                    const bool skip_b = (j + 1 >= nc) || (eps > 0.0 && ob < PM_LS_LOCKED && (int)ob >= B.nr_real);
                    if (!skip_a) {
                        const double w = -va;
                        if (w < w1) { w2 = w1; w1 = w; bj = j; v1 = va; }
                        else if (w < w2) w2 = w;
                    }
                    if (!skip_b) {
                        const double w = -vb;
                        if (w < w1) { w2 = w1; w1 = w; bj = j + 1; v1 = vb; }
                        else if (w < w2) w2 = w;
                    }
                }
            } else {
                // its 4 list slots at the current prices, branch-free
                const int js[4] = {cj.x, cj.y, cj.z, cj.w};
                const float cs[4] = {cc.x, cc.y, cc.z, cc.w};
                double vs[4], ws[4];
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    vs[e] = *reinterpret_cast<volatile double *>(&v[js[e] < 0 ? 0 : js[e]]);
                    const double w = (double)cs[e] - vs[e];
                    ws[e] = js[e] < 0 ? INFINITY : w;
                }
                // smallest and second smallest of four: 7 min/max
                const double lo01 = fmin(ws[0], ws[1]), hi01 = fmax(ws[0], ws[1]);
                const double lo23 = fmin(ws[2], ws[3]), hi23 = fmax(ws[2], ws[3]);
                w1 = fmin(lo01, lo23);
                w2 = fmin(fmax(lo01, lo23), fmin(hi01, hi23));
                const bool m0 = ws[0] == w1, m1 = ws[1] == w1, m2 = ws[2] == w1;
                bj = m0 ? js[0] : m1 ? js[1] : m2 ? js[2] : js[3];
                v1 = m0 ? vs[0] : m1 ? vs[1] : m2 ? vs[2] : vs[3];
            }
            // warp: best value (REDUX on order-preserving keys), one holder lane, second best
            const unsigned long long k1 = pm_ordkey(w1);
            const unsigned long long kb = pm_warp_min_u64(k1);
            const unsigned holders = __ballot_sync(0xffffffffu, k1 == kb);
            const int hl = __ffs(holders) - 1;
            const bool holder = lane == hl;
            const double bw = pm_ordval(kb);
            // smallest value that does not belong to the winning slot
            const double sw = pm_ordval(pm_warp_min_u64(pm_ordkey(holder ? w2 : w1)));
            if (!(bw < INFINITY)) { result = PM_LS_PARK; break; }                 // no finite entry: phase 2 reports it
            if (!(bw < tau) && !(fresh && bw <= tau)) {
                // list exhausted: cannot certify the best column -> rebuild from the dense row
                const long long t0 = clock64();
                pm_ls_refresh_certified<false>(V, B, row, v, nc, lane, cj, cc, tau);
                fresh = true;
                ++refreshes;
                refresh_cycles += clock64() - t0;
                continue;
            }
            double gamma = fmin(sw, tau) - bw;    // certified lower bound of the true increment
            if (!(gamma > 0.0) || !(gamma < INFINITY)) gamma = 0.0;       // (infinite: a dummy with one column to choose from)
            gamma += eps;                         // (eps-scaling phases; 0 in the exact phases)
            result = PM_LS_RETRY;
            if (holder) {
                unsigned short *p = &owner[bj];
                unsigned short old;
                while (true) {      // lock the column: the owner word doubles as the lock
                    old = *reinterpret_cast<volatile unsigned short *>(p);
                    if (old != PM_LS_LOCKED && atomicCAS(p, old, (unsigned short)PM_LS_LOCKED) == old) break;
                }
                const double vj = *reinterpret_cast<volatile double *>(&v[bj]);
                if (vj != v1 || (dummy && eps > 0.0 && old < PM_LS_LOCKED && (int)old >= B.nr_real)) {
                    *reinterpret_cast<volatile unsigned short *>(p) = old;                 // price moved (or another dummy took it): recompute
                } else if (vj - gamma == vj && old != PM_LS_NONE) {
                    *reinterpret_cast<volatile unsigned short *>(p) = old;                 // zero-increment steal: park
                    result = PM_LS_PARK;
                } else {
                    *reinterpret_cast<volatile double *>(&v[bj]) = vj - gamma;
                    __threadfence_block();
                    *reinterpret_cast<volatile unsigned short *>(p) = (unsigned short)row;  // releases the lock
                    result = PM_LS_WON;
                    prev = old;
                    if (old != PM_LS_NONE) {
                        // displaced owner bids again: behind everything that is queued (FIFO needs fewer
                        // bids than depth-first), or right away in this warp when nothing is queued
                        const bool queued = *(volatile int *)&S.fresh < nr ||
                                            (int)(*(volatile unsigned *)&S.tail - *(volatile unsigned *)&S.head) > 0;
                        if (queued) {
                            const unsigned pos = atomicAdd(&S.tail, 1u);
                            ring[pos & ring_mask] = old;
                            prev = PM_LS_NONE;
                        }
                    }
                }
            }
            result = __shfl_sync(0xffffffffu, result, hl);
            prev = __shfl_sync(0xffffffffu, prev, hl);
            if (result != PM_LS_RETRY) break;
            ++retries;
        }
        if (dummy) {
            __threadfence_block();
            if (lane == 0) atomicExch(&S.dummy_token, 0);
        }
        ++bids;
        if (result == PM_LS_PARK) ++parked;
        else if (prev != PM_LS_NONE) carry = prev;
    }
    if (lane == 0) {
        atomicSub(&S.live, 1);
        atomicAdd(&S.stat[0], (unsigned long long)bids);
        atomicAdd(&S.stat[1], (unsigned long long)refreshes);
        atomicAdd(&S.stat[2], (unsigned long long)retries);
        atomicAdd(&S.stat[3], (unsigned long long)parked);
        atomicAdd(&S.stat[4], (unsigned long long)refresh_cycles);
        atomicMax(&S.stat[5], (unsigned long long)(clock64() - t_begin));
        atomicMax(&S.maxbids, (unsigned long long)bids);
    }
    __syncthreads();
    for (int i = t; i < nr; i += blockDim.x) V.col4row[i] = -1;     // (held the bulk kernel's matching until here)
    __syncthreads();
    // hand the state to phase 2: prices, owners, row duals u_i = c_ij - v_j of the assigned edge
    for (int j = t; j < ncp; j += blockDim.x) {
        const unsigned short r = owner[j];
        if (j < nc) {
            V.v[j] = v[j];
            V.cell[j].price = v[j];               // (the next eps-scaling phase / the tight filter read the cells)
            V.cell[j].owner = (r == PM_LS_NONE) ? 0xFFFFFFFFu : (unsigned)r;
            V.row4col[j] = (r == PM_LS_NONE) ? -1 : (int)r;
            if (r != PM_LS_NONE) {
                V.col4row[r] = j;
                V.u[r] = (double)pm_lap_row(V.cost, B, r)[j] - v[j];
            }
        }
    }
    if (t == 0) {
        V.counters[3] = (int32_t)(S.maxbids > 0x7fffffffull ? 0x7fffffffull : S.maxbids);
        if (V.stats) {      // accumulated over the launches of this solve (eps-scaling phases + exact phase)
            V.stats[PM_LAP_STAT_BIDS] += (long long)S.stat[0];
            V.stats[PM_LAP_STAT_BULK_BIDS] = V.counters[PM_LS_CTR_BIDS];
            V.stats[PM_LAP_STAT_REFRESHES] += (long long)S.stat[1];
            V.stats[PM_LAP_STAT_RETRIES] += (long long)S.stat[2];
            V.stats[PM_LAP_STAT_PARKED] = (long long)S.stat[3];
            V.stats[PM_LAP_STAT_REFRESH_CYCLES] += (long long)S.stat[4];
            V.stats[PM_LAP_STAT_AUCTION_CYCLES] += (long long)S.stat[5];
            if (!(B.eps_factor > 0.0)) {     // last auction launch of the solve: fold the bulk kernels' counters in
                V.stats[PM_LAP_STAT_BIDS] += V.counters[PM_LS_CTR_BIDS];
                V.stats[PM_LAP_STAT_REFRESHES] += V.counters[PM_LS_CTR_REFRESHES];
                V.stats[PM_LAP_STAT_RETRIES] += V.counters[PM_LS_CTR_RETRIES];
            }
        }
    }
}

// ------------------------------------------------------------------------------------- phase 2
// Block arg-min over (value, tie) with lexicographic order; every thread receives the result.
__device__ __forceinline__ void pm_argmin_warp(double &val, int &tie) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const double ov = __shfl_xor_sync(0xffffffffu, val, o);
        const int ot = __shfl_xor_sync(0xffffffffu, tie, o);
        if (ov < val || (ov == val && ot < tie)) { val = ov; tie = ot; }
    }
}

// V_IN_REGS: prices of the owned columns live in registers (nc <= 8 * 1024); otherwise they are read
// from global memory (L2-resident) every step and d stays in registers (CPT up to 24).
template <int CPT, bool V_IN_REGS>
__global__ void __launch_bounds__(PM_LAP_MAX_THREADS, 1) pm_lap_sap_kernel(PmLapBatch B, int final_parity) {
    const PmLapView V = pm_lap_view(B, blockIdx.x);
    extern __shared__ __align__(16) unsigned char pm_lap_smem[];
    const int nc = B.nc, nr = B.nr, ldc = B.ldc;
    const int nthreads = blockDim.x, t = threadIdx.x, lane = t & 31, warp = t >> 5;
    const int group_stride = nthreads * 4;           // columns covered by one float4 sweep of the CTA
    int32_t *pred = reinterpret_cast<int32_t *>(pm_lap_smem);
    int32_t *r4c = pred + (size_t)(CPT / 4) * group_stride;
    __shared__ double s_val[2][32];
    __shared__ int s_tie[2][32];
    __shared__ int s_scan[33];
    __shared__ int s_nfree;

    // column owned by slot q of this thread
    auto col_of = [&](int q) { return (q >> 2) * group_stride + t * 4 + (q & 3); };

    double vreg[V_IN_REGS ? CPT : 1];
    double d[CPT];
    unsigned assigned = 0u;
#pragma unroll
    for (int q = 0; q < CPT; ++q) {
        const int c = col_of(q);
        const int r = (c < nc) ? V.row4col[c] : -1;
        r4c[c] = r;
        if (r >= 0) assigned |= 1u << q;
        if (V_IN_REGS) vreg[q] = (c < nc) ? V.v[c] : 0.0;
    }
    // ordered list of free rows (ascending row index -> deterministic), into list 0
    int32_t *flist = V.free_lists;
    if (t == 0) s_nfree = 0;
    __syncthreads();
    for (int base = 0; base < nr; base += nthreads) {
        const int i = base + t;
        const bool is_free = (i < nr) && (V.col4row[i] < 0);
        const unsigned bal = __ballot_sync(0xffffffffu, is_free);
        if (lane == 0) s_scan[warp] = __popc(bal);
        __syncthreads();
        if (t == 0) {
            int acc = s_nfree;
            for (int w = 0; w < (nthreads >> 5); ++w) { const int c = s_scan[w]; s_scan[w] = acc; acc += c; }
            s_scan[32] = acc;
        }
        __syncthreads();
        if (is_free) flist[s_scan[warp] + __popc(bal & ((1u << lane) - 1u))] = i;
        __syncthreads();
        if (t == 0) s_nfree = s_scan[32];
        __syncthreads();
    }
    const int nfree = s_nfree;
    long long steps = 0;
    int status = 0;
    int parity = 0;

    for (int f = 0; f < nfree && status == 0; ++f) {
        const int cur = flist[f];
        double min_val = 0.0;
        int i = cur, sink = -1;
        unsigned scanned = 0u;
#pragma unroll
        for (int q = 0; q < CPT; ++q) d[q] = INFINITY;
        while (true) {
            const float *ci = pm_lap_row(V.cost, B, i);
            const double ui = V.u[i];
            double best = INFINITY;
            int best_tie = INT_MAX;
#pragma unroll
            for (int g = 0; g < CPT / 4; ++g) {
                const int c0 = g * group_stride + t * 4;
                float4 c4 = make_float4(0.f, 0.f, 0.f, 0.f);
                if (c0 < B.ncp) c4 = *reinterpret_cast<const float4 *>(ci + c0);      // (ncp <= ldc; the dummy rows' zero row has ncp + 32 floats)
                double2 va = make_double2(0.0, 0.0), vb = make_double2(0.0, 0.0);
                if (!V_IN_REGS && c0 < nc) {   // v padded to a multiple of 4 doubles in the workspace
                    va = *reinterpret_cast<const double2 *>(V.v + c0);
                    vb = *reinterpret_cast<const double2 *>(V.v + c0 + 2);
                }
                const float cc[4] = {c4.x, c4.y, c4.z, c4.w};
                const double vv[4] = {va.x, va.y, vb.x, vb.y};
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    const int q = g * 4 + e, c = c0 + e;
                    if (c < nc && !((scanned >> q) & 1u)) {
                        const double vj = V_IN_REGS ? vreg[q] : vv[e];
                        const double r = ((min_val + (double)cc[e]) - ui) - vj;
                        if (r < d[q]) { d[q] = r; pred[c] = i; }
                        const int tie = (((assigned >> q) & 1u) ? (1 << 30) : 0) | c;   // prefer a free column
                        if (d[q] < best || (d[q] == best && tie < best_tie)) { best = d[q]; best_tie = tie; }
                    }
                }
            }
            pm_argmin_warp(best, best_tie);
            if (lane == 0) { s_val[parity][warp] = best; s_tie[parity][warp] = best_tie; }
            __syncthreads();
            best = (lane < (nthreads >> 5)) ? s_val[parity][lane] : INFINITY;
            best_tie = (lane < (nthreads >> 5)) ? s_tie[parity][lane] : INT_MAX;
            pm_argmin_warp(best, best_tie);
            parity ^= 1;
            ++steps;
            if (!(best < INFINITY)) { status = PM_ERR_INFEASIBLE; break; }
            min_val = best;
            const int jmin = best_tie & ((1 << 30) - 1);
            {   // owner marks the column as scanned
                const int g = jmin / group_stride, rem = jmin - g * group_stride;
                if ((rem >> 2) == t) scanned |= 1u << (g * 4 + (rem & 3));
            }
            if (!(best_tie >> 30)) { sink = jmin; break; }
            i = r4c[jmin];
        }
        if (status) break;
        // dual update (Crouse: u[cur] += min; scanned rows/cols shift by min - d)
#pragma unroll
        for (int q = 0; q < CPT; ++q) {
            if ((scanned >> q) & 1u) {
                const int c = col_of(q);
                const double delta = min_val - d[q];
                if (V_IN_REGS) vreg[q] -= delta; else V.v[c] -= delta;
                if (c != sink) V.u[r4c[c]] += delta;
            }
        }
        if (t == 0) V.u[cur] += min_val;
        __syncthreads();
        if (t == 0) {   // augment along the predecessor chain
            int j = sink;
            while (true) {
                const int r = pred[j];
                r4c[j] = r;
                const int jn = V.col4row[r];
                V.col4row[r] = j;
                j = jn;
                if (r == cur) break;
            }
        }
        __syncthreads();
        assigned = 0u;
#pragma unroll
        for (int q = 0; q < CPT; ++q)
            if (r4c[col_of(q)] >= 0) assigned |= 1u << q;
    }
#pragma unroll
    for (int q = 0; q < CPT; ++q) {
        const int c = col_of(q);
        if (c < nc) {
            if (V_IN_REGS) V.v[c] = vreg[q];
            V.row4col[c] = r4c[c];
        }
    }
    // total cost, float64, fixed order
    __syncthreads();
    double tot = 0.0;
    for (int r = t; r < B.nr_real; r += nthreads) {       // dummy rows cost nothing and are not reported
        const int c = V.col4row[r];
        V.col4row_out[r] = c;
        if (c >= 0) tot += (double)V.cost[(size_t)r * ldc + c];
    }
    tot = pm_block_sum(tot, &s_val[0][0]);
    if (t == 0) {
        V.total[0] = status ? nan("") : tot;
        V.counters[4] = status;
        if (V.stats) {
            V.stats[PM_LAP_STAT_BID_ROUNDS] = V.counters[3];
            V.stats[PM_LAP_STAT_ROWS_AFTER_BIDDING] = nr - nfree;
            V.stats[PM_LAP_STAT_AUGMENTATIONS] = nfree;
            V.stats[PM_LAP_STAT_DIJKSTRA_STEPS] = steps;
            V.stats[PM_LAP_STAT_STATUS] = status;
            V.stats[PM_LAP_STAT_PATH] = B.path;
        }
    }
    (void)final_parity;
}

// ------------------------------------------------------------------------------------- phase 2 (sparse)
// Shortest augmenting paths over the certified candidate lists of the auction.  A Dijkstra step adds
// one row to the alternating tree; instead of the row's 8000 dense costs (one HBM round trip) it
// relaxes the <= 128 list edges (L2).  The certificate (*) of the lists bounds what that leaves out:
// every edge of tree row i outside its list has reduced cost >= tau_i - u_i, so no path through such
// an edge is shorter than bound_i = D_i + tau_i - u_i.  A column is finalised only while its distance
// is <= the smallest bound over the tree; otherwise the row holding that bound is relaxed densely
// (exactly the dense algorithm's step) and its bound removed.  Same result as the dense search.
//
// dynamic shared memory: v f64[ncp] | d f64[ncp] | pred u16[ncp] | r4c u16[ncp] | front u16[ncp] | scanned u8[ncp]
#define PM_SS_THREADS 1024     // the reached frontier grows to most of the columns within ~60 steps: the scan wants every thread

// warp arg-min over (value, tie) in lexicographic order with three REDUX instead of 15 shuffles
__device__ __forceinline__ void pm_ss_argmin_warp(double &val, int &tie) {
    const unsigned long long k = pm_ordkey(val);
    const unsigned long long kb = pm_warp_min_u64(k);
    tie = (int)__reduce_min_sync(0xffffffffu, k == kb ? (unsigned)tie : 0xffffffffu);
    val = pm_ordval(kb);
}

__global__ void __launch_bounds__(PM_SS_THREADS, 1) pm_lap_sap_sparse_kernel(PmLapBatch B) {
    extern __shared__ __align__(16) unsigned char pm_ss_smem[];
    const PmLapView V = pm_lap_view(B, blockIdx.x);
    const int nc = B.nc, nr = B.nr, ncp = B.ncp, ldc = B.ldc;
    const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
    double *v = reinterpret_cast<double *>(pm_ss_smem);
    double *d = v + ncp;
    unsigned short *pred = reinterpret_cast<unsigned short *>(d + ncp);
    unsigned short *r4c = pred + ncp;
    unsigned short *front = r4c + ncp;             // columns reached so far in this search (finite distance)
    unsigned char *scanned = reinterpret_cast<unsigned char *>(front + ncp);
    __shared__ int s_nfront;
    __shared__ double s_val[2][32];
    __shared__ int s_tie[2][32];
    __shared__ int s_scan[33];
    __shared__ int s_nfree;
    __shared__ double s_lam;
    __shared__ int s_lam_idx;
    int32_t *tree_row = V.bid_col;                 // [nr] scratch of the dense auction, free here
    double *tree_dist = V.bid_gamma;               // [nr]
    double *tree_bound = reinterpret_cast<double *>(V.colbest);   // [nc] >= [nr]

    for (int j = t; j < ncp; j += PM_SS_THREADS) {
        const int r = (j < nc) ? V.row4col[j] : -1;
        v[j] = (j < nc) ? V.v[j] : 0.0;
        r4c[j] = (r < 0) ? (unsigned short)PM_LS_NONE : (unsigned short)r;
    }
    // ordered list of free rows (ascending row index) into free_lists
    int32_t *flist = V.free_lists;
    if (t == 0) s_nfree = 0;
    __syncthreads();
    for (int base = 0; base < nr; base += PM_SS_THREADS) {
        const int i = base + t;
        const bool is_free = (i < nr) && (V.col4row[i] < 0);
        const unsigned bal = __ballot_sync(0xffffffffu, is_free);
        if (lane == 0) s_scan[warp] = __popc(bal);
        __syncthreads();
        if (t == 0) {
            int acc = s_nfree;
            for (int w = 0; w < PM_SS_THREADS / 32; ++w) { const int c = s_scan[w]; s_scan[w] = acc; acc += c; }
            s_scan[32] = acc;
        }
        __syncthreads();
        if (is_free) flist[s_scan[warp] + __popc(bal & ((1u << lane) - 1u))] = i;
        __syncthreads();
        if (t == 0) s_nfree = s_scan[32];
        __syncthreads();
    }
    const int nfree = s_nfree;
    long long steps = 0, dense_relax = 0;
    int status = 0, parity = 0;

    for (int f = 0; f < nfree && status == 0; ++f) {
        const int cur = flist[f];
        for (int j = t; j < ncp; j += PM_SS_THREADS) { d[j] = INFINITY; scanned[j] = 0; }
        if (t == 0) { s_lam = INFINITY; s_lam_idx = -1; s_nfront = 0; }
        __syncthreads();
        int i = cur, sink = -1, nt = 0, jlast = -1;      // jlast: column finalised in the previous step
        double dist = 0.0, min_val = 0.0;
        while (sink < 0 && status == 0) {
            // ---- add row i (distance dist) to the tree: relax its list edges, record its bound
            const double ui = __ldcg(V.u + i);
            if (t < PM_LS_K) {
                const int j = __ldcg(V.lcol + (size_t)i * PM_LS_K + t);          // both list loads in flight together
                const float cij = __ldcg(V.lcost + (size_t)i * PM_LS_K + t);
                if (j >= 0 && j != jlast && !scanned[j]) {     // (its scanned flag may not be visible yet)
                    const double r = ((dist + (double)cij) - ui) - v[j];
                    const double old = d[j];
                    if (r < old) {
                        if (!(old < INFINITY)) front[atomicAdd(&s_nfront, 1)] = (unsigned short)j;   // first time reached
                        d[j] = r; pred[j] = (unsigned short)i;
                    }
                }
            } else if (t == PM_LS_K) {
                const double bound = (dist + __ldcg(V.tau + i)) - ui;
                tree_row[nt] = i; tree_dist[nt] = dist; tree_bound[nt] = bound;
                if (bound < s_lam) { s_lam = bound; s_lam_idx = nt; }
            }
            ++nt;
            __syncthreads();
            while (true) {
                // ---- closest unscanned column (ties: the lower index)
                double best = INFINITY;
                int best_tie = INT_MAX;
                const int nfront = s_nfront;
                for (int q = t; q < nfront; q += PM_SS_THREADS) {
                    const int j = front[q];
                    if (!scanned[j]) {
                        const double dj = d[j];
                        if (dj < best || (dj == best && j < best_tie)) { best = dj; best_tie = j; }
                    }
                }
                pm_ss_argmin_warp(best, best_tie);
                if (lane == 0) { s_val[parity][warp] = best; s_tie[parity][warp] = best_tie; }
                __syncthreads();
                best = (lane < PM_SS_THREADS / 32) ? s_val[parity][lane] : INFINITY;
                best_tie = (lane < PM_SS_THREADS / 32) ? s_tie[parity][lane] : INT_MAX;
                pm_ss_argmin_warp(best, best_tie);
                parity ^= 1;
                const double lam = s_lam;
                const int lam_idx = s_lam_idx;
                if (best <= lam) {
                    if (!(best < INFINITY)) { status = PM_ERR_INFEASIBLE; break; }
                    ++steps;
                    min_val = best;
                    const int jm = best_tie;
                    if (t == 0) scanned[jm] = 1;                // visible to everybody after the next barrier
                    jlast = jm;
                    if (r4c[jm] == PM_LS_NONE) sink = jm;
                    else { i = r4c[jm]; dist = best; }
                    break;
                }
                // ---- an edge outside the list of tree row `il` could be shorter: relax that row densely
                __syncthreads();                               // everybody has read s_lam
                const int il = tree_row[lam_idx];
                const double dl = tree_dist[lam_idx], uil = __ldcg(V.u + il);
                const float *ci = pm_lap_row(V.cost, B, il);
                for (int j = t; j < nc; j += PM_SS_THREADS) {
                    if (!scanned[j]) {
                        const double r = ((dl + (double)ci[j]) - uil) - v[j];
                        const double old = d[j];
                        if (r < old) {
                            if (!(old < INFINITY)) front[atomicAdd(&s_nfront, 1)] = (unsigned short)j;
                            d[j] = r; pred[j] = (unsigned short)il;
                        }
                    }
                }
                ++dense_relax;
                if (t == 0) tree_bound[lam_idx] = INFINITY;
                __syncthreads();
                if (warp == 0) {                               // smallest remaining bound over the tree
                    double lb = INFINITY;
                    int li = INT_MAX;
                    for (int k = lane; k < nt; k += 32) {
                        const double bnd = tree_bound[k];
                        if (bnd < lb || (bnd == lb && k < li)) { lb = bnd; li = k; }
                    }
                    pm_argmin_warp(lb, li);
                    if (lane == 0) { s_lam = lb; s_lam_idx = (lb < INFINITY) ? li : -1; }
                }
                __syncthreads();
            }
        }
        if (status) break;
        __syncthreads();
        // dual update (Crouse: u[cur] += min; scanned rows / columns shift by min - d); prices only fall
        for (int j = t; j < nc; j += PM_SS_THREADS) {
            if (scanned[j]) {
                const double delta = min_val - d[j];
                v[j] -= delta;
                if (j != sink) V.u[r4c[j]] += delta;
            }
        }
        if (t == 0) V.u[cur] += min_val;
        __syncthreads();
        if (t == 0) {   // augment along the predecessor chain
            int j = sink;
            while (true) {
                const int r = pred[j];
                r4c[j] = (unsigned short)r;
                const int jn = V.col4row[r];
                V.col4row[r] = j;
                j = jn;
                if (r == cur) break;
            }
        }
        __syncthreads();
    }
    for (int j = t; j < nc; j += PM_SS_THREADS) {
        V.v[j] = v[j];
        V.row4col[j] = (r4c[j] == PM_LS_NONE) ? -1 : (int)r4c[j];
    }
    __syncthreads();
    double tot = 0.0;
    for (int r = t; r < B.nr_real; r += PM_SS_THREADS) {   // dummy rows cost nothing and are not reported
        const int c = V.col4row[r];
        V.col4row_out[r] = c;
        if (c >= 0) tot += (double)V.cost[(size_t)r * ldc + c];
    }
    tot = pm_block_sum(tot, &s_val[0][0]);
    if (t == 0) {
        V.total[0] = status ? nan("") : tot;
        V.counters[4] = status;
        if (V.stats) {
            V.stats[PM_LAP_STAT_BID_ROUNDS] = V.counters[3];
            V.stats[PM_LAP_STAT_ROWS_AFTER_BIDDING] = nr - nfree;
            V.stats[PM_LAP_STAT_AUGMENTATIONS] = nfree;
            V.stats[PM_LAP_STAT_DIJKSTRA_STEPS] = steps;
            V.stats[PM_LAP_STAT_STATUS] = status;
            V.stats[PM_LAP_STAT_SAP_DENSE_RELAX] = dense_relax;
            V.stats[PM_LAP_STAT_PATH] = B.path;
        }
    }
}

// ------------------------------------------------------------------------------------- host
// A kernel's MaxDynamicSharedMemorySize attribute is process-global state: setting it to the per-call size
// right before each launch races when several host threads solve problems of different sizes (another thread
// can lower it between this thread's SetAttribute and its launch -> "invalid argument").  Raise it ONCE per
// device to the opt-in maximum instead and never lower it.
#include <mutex>
static int pm_lap_raise_smem_limit_impl(const void *kernel, int smem_optin, int dev) {
    static std::mutex mu;
    static const void *seen_kernel[64];
    static int seen_dev[64], n_seen = 0;
    std::lock_guard<std::mutex> g(mu);
    for (int q = 0; q < n_seen; ++q)
        if (seen_kernel[q] == kernel && seen_dev[q] == dev) return PM_OK;
    cudaFuncAttributes fa;                          // the opt-in limit covers static + dynamic shared memory
    PM_CUDA_TRY(cudaFuncGetAttributes(&fa, kernel));
    PM_CUDA_TRY(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                     smem_optin - (int)fa.sharedSizeBytes));
    if (n_seen < 64) { seen_kernel[n_seen] = kernel; seen_dev[n_seen] = dev; ++n_seen; }
    return PM_OK;
}
template <typename K>
static int pm_lap_raise_smem_limit(K kernel, int smem_optin, int dev) {
    return pm_lap_raise_smem_limit_impl((const void *)kernel, smem_optin, dev);
}

// header: progress counters | per-matrix cost scale [batch][2] f64 | one row of zeros (the dummy rows' cost row)
static size_t pm_lap_header_bytes(int batch, int ncp) {
    return 256 + pm_lap_align((size_t)batch * 2 * sizeof(double)) + pm_lap_align((size_t)(ncp + 32) * sizeof(float));
}

extern "C" size_t pm_lap_workspace_bytes(int batch, int nr, int nc) {
    if (batch < 1 || nr < 1 || nc < 1) return 0;
    const int ncp = (nc + 3) & ~3;
    return pm_lap_header_bytes(batch, ncp) + (size_t)batch * pm_lap_layout(nc, ncp).per_item;
}

template <int CPT, bool VR>
static int pm_lap_launch_sap(const PmLapBatch &B, int batch, int threads, int smem_optin, int dev, cudaStream_t s) {
    const size_t smem = (size_t)(CPT / 4) * threads * 4 * 2 * sizeof(int32_t);
    if (int rc = pm_lap_raise_smem_limit(pm_lap_sap_kernel<CPT, VR>, smem_optin, dev)) return rc;
    pm_lap_sap_kernel<CPT, VR><<<batch, threads, smem, s>>>(B, 0);
    PM_LAUNCH_CHECK();
    return PM_OK;
}

static size_t pm_ls_smem_bytes(int ncp) { return (size_t)ncp * (sizeof(double) + sizeof(unsigned short)); }

extern "C" int pm_lap_solve(const float *cost, int batch, int nr, int nc, int ldc, int max_bid_rounds, int algorithm,
                            int32_t *col4row, double *total, int64_t *stats, void *workspace,
                            size_t workspace_bytes, void *stream) {
    PM_REQUIRE(cost && col4row && total && workspace, "null pointer");
    PM_REQUIRE(batch >= 1 && nr >= 1 && nc >= 1, "empty problem");
    PM_REQUIRE(nr <= nc, "need nr <= nc (transpose on the host side, as scipy does)");
    PM_REQUIRE(ldc >= nc && ldc % 4 == 0, "ldc must be >= nc and a multiple of 4");
    // (the dense kernels read a row in float4 sweeps up to the column count rounded up to 4, never further)
    PM_REQUIRE((reinterpret_cast<size_t>(cost) & 15) == 0, "cost must be 16-byte aligned");
    PM_REQUIRE(max_bid_rounds >= 0, "max_bid_rounds < 0");
    PM_REQUIRE(algorithm >= PM_LAP_ALGO_AUTO && algorithm <= PM_LAP_ALGO_DENSE_AUCTION, "unknown algorithm");
    if (nc > 24 * PM_LAP_MAX_THREADS) {
        pm_set_error("pm_lap_solve: nc = %d > %d columns not supported by the single-CTA path", nc,
                     24 * PM_LAP_MAX_THREADS);
        return PM_ERR_UNSUPPORTED;
    }
    if (workspace_bytes < pm_lap_workspace_bytes(batch, nr, nc)) {
        pm_set_error("pm_lap_solve: workspace too small");
        return PM_ERR_WORKSPACE;
    }
    cudaStream_t s = pm_stream(stream);
    PmLapBatch B;
    B.cost = cost; B.cost_stride = (size_t)nr * ldc; B.nr = nr; B.nr_real = nr; B.nc = nc; B.ldc = ldc;
    B.ncp = (nc + 3) & ~3;
    // Few slack columns (and none): solved as a SQUARE problem with nc - nr dummy rows of zero cost, eps-scaling first
    // (see below).  The dummies take the columns that stay unassigned, so the optimum over the real rows is the same.
    bool square = false;
    if (max_bid_rounds > 0 && algorithm != PM_LAP_ALGO_DENSE_AUCTION && nr >= 64) {
        // above this slack the pure epsilon = 0 schedule is faster
        square = (double)(nc - nr) <= PM_LAP_SQUARE_SLACK_DEFAULT * (double)nc;
        const char *e = getenv("PM_LAP_EPS_SCALING");
        if (e) square = atoi(e) != 0;
    }
    if (square) B.nr = nc;
    B.L = pm_lap_layout(nc, B.ncp);                           // (sized for the square case: rows <= nc)
    B.progress = (int32_t *)workspace;
    B.scale = (double *)((char *)workspace + 256);
    B.zero_row = (const float *)((char *)workspace + 256 + pm_lap_align((size_t)batch * 2 * sizeof(double)));
    B.eps_factor = 0.0;
    B.ws = (char *)workspace + pm_lap_header_bytes(batch, B.ncp);
    B.col4row = col4row; B.stats = (long long *)stats; B.total = total;
    // one "round" of the sparse auction = a budget of one bid per row, spread over the 32 warps
    const int rows = B.nr;                               // incl. the dummy rows of a squared problem
    B.max_bids = ((long long)max_bid_rounds * rows + 31) / 32;
    B.max_bids_tail = B.max_bids;
    int bulk_ctas = (rows + 127) / 128;                    // 8 warps per CTA: ~16 rows per warp at the start
    if (bulk_ctas > 64) bulk_ctas = 64;
    {
        const char *e = getenv("PM_LAP_STOP_LIVE");      // tuning knobs
        B.stop_live = e ? atoi(e) : 4;
        e = getenv("PM_LAP_BULK_CTAS");
        if (e && atoi(e) > 0) bulk_ctas = atoi(e);
        B.bulk_warps = bulk_ctas * 8;
        e = getenv("PM_LAP_BULK_STOP");
        B.bulk_stop_live = e ? atoi(e) : (B.bulk_warps / 16 > 8 ? B.bulk_warps / 16 : 8);   // measured optimum at 8k: 24-32 of 512
        // Safety net.  A typical 8k matrix needs 17-36 bids per row in total.  Problems without slack columns
        // (nr == nc) need an order of magnitude more, almost all of them in long sequential price wars that the
        // augmenting-path phase settles much faster: cap the auction at ~64 bids per row (bulk) + ~16 (tail),
        // with a 4x allowance for imbalance between warps.
        const long long cap_bulk = 4ll * 64 * rows / B.bulk_warps, cap_tail = 4ll * 16 * rows / 32;
        if (B.max_bids > (cap_bulk > 1024 ? cap_bulk : 1024)) B.max_bids = cap_bulk > 1024 ? cap_bulk : 1024;
        if (B.max_bids_tail > (cap_tail > 1024 ? cap_tail : 1024)) B.max_bids_tail = cap_tail > 1024 ? cap_tail : 1024;
        e = getenv("PM_LAP_BULK_PATIENCE");
        B.bulk_patience = e ? atoi(e) : 50;
    }

    int dev = 0, smem_optin = 0;
    PM_CUDA_TRY(cudaGetDevice(&dev));
    PM_CUDA_TRY(cudaDeviceGetAttribute(&smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
    size_t ls_smem = pm_ls_smem_bytes(B.ncp);
    const bool sparse_fits = rows <= (int)PM_LS_MAX_ROWS && ls_smem + 2048 <= (size_t)smem_optin;
    B.ring_cap = pm_ls_ring_cap(rows);
    B.ring_in_smem = ls_smem + (size_t)B.ring_cap * 2 + 2048 <= (size_t)smem_optin;
    if (B.ring_in_smem) ls_smem += (size_t)B.ring_cap * 2;
    if (algorithm == PM_LAP_ALGO_SPARSE_AUCTION && !sparse_fits) {
        pm_set_error("pm_lap_solve: %d x %d does not fit the sparse auction (prices in shared memory)", nr, nc);
        return PM_ERR_UNSUPPORTED;
    }
    if (algorithm == PM_LAP_ALGO_AUTO) algorithm = sparse_fits ? PM_LAP_ALGO_SPARSE_AUCTION : PM_LAP_ALGO_DENSE_AUCTION;
    if (algorithm != PM_LAP_ALGO_SPARSE_AUCTION && square) { square = false; B.nr = nr; }   // (only the sparse auction bids for dummy rows)
    B.path = square ? PM_LAP_PATH_SQUARED : 0;
    if (max_bid_rounds > 0)
        B.path |= algorithm == PM_LAP_ALGO_SPARSE_AUCTION
                      ? PM_LAP_PATH_SPARSE_AUCTION | (B.ring_in_smem ? PM_LAP_PATH_RING_SMEM : 0)
                      : PM_LAP_PATH_DENSE_AUCTION;

    pm_lap_init_kernel<<<dim3(32, batch), 256, 0, s>>>(B);
    PM_LAUNCH_CHECK();
    if (max_bid_rounds > 0 && algorithm == PM_LAP_ALGO_SPARSE_AUCTION) {
        int sms = 0;
        PM_CUDA_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
        int blocks = (rows + 7) / 8;                       // 8 warps (rows) per CTA per sweep
        const int cap = (sms * 8 + batch - 1) / batch;   // ~8 resident CTAs per SM over the whole batch
        if (blocks > cap) blocks = cap;
        pm_ls_build_lists<false><<<dim3(blocks, batch), 256, 0, s>>>(B);
        PM_LAUNCH_CHECK();
        // the tail kernel is issue-bound: ask for more than half of an SM's shared memory so that two of its
        // 1024-thread CTAs (a batch of matrices) are never placed on the same SM
        size_t tail_smem = ls_smem;
        if (tail_smem < 120 * 1024 && (size_t)smem_optin >= 120 * 1024 + 2048) tail_smem = 120 * 1024;
        if (int rc = pm_lap_raise_smem_limit(pm_ls_auction_kernel, smem_optin, dev)) return rc;
        // Problems WITHOUT slack columns (nr == nc: every column must be sold) are where an epsilon = 0 auction
        // degenerates into long sequential price wars (8000 x 8000: seconds).  They get eps-scaling first: a few
        // phases of the same certified bids with increment + eps (eps = a fraction of the matrix' own cost scale,
        // divided by theta from phase to phase; every phase restarts with all rows free and keeps the prices), which
        // brings the prices within eps of an optimal dual solution with ~30 bids per row in total, all of them with
        // thousands of rows bidding in parallel.  The tight filter (pm_ls_build_lists<true>) then keeps the exactly
        // tight edges as the warm start of the exact (epsilon = 0) phase + augmenting paths below, so the result is
        // the exact optimum as before.  (With slack columns the prices of columns that end up unassigned would have
        // to return to zero, which eps-scaling cannot guarantee: those keep the pure epsilon = 0 schedule.)
        if (square) {
            // The end of an eps phase is a handful of chains that fight sequentially (measured at 8000 x 8000: bulk
            // kernel 4.0 / 0.8 / 0.4 ms, then 54 / 31 / 14 ms of ONE CTA finishing phases 1-3 to the last row).  The phases
            // only prepare prices (exactness comes from the finish below), so they are TRUNCATED: the bulk kernel ends
            // when its parallelism has collapsed, and the tail kernel (where the dummies bid) stops carrying displaced
            // rows once PM_LAP_EPS_STOP_LIVE warps are left.
            const int stop_live = B.stop_live;
            B.stop_live = PM_LAP_EPS_STOP_LIVE;
            double factor = PM_LAP_EPS0;
            for (int k = 0; k < PM_LAP_EPS_PHASES; ++k, factor /= PM_LAP_EPS_THETA) {
                B.eps_factor = factor;
                if (k > 0) {
                    pm_ls_phase_reset_kernel<<<dim3(32, batch), 256, 0, s>>>(B);
                    PM_LAUNCH_CHECK();
                }
                pm_ls_bulk_kernel<<<batch * bulk_ctas, 256, 0, s>>>(B, bulk_ctas);
                PM_LAUNCH_CHECK();
                pm_ls_auction_kernel<<<batch, 1024, tail_smem, s>>>(B);
                PM_LAUNCH_CHECK();
            }
            B.eps_factor = 0.0;
            B.stop_live = stop_live;
            if (B.nr > B.nr_real) {
                pm_ls_equalise_dummies_kernel<<<batch, 1024, 0, s>>>(B);
                PM_LAUNCH_CHECK();
            }
            pm_ls_build_lists<true><<<dim3(blocks, batch), 256, 0, s>>>(B);       // lists at these prices + tight filter
            PM_LAUNCH_CHECK();
        } else {
            pm_ls_bulk_kernel<<<batch * bulk_ctas, 256, 0, s>>>(B, bulk_ctas);
            PM_LAUNCH_CHECK();
        }
        pm_ls_auction_kernel<<<batch, 1024, tail_smem, s>>>(B);                   // exact phase (rest of it)
        PM_LAUNCH_CHECK();
    } else if (max_bid_rounds > 0) {
        int sms = 0, per_sm = 0;
        PM_CUDA_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
        PM_CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, pm_lap_bid_persistent, PM_LAP_BID_THREADS, 0));
        if (per_sm < 1) { pm_set_error("pm_lap_solve: bidding kernel does not fit on an SM"); return PM_ERR_CUDA; }
        if (per_sm > 1) per_sm = 1;          // one CTA per SM: the grid barrier scales with the CTA count
        int grid = sms * per_sm;
        void *args[] = {(void *)&B, (void *)&batch, (void *)&max_bid_rounds};
        PM_CUDA_TRY(cudaLaunchCooperativeKernel((const void *)pm_lap_bid_persistent, dim3(grid), dim3(PM_LAP_BID_THREADS),
                                                args, 0, s));
        PM_LAUNCH_CHECK();
    }
    int rc;
    const size_t ss_smem = (size_t)B.ncp * (8 + 8 + 2 + 2 + 2 + 1);
    if (max_bid_rounds > 0 && algorithm == PM_LAP_ALGO_SPARSE_AUCTION && ss_smem + 2048 <= (size_t)smem_optin) {
        if (int rc = pm_lap_raise_smem_limit(pm_lap_sap_sparse_kernel, smem_optin, dev)) return rc;
        B.path |= PM_LAP_PATH_SAP_SPARSE;
        pm_lap_sap_sparse_kernel<<<batch, PM_SS_THREADS, ss_smem, s>>>(B);
        PM_LAUNCH_CHECK();
        rc = PM_OK;
    } else if (nc <= PM_LAP_CPT * PM_LAP_MAX_THREADS) {
        int threads = ((nc + PM_LAP_CPT - 1) / PM_LAP_CPT + 31) & ~31;
        if (threads < 64) threads = 64;
        if (threads > PM_LAP_MAX_THREADS) threads = PM_LAP_MAX_THREADS;
        B.path |= PM_LAP_PATH_SAP_DENSE8;
        rc = pm_lap_launch_sap<PM_LAP_CPT, true>(B, batch, threads, smem_optin, dev, s);
    } else if (nc <= 16 * PM_LAP_MAX_THREADS) {
        B.path |= PM_LAP_PATH_SAP_DENSE16;
        rc = pm_lap_launch_sap<16, false>(B, batch, PM_LAP_MAX_THREADS, smem_optin, dev, s);
    } else {
        B.path |= PM_LAP_PATH_SAP_DENSE24;
        rc = pm_lap_launch_sap<24, false>(B, batch, PM_LAP_MAX_THREADS, smem_optin, dev, s);
    }
    return rc;
}
