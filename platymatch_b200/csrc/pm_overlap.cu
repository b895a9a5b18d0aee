// pm_overlap.cu — two label volumes -> their contingency table (DESIGN §8 row 7).
//
// For volumes A and B of one shape, every pair of ids (a, b) != (0, 0) that meet at some voxel and the number of such
// voxels (ids <= 0 are background, as in pm_label_centroids).  This is what segmentation metrics are built from:
// instance sizes are its row and column sums, IoU(a, b) = n / (|A_a| + |B_b| - n).
//
// ONE streaming pass reads both volumes once (HBM-bound), with the structure of pm_label_stream_kernel (pm_labels.cu):
// a chunk is 8 consecutive voxels of each volume (two 16-byte loads for int32, one for uint16), loads are software-
// pipelined through two register buffers, one wave of resident CTAs, and the all-background case costs a ballot per
// chunk.  A chunk that is non-zero on either side is queued per warp in shared memory and processed later, one chunk
// per lane.  There a thread keeps ONE pending run {key, count} across everything it processes: voxels with the key of
// the run extend it, any other non-background key ends it.  A run needs no coordinates, so it may cross image rows and
// chunks (a large region of one pair costs one insert per thread, not one per chunk).  An ended run is one insert into
// an open-addressing hash table: key a << 32 | b (0 = empty slot), 64-bit atomicCAS to claim a slot, 64-bit atomicAdd
// for the count.  Keys only ever go from 0 to their final value, so a stale read of a slot is harmless: a stale 0 goes
// to the CAS, which returns the true content.  A pair that finds no slot within PM_OVERLAP_MAX_PROBE probes is not
// stored: its voxels are added to a dropped-voxel count, and the caller reruns with a larger table.
// A compaction kernel writes the occupied slots (any order) and the pair count.
#include "pm_common.cuh"

#define PM_OVERLAP_MAX_PROBE 128   // linear probes before a pair counts as overflow (a table at load <= 1/2 needs ~2)
#define PM_OVERLAP_QCAP 64         // queue slots per warp (a trip adds at most 32 per chunk slot)

typedef unsigned long long u64;

__device__ __forceinline__ u64 pm_ov_hash(u64 x) {            // splitmix64's finaliser: keys of a grid of ids spread
    x ^= x >> 30; x *= 0xbf58476d1ce4e5b9ull;
    x ^= x >> 27; x *= 0x94d049bb133111ebull;
    return x ^ (x >> 31);
}

__device__ __noinline__ void pm_ov_insert(u64 key, u64 n, u64 *keys, u64 *__restrict__ counts, u64 mask,
                                          u64 *__restrict__ dropped) {
    u64 h = pm_ov_hash(key) & mask;
    const u64 probes = mask < PM_OVERLAP_MAX_PROBE ? mask + 1 : PM_OVERLAP_MAX_PROBE;
    for (u64 p = 0; p < probes; ++p, h = (h + 1) & mask) {
        u64 k = keys[h];                                          // (a stale 0 is resolved by the CAS)
        if (k == 0ull) {
            k = atomicCAS(keys + h, 0ull, key);
            if (k == 0ull) k = key;
        }
        if (k == key) {
            atomicAdd(counts + h, n);
            return;
        }
    }
    atomicAdd(dropped, n);
}

// 16-byte loads per 8-voxel chunk: 2 for int32, 1 for uint16
template <typename T> __host__ __device__ constexpr int pm_ov_loads() { return (int)sizeof(T) / 2; }

template <typename TA, typename TB> struct PmOvChunk {
    uint4 a[pm_ov_loads<TA>()];
    uint4 b[pm_ov_loads<TB>()];
};

// id e of a queued chunk (read from shared memory), background (<= 0) as 0
template <typename T, int L> __device__ __forceinline__ unsigned pm_ov_id(const uint4 (&q)[L], int e) {
    if constexpr (sizeof(T) == 4) return (unsigned)max(reinterpret_cast<const int *>(q)[e], 0);
    else return reinterpret_cast<const unsigned short *>(q)[e];
}

struct PmOvRun { u64 key, n; };

__device__ __forceinline__ void pm_ov_add(PmOvRun &run, u64 key, u64 *keys, u64 *counts, u64 mask, u64 *dropped) {
    if (key == 0ull) return;                                      // (0, 0): not in the table, does not end the run
    if (key != run.key) {
        if (run.n) pm_ov_insert(run.key, run.n, keys, counts, mask, dropped);
        run.key = key;
        run.n = 0;
    }
    ++run.n;
}

// (a rolled loop over the chunk in shared memory: one call site of the insert, no chunk held in registers)
template <typename TA, typename TB>
__device__ __forceinline__ void pm_ov_chunk(const PmOvChunk<TA, TB> &c, PmOvRun &run, u64 *keys, u64 *counts, u64 mask,
                                            u64 *dropped) {
#pragma unroll 1
    for (int e = 0; e < 8; ++e)
        pm_ov_add(run, ((u64)pm_ov_id<TA>(c.a, e) << 32) | pm_ov_id<TB>(c.b, e), keys, counts, mask, dropped);
}

// chunks per register buffer: about four 16-byte loads per buffer, as in pm_label_stream_kernel
template <typename TA, typename TB> __host__ __device__ constexpr int pm_ov_half() {
    return pm_ov_loads<TA>() + pm_ov_loads<TB>() >= 3 ? 1 : 2;
}

// la, lb 16-byte aligned; the voxels beyond the last full chunk are handled by thread 0 of block 0
template <typename TA, typename TB>
__global__ void __launch_bounds__(256, 3) pm_overlap_stream_kernel(const TA *__restrict__ la, const TB *__restrict__ lb,
                                                                size_t n_vox, u64 *keys, u64 *__restrict__ counts,
                                                                u64 mask, u64 *__restrict__ dropped) {
    constexpr int LA = pm_ov_loads<TA>(), LB = pm_ov_loads<TB>(), HALF = pm_ov_half<TA, TB>();
    __shared__ PmOvChunk<TA, TB> s_q[8][PM_OVERLAP_QCAP];
    const size_t n_chunks = n_vox / 8;
    const uint4 *__restrict__ pa = reinterpret_cast<const uint4 *>(la);
    const uint4 *__restrict__ pb = reinterpret_cast<const uint4 *>(lb);
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const unsigned lt = (1u << lane) - 1u;
    PmOvRun run = {0ull, 0ull};
    int queued = 0;                                               // warp-uniform
    auto flush = [&]() {
        __syncwarp();
        for (int i = lane; i < queued; i += 32) pm_ov_chunk<TA, TB>(s_q[w][i], run, keys, counts, mask, dropped);
        queued = 0;
        __syncwarp();
    };
    const size_t step = stride * HALF;
    auto load = [&](PmOvChunk<TA, TB> (&q)[HALF], size_t base) {
#pragma unroll
        for (int u = 0; u < HALF; ++u) {
            const size_t idx = base + lane + (size_t)u * stride;
#pragma unroll
            for (int i = 0; i < LA; ++i) q[u].a[i] = make_uint4(0u, 0u, 0u, 0u);
#pragma unroll
            for (int i = 0; i < LB; ++i) q[u].b[i] = make_uint4(0u, 0u, 0u, 0u);
            if (idx < n_chunks) {                                 // streamed once: evict first
#pragma unroll
                for (int i = 0; i < LA; ++i) q[u].a[i] = __ldcs(pa + idx * LA + i);
#pragma unroll
                for (int i = 0; i < LB; ++i) q[u].b[i] = __ldcs(pb + idx * LB + i);
            }
        }
    };
    auto examine = [&](const PmOvChunk<TA, TB> (&q)[HALF]) {
#pragma unroll
        for (int u = 0; u < HALF; ++u) {
            unsigned any = 0u;
#pragma unroll
            for (int i = 0; i < LA; ++i) any |= q[u].a[i].x | q[u].a[i].y | q[u].a[i].z | q[u].a[i].w;
#pragma unroll
            for (int i = 0; i < LB; ++i) any |= q[u].b[i].x | q[u].b[i].y | q[u].b[i].z | q[u].b[i].w;
            const bool fg = any != 0u;
            const unsigned bal = __ballot_sync(0xffffffffu, fg);
            if (bal) {
                if (queued + __popc(bal) > PM_OVERLAP_QCAP) flush();
                if (fg) s_q[w][queued + __popc(bal & lt)] = q[u];
                queued += __popc(bal);
            }
        }
        if (queued >= 32) flush();
    };
    // (the loop bound is the warp's first chunk, so that all 32 lanes stay in the loop for the ballots)
    PmOvChunk<TA, TB> qa[HALF], qb[HALF];
    size_t base = (size_t)blockIdx.x * blockDim.x + (size_t)w * 32;
    if (base < n_chunks) load(qa, base);
    while (base < n_chunks) {
        const size_t next = base + step;                          // (warp-uniform)
        if (next < n_chunks) load(qb, next);
        examine(qa);
        if (!(next < n_chunks)) break;
        const size_t next2 = next + step;
        if (next2 < n_chunks) load(qa, next2);
        examine(qb);
        base = next2;
    }
    flush();
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        for (size_t v = n_chunks * 8; v < n_vox; ++v) {           // < 8 voxels
            const u64 a = (u64)(unsigned)max((int)la[v], 0), b = (u64)(unsigned)max((int)lb[v], 0);
            pm_ov_add(run, (a << 32) | b, keys, counts, mask, dropped);
        }
    }
    if (run.n) pm_ov_insert(run.key, run.n, keys, counts, mask, dropped);
}

// occupied slots -> keys_out / counts_out (any order), n_out[0] = pairs, n_out[1] = dropped voxels (n_out zeroed)
__global__ void __launch_bounds__(256) pm_overlap_compact_kernel(const u64 *__restrict__ keys,
                                                                 const u64 *__restrict__ counts, u64 capacity,
                                                                 const u64 *__restrict__ dropped,
                                                                 u64 *__restrict__ keys_out,
                                                                 u64 *__restrict__ counts_out, u64 *__restrict__ n_out) {
    const int lane = threadIdx.x & 31;
    const u64 stride = (u64)gridDim.x * blockDim.x;
    // (the loop bound is the warp's first slot: all 32 lanes stay in the loop for the ballot)
    for (u64 w0 = (u64)blockIdx.x * blockDim.x + (threadIdx.x & ~31u); w0 < capacity; w0 += stride) {
        const u64 i = w0 + lane;
        const u64 k = i < capacity ? keys[i] : 0ull;
        const unsigned bal = __ballot_sync(0xffffffffu, k != 0ull);
        if (!bal) continue;
        u64 first = 0;
        if (lane == __ffs(bal) - 1) first = atomicAdd(n_out, (u64)__popc(bal));
        first = __shfl_sync(0xffffffffu, first, __ffs(bal) - 1);
        if (k) {
            const u64 pos = first + __popc(bal & ((1u << lane) - 1u));
            keys_out[pos] = k;
            counts_out[pos] = counts[i];
        }
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) n_out[1] = *dropped;
}

// workspace: the table's keys [capacity], counts [capacity], then the dropped-voxel count
extern "C" size_t pm_label_overlap_workspace_bytes(uint64_t capacity) {
    if (capacity > ((uint64_t)1 << 58)) return (size_t)-1;
    return (size_t)capacity * 2 * sizeof(u64) + 16;
}

template <typename TA, typename TB>
static int pm_overlap_run(const TA *la, const TB *lb, size_t n_vox, u64 capacity, u64 *keys_out, u64 *counts_out,
                          u64 *n_out, u64 *ws, cudaStream_t s) {
    u64 *keys = ws, *counts = ws + capacity, *dropped = ws + 2 * capacity;
    PM_CUDA_TRY(cudaMemsetAsync(ws, 0, pm_label_overlap_workspace_bytes(capacity), s));
    PM_CUDA_TRY(cudaMemsetAsync(n_out, 0, 2 * sizeof(u64), s));
    int dev = 0, sms = 0;
    PM_CUDA_TRY(cudaGetDevice(&dev));
    PM_CUDA_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    const size_t per_cta = (size_t)256 * pm_ov_half<TA, TB>();
    int blocks = 0;
    if (int rc = pm_resident_wave((const void *)pm_overlap_stream_kernel<TA, TB>, 256, dev, sms,
                                  (n_vox / 8 + per_cta - 1) / per_cta, &blocks))
        return rc;
    pm_overlap_stream_kernel<TA, TB><<<blocks, 256, 0, s>>>(la, lb, n_vox, keys, counts, capacity - 1, dropped);
    PM_LAUNCH_CHECK();
    const u64 cwant = (capacity + 255) / 256;
    const int cblocks = (int)(cwant < (u64)sms * 8 ? cwant : (u64)sms * 8);
    pm_overlap_compact_kernel<<<cblocks, 256, 0, s>>>(keys, counts, capacity, dropped, keys_out, counts_out, n_out);
    PM_LAUNCH_CHECK();
    return PM_OK;
}

extern "C" int pm_label_overlap(const void *labels_a, int dtype_a, const void *labels_b, int dtype_b, int nz, int ny,
                                int nx, uint64_t capacity, uint64_t *keys, uint64_t *counts, uint64_t *n_out,
                                void *workspace, size_t workspace_bytes, void *stream) {
    PM_REQUIRE(labels_a && labels_b && keys && counts && n_out && workspace, "null pointer");
    PM_REQUIRE(pm_volume_dtype_ok(dtype_a, false) && pm_volume_dtype_ok(dtype_b, false),
               "dtype must be PM_LABEL_I32 or PM_LABEL_U16");
    PM_REQUIRE(nz >= 1 && ny >= 1 && nx >= 1, "every extent must be >= 1");
    PM_REQUIRE(capacity >= 1 && capacity <= ((uint64_t)1 << 58) && (capacity & (capacity - 1)) == 0,
               "capacity must be a power of two");
    const void *ptrs[6] = {labels_a, labels_b, keys, counts, n_out, workspace};
    for (const void *p : ptrs) PM_REQUIRE(((uintptr_t)p & 15) == 0, "pointers must be 16-byte aligned");
    if (workspace_bytes < pm_label_overlap_workspace_bytes(capacity)) {
        pm_set_error("pm_label_overlap: workspace too small");
        return PM_ERR_WORKSPACE;
    }
    const size_t n_vox = (size_t)nz * ny * nx;
    u64 *ws = (u64 *)workspace, *ko = (u64 *)keys, *co = (u64 *)counts, *no = (u64 *)n_out;
    return pm_volume_dispatch<false>(dtype_a, [&](auto a) {
        return pm_volume_dispatch<false>(dtype_b, [&](auto b) {
            return pm_overlap_run((const decltype(a) *)labels_a, (const decltype(b) *)labels_b, n_vox, capacity, ko, co,
                                  no, ws, pm_stream(stream));
        });
    });
}
