// pm_labels.cu — label image -> nucleus centroids and sizes (SURVEY §8f row 2).
//
// Reference: platymatch/_dock_widget.py:497-521 (inside EstimateTransform._click_run): for every
// non-zero id of np.unique(label_image), z, y, x = np.where(image == id); centroid = (mean z, mean y,
// mean x); size = anisotropy * len(z) — one full pass over the volume PER ID (O(ids x voxels)).
//
// Here: ONE streaming pass over the volume (HBM-bound: 4 B per voxel read once).  Every thread
// loads 4 x four consecutive voxels; lanes of a warp that hold the same non-zero id form a group
// (match.any), the group's voxel count and coordinate sums are reduced with REDUX and its leader
// issues four 64-bit atomic adds on the id's accumulator
// {count, sum z, sum y, sum x}.  The sums are exact integers, so mean = sum / count rounds once and
// equals np.mean of the integer coordinates bit for bit (sums stay far below 2^53).
// A second small kernel compacts the non-empty ids in ascending order (np.unique order).
#include <stdlib.h>
#include "pm_common.cuh"

template <typename T>
__global__ void __launch_bounds__(256) pm_label_max_kernel(const T *__restrict__ labels, size_t n_vox,
                                                           unsigned *__restrict__ max_id) {
    unsigned m = 0u;
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t v = (size_t)blockIdx.x * blockDim.x + threadIdx.x; v < n_vox; v += stride) {
        const long long id = (long long)labels[v];
        m = max(m, id > 0 ? (unsigned)id : 0u);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = max(m, __shfl_xor_sync(0xffffffffu, m, o));
    if ((threadIdx.x & 31) == 0 && m) atomicMax(max_id, m);
}

template <typename T>
__device__ __forceinline__ void pm_label_load4(const T *__restrict__ labels, size_t base, size_t n_vox, bool aligned,
                                               int ids[4]) {
    if (base + 3 < n_vox && aligned) {          // one 16- / 8-byte load
        if (sizeof(T) == 4) {
            const int4 q = __ldcs(reinterpret_cast<const int4 *>(labels + base));     // streamed once: evict first
            ids[0] = q.x; ids[1] = q.y; ids[2] = q.z; ids[3] = q.w;
        } else {
            const ushort4 q = __ldcs(reinterpret_cast<const ushort4 *>(labels + base));
            ids[0] = q.x; ids[1] = q.y; ids[2] = q.z; ids[3] = q.w;
        }
    } else {
#pragma unroll
        for (int e = 0; e < 4; ++e) ids[e] = (base + e < n_vox) ? (int)labels[base + e] : 0;
    }
}

#define PM_LABEL_UNROLL 4      // independent 16-byte loads in flight per thread

struct PmVox { unsigned z, y, x; };

// advance a voxel coordinate by a fixed linear step given as (dz, dy, dx), dy < ny, dx < nx
__device__ __forceinline__ void pm_vox_advance(PmVox &v, const PmVox &d, unsigned ny, unsigned nx) {
    v.x += d.x;
    unsigned cy = 0;
    if (v.x >= nx) { v.x -= nx; cy = 1; }
    v.y += d.y + cy;
    unsigned cz = 0;
    if (v.y >= ny) { v.y -= ny; cz = 1; }
    v.z += d.z + cz;
}

template <typename T>
__global__ void __launch_bounds__(256) pm_label_accumulate_kernel(const T *__restrict__ labels, int nz, int ny, int nx,
                                                                  unsigned table_size,
                                                                  unsigned long long *__restrict__ acc) {
    const size_t n_vox = (size_t)nz * ny * nx;
    const size_t plane = (size_t)ny * nx;
    const size_t sweep = (size_t)gridDim.x * blockDim.x * 4;          // voxels covered by one load of the whole grid
    const bool aligned = (reinterpret_cast<size_t>(labels) & 15) == 0;
    const int lane = threadIdx.x & 31;
    // voxel coordinates of this thread's first voxel and of one sweep: 64-bit divisions once, carries afterwards
    const size_t first = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) * 4;
    PmVox pos, step;
    pos.z = (unsigned)(first / plane);
    pos.y = (unsigned)((first - (size_t)pos.z * plane) / nx);
    pos.x = (unsigned)(first - (size_t)pos.z * plane - (size_t)pos.y * nx);
    step.z = (unsigned)(sweep / plane);
    step.y = (unsigned)((sweep - (size_t)step.z * plane) / nx);
    step.x = (unsigned)(sweep - (size_t)step.z * plane - (size_t)step.y * nx);
    // the trip count is uniform across a warp (bounds are checked per load), so the warp stays converged for
    // the match / redux collectives below
    const size_t warp_base = ((size_t)blockIdx.x * blockDim.x + (threadIdx.x & ~31)) * 4;
    for (size_t wb = warp_base; wb < n_vox; wb += sweep * PM_LABEL_UNROLL) {
        int ids[PM_LABEL_UNROLL][4];
        bool any_fg = false;
#pragma unroll
        for (int u = 0; u < PM_LABEL_UNROLL; ++u) {
            const size_t base = wb + (size_t)u * sweep + (size_t)lane * 4;
            ids[u][0] = ids[u][1] = ids[u][2] = ids[u][3] = 0;
            if (base < n_vox) pm_label_load4(labels, base, n_vox, aligned, ids[u]);
            any_fg |= (ids[u][0] | ids[u][1] | ids[u][2] | ids[u][3]) != 0;
        }
        if (__any_sync(0xffffffffu, any_fg)) {
#pragma unroll
            for (int u = 0; u < PM_LABEL_UNROLL; ++u) {
                const bool fg = (ids[u][0] | ids[u][1] | ids[u][2] | ids[u][3]) != 0;
                if (__any_sync(0xffffffffu, fg)) {
                    // common case: the (up to four) foreground voxels of a thread belong to ONE nucleus and sit in
                    // one image row -> the thread contributes one pre-summed item, the warp needs one round
                    int id1 = 0, k = 0;
                    unsigned sxl = 0;
                    bool simple = pos.x + 3 < (unsigned)nx;
#pragma unroll
                    for (int e = 0; e < 4; ++e) {
                        const int id = ids[u][e];
                        if (id != 0) {
                            if (id < 0 || (unsigned)id >= table_size) continue;      // background / out of table
                            if (id1 == 0) id1 = id;
                            simple &= (id == id1);
                            ++k;
                            sxl += pos.x + e;
                        }
                    }
                    if (__all_sync(0xffffffffu, simple)) {
                        // one pre-summed item per thread, added with four fire-and-forget reductions (RED.ADD.64):
                        // cheaper than grouping the 1-3 lanes of a nucleus row first
                        if (k > 0) {
                            unsigned long long *a = acc + (size_t)id1 * 4;
                            atomicAdd(a + 0, (unsigned long long)k);
                            atomicAdd(a + 1, (unsigned long long)((unsigned)k * pos.z));
                            atomicAdd(a + 2, (unsigned long long)((unsigned)k * pos.y));
                            atomicAdd(a + 3, (unsigned long long)sxl);
                        }
                    } else {
                        PmVox p = pos;
#pragma unroll
                        for (int e = 0; e < 4; ++e) {
                            const int id = ids[u][e];
                            const bool valid = id > 0 && (unsigned)id < table_size;
                            const unsigned voters = __ballot_sync(0xffffffffu, valid);
                            if (voters != 0u && valid) {
                                // lanes holding the same id: one group, its sums by REDUX, one leader
                                const unsigned peers = __match_any_sync(voters, (unsigned)id);
                                const unsigned sz = __reduce_add_sync(peers, p.z);
                                const unsigned sy = __reduce_add_sync(peers, p.y);
                                const unsigned sx = __reduce_add_sync(peers, p.x);
                                if (lane == __ffs(peers) - 1) {
                                    unsigned long long *a = acc + (size_t)id * 4;
                                    atomicAdd(a + 0, (unsigned long long)__popc(peers));
                                    atomicAdd(a + 1, (unsigned long long)sz);
                                    atomicAdd(a + 2, (unsigned long long)sy);
                                    atomicAdd(a + 3, (unsigned long long)sx);
                                }
                            }
                            if (++p.x >= (unsigned)nx) { p.x = 0; if (++p.y >= (unsigned)ny) { p.y = 0; ++p.z; } }
                        }
                    }
                }
                pm_vox_advance(pos, step, (unsigned)ny, (unsigned)nx);
            }
        } else {
#pragma unroll
            for (int u = 0; u < PM_LABEL_UNROLL; ++u) pm_vox_advance(pos, step, (unsigned)ny, (unsigned)nx);
        }
    }
}

// ---- round 2: the streaming kernel -------------------------------------------------------------------------
// The kernel above is bound by instruction issue (~300 instructions per 16 voxels in volumes where every other
// 128-voxel run touches a nucleus: warp votes, REDUX groups, carry arithmetic for the voxel coordinates on every load).
// A label volume is ~98 % background, so this one spends ~8 instructions per 16-byte chunk on the common case and
// does everything else per THREAD, only for chunks that contain foreground: no warp collective anywhere (a chunk
// is 4 / 8 consecutive voxels of one thread), the voxel coordinates come from two divisions when they are needed,
// and the chunk's voxels are run-length merged (same id, same image row) into items {count, k z, k y, sum x} that are
// added with four fire-and-forget 64-bit reductions.  Same exact integer sums as before.
template <typename T>
__device__ __noinline__ void pm_label_chunk(const uint4 q, size_t v0, unsigned plane, unsigned ny, unsigned nx,
                                            unsigned table_size, unsigned long long *__restrict__ acc) {
    constexpr int VPC = 16 / (int)sizeof(T);
    int ids[VPC];
    if (sizeof(T) == 4) {
        ids[0] = (int)q.x; ids[1] = (int)q.y; ids[2] = (int)q.z; ids[3] = (int)q.w;
    } else {
        const unsigned w[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
        for (int e = 0; e < VPC; ++e) ids[e] = (int)((w[e >> 1] >> ((e & 1) * 16)) & 0xffffu);
    }
    unsigned pz, rem;
    if (v0 <= 0xFFFFFFFFull) {                    // (almost always: a 32-bit division is ~5x cheaper than a 64-bit one)
        pz = (unsigned)v0 / plane;
        rem = (unsigned)v0 - pz * plane;
    } else {
        pz = (unsigned)(v0 / plane);
        rem = (unsigned)(v0 - (size_t)pz * plane);
    }
    unsigned py = rem / nx, px = rem - py * nx;
    int run_id = 0;
    unsigned k = 0, sx = 0, ry = 0, rz = 0;
#pragma unroll
    for (int e = 0; e < VPC; ++e) {
        const int id = ids[e];
        const bool valid = id > 0 && (unsigned)id < table_size;
        if (k && (!valid || id != run_id || py != ry || pz != rz)) {          // the run ends: flush it
            unsigned long long *a = acc + (size_t)run_id * 4;
            atomicAdd(a + 0, (unsigned long long)k);
            atomicAdd(a + 1, (unsigned long long)k * rz);
            atomicAdd(a + 2, (unsigned long long)k * ry);
            atomicAdd(a + 3, (unsigned long long)sx);
            k = 0; sx = 0;
        }
        if (valid) {
            if (!k) { run_id = id; ry = py; rz = pz; }
            ++k;
            sx += px;
        }
        if (++px >= nx) { px = 0; if (++py >= ny) { py = 0; ++pz; } }
    }
    if (k) {
        unsigned long long *a = acc + (size_t)run_id * 4;
        atomicAdd(a + 0, (unsigned long long)k);
        atomicAdd(a + 1, (unsigned long long)k * rz);
        atomicAdd(a + 2, (unsigned long long)k * ry);
        atomicAdd(a + 3, (unsigned long long)sx);
    }
}

#define PM_LABEL_STREAM_UNROLL 8      // independent 16-byte loads in flight per thread (128 B)
#define PM_LABEL_STREAM_HALF 4        // ... in two register buffers of 4 (software pipeline)

// labels must be 16-byte aligned; the voxels beyond the last full chunk are handled by thread 0 of block 0.
// Foreground chunks are not processed where they are found: with ~3 % of the chunks touching a nucleus, 5 of the 8
// chunk slots of a warp trip have SOME lane with foreground, and each of them ran the ~100-instruction run-length
// path with one or two live lanes (ncu, round 2: 70 warp instructions per 512 bytes, issue slots 62 % busy, 4.6 TB/s).
// Each warp therefore queues its foreground chunks {16 bytes, chunk index} in shared memory (ballot + popc) and runs
// the run-length path once 32 are waiting, one chunk per lane.
#define PM_LABEL_QCAP 64                 // queue slots per warp (a trip adds at most 32 per chunk slot)
template <typename T>
__global__ void __launch_bounds__(256, 3) pm_label_stream_kernel(const T *__restrict__ labels, int nz, int ny, int nx,
                                                              unsigned table_size, unsigned long long *__restrict__ acc) {
    constexpr int VPC = 16 / (int)sizeof(T);
    __shared__ uint4 s_q[8][PM_LABEL_QCAP];
    __shared__ unsigned s_c[8][PM_LABEL_QCAP];                   // chunk index (the host checks n_chunks < 2^32)
    const size_t n_vox = (size_t)nz * ny * nx;
    const size_t n_chunks = n_vox / VPC;
    const unsigned plane = (unsigned)ny * (unsigned)nx;          // (ny, nx < 2^26 and the host checks ny * nx < 2^32)
    const uint4 *__restrict__ p = reinterpret_cast<const uint4 *>(labels);
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const unsigned lt = (1u << lane) - 1u;
    int queued = 0;                                              // warp-uniform
    auto flush = [&]() {
        __syncwarp();
        for (int i = lane; i < queued; i += 32)
            pm_label_chunk<T>(s_q[w][i], (size_t)s_c[w][i] * VPC, plane, (unsigned)ny, (unsigned)nx, table_size, acc);
        queued = 0;
        __syncwarp();
    };
    // (the loop bound is the warp's first chunk, so that all 32 lanes stay in the loop for the ballots)
    // Software pipeline: two register buffers of PM_LABEL_STREAM_HALF chunks; the loads of the next half-trip are
    // issued BEFORE the current one is examined, so a warp always has loads in flight (the first version loaded 8,
    // examined 8, loaded 8 ...: nothing in flight while it worked).
    const size_t step = stride * PM_LABEL_STREAM_HALF;
    auto load = [&](uint4 (&q)[PM_LABEL_STREAM_HALF], size_t base) {
#pragma unroll
        for (int u = 0; u < PM_LABEL_STREAM_HALF; ++u) {
            const size_t idx = base + lane + (size_t)u * stride;
            q[u] = make_uint4(0u, 0u, 0u, 0u);
            if (idx < n_chunks) q[u] = __ldcs(p + idx);            // streamed once: evict first
        }
    };
    auto examine = [&](const uint4 (&q)[PM_LABEL_STREAM_HALF], size_t base) {
#pragma unroll
        for (int u = 0; u < PM_LABEL_STREAM_HALF; ++u) {
            const bool fg = (q[u].x | q[u].y | q[u].z | q[u].w) != 0u;
            const unsigned bal = __ballot_sync(0xffffffffu, fg);
            if (bal) {
                if (queued + __popc(bal) > PM_LABEL_QCAP) flush();
                if (fg) {
                    const int pos = queued + __popc(bal & lt);
                    s_q[w][pos] = q[u];
                    s_c[w][pos] = (unsigned)(base + lane + (size_t)u * stride);
                }
                queued += __popc(bal);
            }
        }
        if (queued >= 32) flush();
    };
    uint4 qa[PM_LABEL_STREAM_HALF], qb[PM_LABEL_STREAM_HALF];
    size_t base = (size_t)blockIdx.x * blockDim.x + (size_t)w * 32;
    if (base < n_chunks) load(qa, base);
    while (base < n_chunks) {
        const size_t next = base + step;                         // (warp-uniform)
        if (next < n_chunks) load(qb, next);
        examine(qa, base);
        if (!(next < n_chunks)) break;
        const size_t next2 = next + step;
        if (next2 < n_chunks) load(qa, next2);
        examine(qb, next);
        base = next2;
    }
    flush();
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        for (size_t v = n_chunks * VPC; v < n_vox; ++v) {         // < VPC voxels
            const int id = (int)labels[v];
            if (id > 0 && (unsigned)id < table_size) {
                const unsigned pz = (unsigned)(v / plane), rem = (unsigned)(v - (size_t)pz * plane);
                unsigned long long *a = acc + (size_t)id * 4;
                atomicAdd(a + 0, 1ull);
                atomicAdd(a + 1, (unsigned long long)pz);
                atomicAdd(a + 2, (unsigned long long)(rem / nx));
                atomicAdd(a + 3, (unsigned long long)(rem % nx));
            }
        }
    }
}

// ids with a non-zero count, ascending (np.unique order), -> ids / centroids (z, y, x) / sizes.
// One CTA per 1024 ids, one id per thread: the three float64 divisions per nucleus and the loads of its sums spread
// over as many SMs as there are chunks (one CTA doing all of it took 19-36 us for 6000 ids, a quarter of the whole
// label pass).  The output offset of a chunk = the number of non-empty ids before it, which every CTA counts itself
// from the table (b x 1024 count loads for chunk b, all in flight together: no second launch, no inter-CTA
// dependency; quadratic only in the number of chunks, ~1 ms for a million ids).
__global__ void __launch_bounds__(1024) pm_label_finalize_kernel(const unsigned long long *__restrict__ acc,
                                                                 unsigned table_size, double anisotropy, int capacity,
                                                                 int32_t *__restrict__ ids, double *__restrict__ centroids,
                                                                 double *__restrict__ sizes, int32_t *__restrict__ n_out) {
    __shared__ int s_warp[32];
    __shared__ int s_before;
    const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
    const unsigned first = 1u + blockIdx.x * 1024u;                 // ids of this chunk: first .. first + 1023
    const unsigned id = first + (unsigned)t;
    const unsigned long long cnt = (id < table_size) ? __ldcg(acc + (size_t)id * 4) : 0ull;
    unsigned long long sz = 0ull, sy = 0ull, sx = 0ull;
    if (cnt) {                                                      // (issued before the counting loop: in flight with it)
        sz = __ldcg(acc + (size_t)id * 4 + 1); sy = __ldcg(acc + (size_t)id * 4 + 2); sx = __ldcg(acc + (size_t)id * 4 + 3);
    }
    int before = 0;                                                 // non-empty ids in the chunks before this one
#pragma unroll 4
    for (unsigned j = 1u + (unsigned)t; j < first; j += 1024u) before += __ldcg(acc + (size_t)j * 4) != 0ull;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) before += __shfl_xor_sync(0xffffffffu, before, o);
    const unsigned bal = __ballot_sync(0xffffffffu, cnt != 0ull);
    if (lane == 0) s_warp[warp] = before;                           // (reused below for the in-chunk scan)
    __syncthreads();
    if (t == 0) {
        int a = 0;
        for (int w = 0; w < 32; ++w) a += s_warp[w];
        s_before = a;
    }
    __syncthreads();
    if (lane == 0) s_warp[warp] = __popc(bal);
    __syncthreads();
    if (warp == 0) {
        const int w = s_warp[lane];
        int wi = w;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int v = __shfl_up_sync(0xffffffffu, wi, o);
            if (lane >= o) wi += v;
        }
        s_warp[lane] = wi - w;                                      // exclusive offset of every warp
        if (lane == 31 && blockIdx.x == gridDim.x - 1) n_out[0] = s_before + wi;
    }
    __syncthreads();
    if (cnt) {
        const int k = s_before + s_warp[warp] + __popc(bal & ((1u << lane) - 1u));
        if (k < capacity) {
            const double c = (double)cnt;
            ids[k] = (int32_t)id;
            centroids[3 * (size_t)k + 0] = (double)sz / c;                                   // np.mean(z)
            centroids[3 * (size_t)k + 1] = (double)sy / c;
            centroids[3 * (size_t)k + 2] = (double)sx / c;
            sizes[k] = anisotropy * c;                                                       // anisotropy * len(z)  (:508)
        }
    }
}

template <typename T>
static int pm_label_run(const T *labels, int nz, int ny, int nx, unsigned table_size, double anisotropy,
                        unsigned long long *acc, int capacity, int32_t *ids, double *centroids, double *sizes,
                        int32_t *n_out, cudaStream_t s) {
    const size_t n_vox = (size_t)nz * ny * nx;
    PM_CUDA_TRY(cudaMemsetAsync(acc, 0, (size_t)table_size * 4 * sizeof(unsigned long long), s));
    int dev = 0, sms = 0;
    PM_CUDA_TRY(cudaGetDevice(&dev));
    PM_CUDA_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    size_t want = (n_vox + 1023) / 1024;
    const int blocks = (int)(want < (size_t)sms * 8 ? (want ? want : 1) : (size_t)sms * 8);   // 8 resident CTAs per SM
    const bool stream_ok = (reinterpret_cast<size_t>(labels) & 15) == 0 && (size_t)ny * nx < ((size_t)1 << 32) &&
                           n_vox / (16 / sizeof(T)) < ((size_t)1 << 32) && !getenv("PM_LABEL_WARP_KERNEL");
    if (stream_ok) {
        const size_t chunks = n_vox / (16 / sizeof(T));
        const size_t want2 = (chunks + 256 * PM_LABEL_STREAM_HALF - 1) / (256 * PM_LABEL_STREAM_HALF);
        int blocks2 = 0;
        if (int rc = pm_resident_wave((const void *)pm_label_stream_kernel<T>, 256, dev, sms, want2, &blocks2))
            return rc;
        pm_label_stream_kernel<T><<<blocks2, 256, 0, s>>>(labels, nz, ny, nx, table_size, acc);
    } else {
        pm_label_accumulate_kernel<T><<<blocks, 256, 0, s>>>(labels, nz, ny, nx, table_size, acc);
    }
    PM_LAUNCH_CHECK();
    const unsigned chunks = table_size > 1 ? (table_size - 1 + 1023) / 1024 : 1;
    pm_label_finalize_kernel<<<chunks, 1024, 0, s>>>(acc, table_size, anisotropy, capacity, ids, centroids, sizes, n_out);
    PM_LAUNCH_CHECK();
    return PM_OK;
}

template <typename T>
static int pm_label_max(const T *labels, size_t n_vox, unsigned *max_id, cudaStream_t s) {
    PM_CUDA_TRY(cudaMemsetAsync(max_id, 0, sizeof(unsigned), s));
    int dev = 0, sms = 0;
    PM_CUDA_TRY(cudaGetDevice(&dev));
    PM_CUDA_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    pm_label_max_kernel<T><<<sms * 8, 256, 0, s>>>(labels, n_vox, max_id);
    PM_LAUNCH_CHECK();
    return PM_OK;
}

extern "C" int pm_label_max_id(const void *labels, int dtype, size_t n_voxels, uint32_t *max_id, void *stream) {
    PM_REQUIRE(labels && max_id, "null pointer");
    PM_REQUIRE(pm_volume_dtype_ok(dtype, false), "dtype must be PM_LABEL_I32 or PM_LABEL_U16");
    return pm_volume_dispatch<false>(dtype, [&](auto t) {
        return pm_label_max((const decltype(t) *)labels, n_voxels, max_id, pm_stream(stream));
    });
}

extern "C" size_t pm_label_workspace_bytes(uint32_t table_size) { return (size_t)table_size * 4 * sizeof(unsigned long long); }

extern "C" int pm_label_centroids(const void *labels, int dtype, int nz, int ny, int nx, uint32_t table_size,
                                  double anisotropy, int capacity, int32_t *ids, double *centroids, double *sizes,
                                  int32_t *n_out, void *workspace, size_t workspace_bytes, void *stream) {
    PM_REQUIRE(labels && ids && centroids && sizes && n_out && workspace, "null pointer");
    PM_REQUIRE(pm_volume_dtype_ok(dtype, false), "dtype must be PM_LABEL_I32 or PM_LABEL_U16");
    PM_REQUIRE(nz >= 1 && ny >= 1 && nx >= 1 && nz < (1 << 26) && ny < (1 << 26) && nx < (1 << 26), "bad volume shape");
    PM_REQUIRE(table_size >= 1 && capacity >= 0, "bad table size / capacity");
    if (workspace_bytes < pm_label_workspace_bytes(table_size)) {
        pm_set_error("pm_label_centroids: workspace too small");
        return PM_ERR_WORKSPACE;
    }
    unsigned long long *acc = (unsigned long long *)workspace;
    return pm_volume_dispatch<false>(dtype, [&](auto t) {
        return pm_label_run((const decltype(t) *)labels, nz, ny, nx, table_size, anisotropy, acc, capacity, ids,
                            centroids, sizes, n_out, pm_stream(stream));
    });
}
