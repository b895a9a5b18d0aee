"""Multi-GPU sharding of the registration path (SURVEY.md §8e): one process per GPU,
`torch.distributed` (NCCL over NVLink on the GPU box, gloo in the CPU tests) for the plumbing.

Three ways the path shards:

  * specimen pairs      independent registrations (config 5: 12 specimens, 66 pairs).  Descriptors of the
                        specimens are computed once, spread over the ranks, and all-gathered; the pairs are then
                        pulled from ONE shared work counter (a fetch-add on the job's rendezvous store) by every
                        in-flight worker of every rank, so neither the 66 / 8 remainder nor the 8-20 ms spread of
                        the assignment stage leaves a rank idle.  No data-path collective; one all-reduce of the
                        4x4 results at the end (`register_all_pairs`).
  * hypotheses          the H {cost matrix -> LAP -> RANSAC} chains are independent -> hypothesis q is owned by
                        rank `owner_of_hypothesis(q)`; one all-gather of (inliers, 4x4) picks the winner
                        (`reduce_best_hypothesis`), every rank then refines with ICP (replicated, deterministic)
                        so all ranks return the same transform.
  * rows                for large clouds (config 4, 20k x 20k) the query rows of the descriptor kernel and the
                        rows of every cost matrix are split over ALL ranks.  Descriptor rows come back with one
                        all-gather (`allgather_counts`); cost rows are delivered to the matrix OWNER ONLY: on NCCL
                        the chi^2 kernel stores them straight into the owner's matrix through a peer-mapped window
                        (device.PeerWindow, CUDA IPC over NVLink: compute and transfer are one kernel), otherwise
                        (gloo, or peer_stores=False) with one `dist.gather` per matrix (`gather_rows_to_owner`).
                        The LAP itself does not shard across GPUs ("replicas only"): one matrix, one GPU.

The partition arithmetic and the exchange steps are plain-tensor code (CPU or CUDA), covered by world_size-2
gloo tests in tests/test_distributed_cpu.py; `register_pair_sharded` and `register_all_pairs` touch the CUDA
library and are covered by tests/test_gpu_distributed.py (torchrun, NCCL, 2 GPUs).
"""
import itertools
import collections
import threading
import time

import numpy as np


def world_info(group=None):
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized():
        return dist.get_rank(group), dist.get_world_size(group)
    return 0, 1


# ----------------------------------------------------------------------------- partitions
def shard_rows(n_rows, rank, world, align=128):
    """Row range [begin, end) of `rank`: equal shards of ceil(n/world) rounded up to `align`
    (the chi2 kernel's 128-row tile), the tail ranks may be short or empty."""
    per = -(-n_rows // world)
    per = -(-per // align) * align
    begin = min(rank * per, n_rows)
    end = min(begin + per, n_rows)
    return begin, end, per


def owner_of_hypothesis(q, n_hyp, world):
    """Rank that solves hypothesis q's assignment: owners are spread evenly over the ranks (4 hypotheses on 8 GPUs
    -> ranks 0, 2, 4, 6), round-robin when there are more hypotheses than ranks."""
    if world >= n_hyp:
        return q * (world // n_hyp)
    return q % world


def hypotheses_for_rank(n_hyp, rank, world):
    return [q for q in range(n_hyp) if owner_of_hypothesis(q, n_hyp, world) == rank]


def all_pairs(n_specimens):
    """Unordered specimen pairs (i < j) in lexicographic order: 66 pairs for 12 specimens."""
    return list(itertools.combinations(range(n_specimens), 2))


def pairs_for_rank(n_specimens, rank, world):
    """Static round-robin of the pair list (pair p -> rank p % world): the schedule `register_all_pairs` falls back
    to without a work counter (`dynamic=False`)."""
    return [p for k, p in enumerate(all_pairs(n_specimens)) if k % world == rank]


class WorkCounter:
    """Shared fetch-add counter for dynamic scheduling across ranks: `next()` returns 0, 1, 2, ... exactly once over
    all callers (threads and ranks).  Backed by the process group's rendezvous store (an atomic `add` on the TCP
    store: ~0.1 ms per item, against ~19 ms of GPU work per registration)."""
    _serial = 0

    def __init__(self, group=None):
        self._local = itertools.count()
        self._lock = threading.Lock()
        self._store = None
        rank, world = world_info(group)
        if world > 1:
            from torch.distributed.distributed_c10d import _get_default_store
            self._store = _get_default_store()
            # the same key on every rank, a fresh one per counter: counters are created collectively, in the same order
            WorkCounter._serial += 1
            self._key = "platymatch_b200/work/%d" % WorkCounter._serial

    def next(self):
        if self._store is None:
            with self._lock:
                return next(self._local)
        return int(self._store.add(self._key, 1)) - 1


# ----------------------------------------------------------------------------- exchange steps
def _raise_together(error, group=None):
    """All ranks learn whether ANY rank failed before the next collective, and raise together: a rank that raised
    alone would leave the others blocked in that collective for ever."""
    import torch
    import torch.distributed as dist
    rank, world = world_info(group)
    if world > 1:
        dev = "cuda" if dist.get_backend(group) == "nccl" else "cpu"
        flag = torch.tensor([1 if error is not None else 0], dtype=torch.int32, device=dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MAX, group=group)
        failed = int(flag.item()) != 0
    else:
        failed = error is not None
    if error is not None:
        raise error
    if failed:
        raise RuntimeError("platymatch_b200: another rank failed in this collective step (see its traceback)")


def gather_rows_to_owner(local_rows, n_rows, per, owner, group=None):
    """Row shards -> the owner only.  local_rows is this rank's [per, ld] block (rows beyond the rank's range are
    padding); returns the full [n_rows, ld] matrix on `owner`, None elsewhere.  (1 / world of the bytes and of the
    memory of an all-gather: only the rank that solves the matrix needs it.)"""
    import torch
    import torch.distributed as dist
    rank, world = world_info(group)
    if world == 1:
        return local_rows[:n_rows]
    assert local_rows.shape[0] == per
    local_rows = local_rows.contiguous()
    if rank == owner:
        parts = [torch.empty_like(local_rows) for _ in range(world)]
        dist.gather(local_rows, parts, dst=dist.get_global_rank(group, owner) if group is not None else owner, group=group)
        return torch.cat(parts, 0)[:n_rows]
    dist.gather(local_rows, None, dst=dist.get_global_rank(group, owner) if group is not None else owner, group=group)
    return None


def allgather_rows(local_rows, n_rows, per, group=None):
    """All-gather of row shards (used for the descriptor histograms, which every rank needs): local_rows is this
    rank's [per, ...] block; returns the full [n_rows, ...] array on every rank."""
    import torch
    import torch.distributed as dist
    rank, world = world_info(group)
    if world == 1:
        return local_rows[:n_rows]
    assert local_rows.shape[0] == per
    full = torch.empty((world * per,) + tuple(local_rows.shape[1:]), dtype=local_rows.dtype, device=local_rows.device)
    dist.all_gather_into_tensor(full, local_rows.contiguous(), group=group)
    return full[:n_rows]


def reduce_best_hypothesis(inliers_local, transforms_local, hyp_ids_local, n_hyp, group=None):
    """Best-hypothesis reduction.  Each rank contributes (inliers, 4x4) of the hypotheses it owns; returns
    (inliers[n_hyp], transforms[n_hyp,16], best) on every rank, best = first maximum in hypothesis order
    (np.argmax semantics of reference _dock_widget.py:683-703)."""
    import torch
    import torch.distributed as dist
    rank, world = world_info(group)
    dev = transforms_local.device
    slots = max(1, -(-n_hyp // world))
    pack = torch.full((slots, 18), -1.0, dtype=torch.float64, device=dev)
    for k, q in enumerate(hyp_ids_local):
        pack[k, 0] = float(q)
        pack[k, 1] = inliers_local[k].to(torch.float64)
        pack[k, 2:] = transforms_local[k].reshape(16)
    if world > 1:
        gathered = torch.empty((world * slots, 18), dtype=torch.float64, device=dev)
        dist.all_gather_into_tensor(gathered, pack, group=group)
    else:
        gathered = pack
    inliers = torch.zeros(n_hyp, dtype=torch.int64, device=dev)
    transforms = torch.ones((n_hyp, 16), dtype=torch.float64, device=dev)
    g = gathered.cpu()
    for row in g:
        q = int(row[0].item())
        if q >= 0:
            inliers[q] = int(row[1].item())
            transforms[q] = row[2:].to(dev)
    best = int(torch.argmax(inliers).item())
    return inliers, transforms, best


def gather_results(local, n_total, owner_of, group=None):
    """Gather per-item float64 rows (e.g. 16-element transforms) computed by their owner ranks."""
    import torch
    import torch.distributed as dist
    rank, world = world_info(group)
    width = 16
    out = torch.zeros((n_total, width), dtype=torch.float64)
    for k, row in local.items():
        out[k] = torch.as_tensor(row, dtype=torch.float64).reshape(width)
    if world > 1:
        dev = "cuda" if dist.get_backend(group) == "nccl" else "cpu"
        t = out.to(dev)
        dist.all_reduce(t, op=dist.ReduceOp.SUM, group=group)    # rows are disjoint by owner
        out = t.cpu()
    return out


# ----------------------------------------------------------------------------- CUDA paths
def describe_cloud_sharded(cloud, n_variants, group=None, transposed=False):
    """pipeline.describe_cloud with the query rows of the shape-context kernel (the O(N^2) part) split over the
    ranks and the integer histograms all-gathered.  Centroid / PCA axis / mean distance are replicated (cheap and
    deterministic, so every rank bins against bit-identical frames).  Returns the same Descriptors on every rank."""
    import torch
    from . import device as D, pipeline as P
    rank, world = world_info(group)
    if world == 1:
        return P.describe_cloud(cloud, n_variants, transposed)
    pts = cloud if (torch.is_tensor(cloud) and cloud.is_cuda and transposed) else D.to_device_points(cloud, transposed=transposed)
    n = pts.shape[0]
    stats = D.cloud_stats(pts)
    md = D.mean_distance(pts)
    begin, end, per = shard_rows(n, rank, world, align=8)
    local = torch.zeros((per, n_variants, D.NBINS + 1), dtype=torch.int32, device=pts.device)   # [..., 360] = dropped
    ties = torch.zeros(1, dtype=torch.int64, device=pts.device)
    if end > begin:
        counts, dropped, ties = D.shape_context_counts(pts, stats[0:3], stats[3:6], md, n_variants, rows=(begin, end))
        local[:end - begin, :, :D.NBINS] = counts.permute(1, 0, 2)
        local[:end - begin, :, D.NBINS] = dropped.permute(1, 0)
    full = allgather_rows(local, n, per, group)                      # [n, V, 361]
    counts = full[:, :, :D.NBINS].permute(1, 0, 2).contiguous()
    dropped = full[:, :, D.NBINS].permute(1, 0).contiguous()
    import torch.distributed as dist
    dist.all_reduce(ties, group=group)
    return P.Descriptors(pts, stats, md, counts, dropped, ties)


_WINDOWS = {}
_PEER_BROKEN = set()


def _cost_window(nbytes, group=None):
    """This rank's peer-mapped cost-matrix window (grown on demand, reused across registrations), or None when CUDA IPC
    is not available between the ranks (then every later call goes through dist.gather).  Collective: all ranks
    decide together."""
    import torch
    import torch.distributed as dist
    from . import device as D
    key = id(group)
    if key in _PEER_BROKEN:
        return None
    win = _WINDOWS.get(key)
    if win is not None and win.nbytes >= nbytes:
        return win
    if win is not None:
        win.close()
        del _WINDOWS[key]
    err = None
    try:
        win = D.PeerWindow(nbytes, group)
    except Exception as e:          # e.g. IPC disabled in the container
        err, win = e, None
    flag = torch.tensor([0 if err is None else 1], dtype=torch.int32, device="cuda")
    dist.all_reduce(flag, op=dist.ReduceOp.MAX, group=group)
    if int(flag.item()):
        if win is not None:
            win.close()
        _PEER_BROKEN.add(key)
        import warnings
        warnings.warn("platymatch_b200: peer-mapped windows unavailable (%s); cost rows go through dist.gather" % (err,))
        return None
    _WINDOWS[key] = win
    return win


def close_windows():
    for win in _WINDOWS.values():
        win.close()
    _WINDOWS.clear()


def register_pair_sharded(moving, fixed, *, ransac_samples=4, ransac_trials=8000, ransac_error=16, icp_iterations=50,
                          seed=0, hypotheses=None, max_bid_rounds=2048, transform='Affine', peer_stores=None,
                          group=None, timings=None):
    """One registration spread over all ranks (config 4, 20k x 20k).

    descriptor rows   split over the ranks, histograms all-gathered (describe_cloud_sharded);
    cost rows         rank r computes rows [r * per, (r + 1) * per) of EVERY hypothesis' matrix and delivers them to
                      that matrix' owner only — through the owner's peer-mapped window (the kernel's own stores, NCCL)
                      or one gather per matrix;
    LAP + RANSAC      on the owner of each hypothesis; (inliers, A) all-gathered; first maximum wins;
    ICP               replicated on every rank (deterministic).
    Returns the same dict of numpy results on every rank.  timings: optional dict that receives the host-clock
    duration of the stages of THIS rank (synchronising; for benchmarks only)."""
    import torch
    import torch.distributed as dist
    from . import device as D, pipeline as P
    rank, world = world_info(group)
    hyps = P.HYPOTHESES_DISTINCT if hypotheses is None else list(hypotheses)
    H = len(hyps)
    need_m, need_f = max(a for a, _ in hyps), max(b for _, b in hyps)
    nccl = world > 1 and dist.get_backend(group) == "nccl"
    if peer_stores is None:
        peer_stores = nccl

    def mark(name, t0):
        if timings is not None:
            torch.cuda.synchronize()
            timings[name] = timings.get(name, 0.0) + (time.perf_counter() - t0) * 1e3
        return time.perf_counter()

    t0 = time.perf_counter()
    dm = describe_cloud_sharded(moving, 1 if need_m == 1 else 2, group)
    df = describe_cloud_sharded(fixed, 1 if need_f == 1 else (2 if need_f == 2 else 4), group)
    n1, n2 = dm.n, df.n
    if n1 > n2:
        raise ValueError("sharded path expects n_moving <= n_fixed (swap the clouds otherwise)")
    for a, _ in hyps:
        dm.operand(a)
    for _, b in hyps:
        df.operand(b)
    t0 = mark("describe", t0)
    ldc = (n2 + 3) // 4 * 4
    mine = hypotheses_for_rank(H, rank, world)
    begin, end, per = shard_rows(n1, rank, world)
    dev = dm.pts.device
    costs = {}
    exchanged = 0
    if world == 1:
        for q, (a, b) in enumerate(hyps):
            costs[q] = D.chi2_cost(dm.operand(a), df.operand(b))
    win = None
    if world > 1 and peer_stores:
        slots = max(1, -(-H // world))
        win = _cost_window(slots * n1 * ldc * 4, group)             # collective (first call / growth only)
        peer_stores = win is not None
    if world == 1:
        pass
    elif peer_stores:
        for q in mine:
            costs[q] = win.tensor((n1, ldc), torch.float32, offset_bytes=mine.index(q) * n1 * ldc * 4)
        dist.barrier(group)                                          # the owners' previous matrices are no longer in use
        order = [(q + rank) % H for q in range(H)]                   # spread the inbound traffic over the owners
        for q in order:
            a, b = hyps[q]
            own = owner_of_hypothesis(q, H, world)
            slot = hypotheses_for_rank(H, own, world).index(q)
            if end > begin:
                D.chi2_cost(dm.operand(a), df.operand(b), row_begin=begin, row_end=end, out_ld=ldc,
                            out_ptr=win.remote[own] + (slot * n1 + begin) * ldc * 4)
                if own != rank:
                    exchanged += (end - begin) * ldc * 4
        # stream-ordered barrier: when it completes here, every rank's kernels (and with them their peer stores) have
        flag = torch.zeros(1, dtype=torch.int32, device=dev)
        dist.all_reduce(flag, group=group)
    else:
        for q, (a, b) in enumerate(hyps):
            local = torch.zeros((per, ldc), dtype=torch.float32, device=dev)
            if end > begin:
                D.chi2_cost(dm.operand(a), df.operand(b), out=local, row_begin=begin, row_end=end)
            own = owner_of_hypothesis(q, H, world)
            full = gather_rows_to_owner(local, n1, per, own, group)
            if own == rank:
                costs[q] = full.contiguous()
            else:
                exchanged += (end - begin) * ldc * 4
    t0 = mark("chi2_cost+exchange", t0)
    a_local = torch.empty((len(mine), 16), dtype=torch.float64, device=dev)
    inl_local = torch.empty(max(len(mine), 1), dtype=torch.int32, device=dev)
    lap_cost, error = {}, None
    try:
        for k, q in enumerate(mine):
            col4row, total, _ = D.lap_solve(costs[q], n1, n2, max_bid_rounds)
            fk = D.gather_points(df.pts, col4row[0])
            D.ransac(dm.pts, fk, int(ransac_trials), float(ransac_error), int(ransac_samples), None,
                     seed=(int(seed) << 8) + q, transform=transform, out=(a_local[k], inl_local[k:k + 1]))
            lap_cost[q] = total
    except Exception as e:          # raised on all ranks together, below
        error = e
    _raise_together(error, group)
    t0 = mark("lap+ransac", t0)
    inliers, transforms, best = reduce_best_hypothesis(inl_local, a_local, mine, H, group)
    a_sc = transforms[best].contiguous()
    moved = D.apply_affine(dm.pts, a_sc)
    a_icp, resid, _ = D.icp(moved, df.pts, int(icp_iterations), transform=transform)
    a_final = D.compose(a_icp, a_sc)
    out = dict(transform=a_final.cpu().numpy().reshape(4, 4), transform_sc=a_sc.cpu().numpy().reshape(4, 4),
               transform_icp=a_icp.cpu().numpy().reshape(4, 4), inliers=inliers.cpu().numpy(), best=best,
               lap_cost={q: float(v.item()) for q, v in lap_cost.items()}, icp_residuals=resid.cpu().numpy(),
               exchanged_bytes=exchanged, peer_stores=bool(peer_stores and world > 1))
    mark("reduce+icp", t0)
    return out


def describe_specimens(specimens, n_variants=4, group=None):
    """Descriptors of every specimen on every rank: specimen s is described by rank s % world, the integer
    histograms are all-gathered (config 5: 12 x 8000 x 360 x 4 variants = 553 MB over NVLink instead of 12 x the
    O(N^2) kernel on every rank)."""
    import torch
    import torch.distributed as dist
    from . import device as D, pipeline as P
    rank, world = world_info(group)
    if world == 1:
        return [P.describe_cloud(s, n_variants) for s in specimens]
    pts = [D.to_device_points(s) for s in specimens]
    out = []
    rounds = -(-len(specimens) // world)
    for r in range(rounds):
        batch = list(range(r * world, min((r + 1) * world, len(specimens))))
        n_max = max(pts[s].shape[0] for s in batch)
        local = torch.zeros((n_max, n_variants, D.NBINS + 1), dtype=torch.int32, device="cuda")
        small = torch.zeros(18, dtype=torch.float64, device="cuda")            # stats[16], mean distance, edge ties
        s = r * world + rank
        if s < len(specimens):
            d = P.describe_cloud(pts[s], n_variants, transposed=True)
            local[:d.n, :, :D.NBINS] = d.counts.permute(1, 0, 2)
            local[:d.n, :, D.NBINS] = d.dropped.permute(1, 0)
            small[:16], small[16], small[17] = d.stats, d.mean_dist[0], d.ties[0].to(torch.float64)
        full = torch.empty((world,) + tuple(local.shape), dtype=torch.int32, device="cuda")
        smalls = torch.empty((world, 18), dtype=torch.float64, device="cuda")
        dist.all_gather_into_tensor(full, local, group=group)
        dist.all_gather_into_tensor(smalls, small, group=group)
        for k, s in enumerate(batch):
            n = pts[s].shape[0]
            counts = full[k, :n, :, :D.NBINS].permute(1, 0, 2).contiguous()
            dropped = full[k, :n, :, D.NBINS].permute(1, 0).contiguous()
            out.append(P.Descriptors(pts[s], smalls[k, :16].clone(), smalls[k, 16:17].clone(), counts, dropped,
                                     smalls[k, 17:18].to(torch.int64)))
    return out


def register_all_pairs(specimens, *, group=None, in_flight=6, dynamic=True, stats=None, **kw):
    """Batched all-pairs registration (config 5): descriptors of each specimen are computed once (spread over the
    ranks, all-gathered), the pairs are pulled from one shared work counter by every in-flight worker of every rank
    (`dynamic=False`: static round-robin), the 4x4 results are gathered on every rank.
    On each rank `in_flight` independent registrations overlap on separate CUDA streams (one host thread each):
    the assignment stage is latency-bound on a few SMs and hides behind the cost-matrix / ICP kernels of the
    other pairs.  specimens: list of 3xN arrays.  Returns (pairs, transforms[n_pairs,4,4]).
    stats: optional dict receiving this rank's pair count and busy time."""
    import torch
    from . import pipeline as P
    rank, world = world_info(group)
    pairs = all_pairs(len(specimens))
    desc = describe_specimens(specimens, 4, group)
    for d in desc:               # operands are built lazily: do it here, before the streams fork
        for v in (1, 2, 3, 4):
            d.operand(v)
    torch.cuda.synchronize()
    counter = WorkCounter(group) if dynamic else None
    static = [k for k in range(len(pairs)) if k % world == rank]
    local, errors, done = {}, [], []
    nfl = max(1, int(in_flight))
    dev = torch.cuda.current_device()
    t_begin = time.perf_counter()

    def worker(w):
        try:
            torch.cuda.set_device(dev)
            with torch.cuda.stream(torch.cuda.Stream()):
                mine = iter(static[w::nfl])
                results, queued = [], collections.deque()
                while True:
                    # A registration is ENQUEUED in ~0.5 ms and runs for 20-100 ms: a worker that pulled as fast as it can
                    # enqueue would claim the whole counter before its first pair has finished (measured at 4 GPUs: 21 /
                    # 18 / 22 / 5 pairs per rank).  At most two registrations of a worker are unfinished at any time
                    # (one running, one queued behind it), so the counter follows the progress of the GPUs.
                    if len(queued) >= 2:
                        queued.popleft().synchronize()
                    k = counter.next() if dynamic else next(mine, len(pairs))
                    if k >= len(pairs):
                        break
                    i, j = pairs[k]     # moving = specimen i, fixed = specimen j (tall problems are transposed inside)
                    res = P.register_described(desc[i], desc[j], seed=k, overlap_hypotheses=(nfl == 1), **kw)
                    results.append((k, res["transform"]))
                    ev = torch.cuda.Event()
                    ev.record()
                    queued.append(ev)
                torch.cuda.current_stream().synchronize()
                for k, t in results:
                    local[k] = t.cpu().numpy().reshape(4, 4)
                done.append(len(results))
        except Exception as e:     # surfaced below, on all ranks together: a worker must not die silently
            errors.append(e)

    if nfl == 1:
        worker(0)
    else:
        ts = [threading.Thread(target=worker, args=(w,)) for w in range(nfl)]
        for t in ts:
            t.start()
        for t in ts:
            t.join()
    busy = time.perf_counter() - t_begin
    _raise_together(errors[0] if errors else None, group)
    if stats is not None:
        stats.update(pairs_done=int(sum(done)), busy_s=busy, rank=rank)
    out = gather_results(local, len(pairs), None, group)
    return pairs, out.numpy().reshape(-1, 4, 4)
