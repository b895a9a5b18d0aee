"""Device-resident building blocks: thin Python over the C ABI, torch tensors as device buffers.

Every function here takes / returns CUDA tensors and enqueues on the current torch stream; nothing
synchronises unless stated.  The reference-named numpy API (utils/, estimate_transform/) and the
fused pipeline (pipeline.py) are built from these.
"""
import numpy as np

from . import _lib
from ._lib import NBINS, LAP_STATS, CHI2_TILE, TRANSFORMS, check, ptr, stream_ptr, load

R_EDGES = np.logspace(np.log10(1 / 8), np.log10(2), 5)  # shape_context.py:24 — numpy's exact doubles


def transform_code(transform):
    """The widget's transform string ('Affine' / 'Similar', _dock_widget.py:627) -> PM_TRANSFORM_*."""
    try:
        return TRANSFORMS[transform]
    except KeyError:
        raise ValueError("transform must be 'Affine' or 'Similar', got %r" % (transform,))


def _torch():
    return _lib.require_cuda()


def to_device_points(cloud, transposed=False, device=None):
    """numpy 3xN / 4xN (reference layout) or Nx3/4 (transposed=True) -> CUDA [N,3] float64."""
    torch = _torch()
    if torch.is_tensor(cloud):
        t = cloud.to(dtype=torch.float64)
        t = t if transposed else t.t()
        return t[:, :3].contiguous().to(device or "cuda")
    a = np.asarray(cloud, dtype=np.float64)
    a = a if transposed else a.T
    # the layout change (3xN -> [N,3]) lands directly in PINNED host memory, so the host -> device copy is one
    # asynchronous DMA (torch's pinned-block cache keeps the block alive until the copy has completed)
    staged = torch.empty((a.shape[0], 3), dtype=torch.float64, pin_memory=True)
    staged.numpy()[...] = a[:, :3]
    return staged.to(device or "cuda", non_blocking=True)


def cloud_stats(pts):
    """[16] float64: centroid[0:3], PCA first axis[3:6], covariance[6:12], n, eigenvalues[13:16]."""
    torch = _torch()
    stats = torch.empty(16, dtype=torch.float64, device=pts.device)
    check(load().pm_cloud_stats(ptr(pts), pts.shape[0], ptr(stats), stream_ptr()), "pm_cloud_stats")
    return stats


def mean_distance(pts):
    """[1] float64 device scalar (utils.py:58-75)."""
    torch = _torch()
    n = pts.shape[0]
    nbytes = load().pm_mean_distance_workspace_bytes(n)
    ws = torch.empty(max(nbytes // 8, 1), dtype=torch.float64, device=pts.device)
    out = torch.empty(1, dtype=torch.float64, device=pts.device)
    check(load().pm_mean_distance(ptr(pts), n, ptr(out), ptr(ws), nbytes, stream_ptr()), "pm_mean_distance")
    return out


def shape_context_counts(pts, centroid, x0, mean_dist, n_variants, r_edges=None, rows=None):
    """Integer histograms [n_variants, N, 360] uint32 (as int32 tensor), dropped [n_variants, N], ties [1].
    rows = (begin, end): only those query nuclei -> [n_variants, end - begin, 360] (descriptor rows shard across GPUs)."""
    torch = _torch()
    n = pts.shape[0]
    begin, end = (0, n) if rows is None else rows
    if r_edges is None:
        r_edges = torch.from_numpy(R_EDGES).to(pts.device)
    counts = torch.empty((n_variants, end - begin, NBINS), dtype=torch.int32, device=pts.device)
    dropped = torch.empty((n_variants, end - begin), dtype=torch.int32, device=pts.device)
    ties = torch.zeros(1, dtype=torch.int64, device=pts.device)
    check(load().pm_shape_context_hist_rows(ptr(pts), n, ptr(centroid), ptr(x0), ptr(mean_dist), ptr(r_edges),
                                            r_edges.numel(), n_variants, begin, end, ptr(counts), ptr(dropped),
                                            ptr(ties), stream_ptr()), "pm_shape_context_hist_rows")
    return counts, dropped, ties


def padded(n, tile=CHI2_TILE):
    return ((n + tile - 1) // tile) * tile


class Chi2Operand:
    """One side of the chi^2 cost kernel: bin-major float32 histograms [361, ld] (empty bins = 2^-60, row
    360 = null bin) and the per-128-block non-empty-bin masks [ld/128, 12] (see pm_chi2_operand)."""

    def __init__(self, t, mask, n):
        self.t, self.mask, self.n, self.ld = t, mask, n, t.shape[1]


def chi2_operand(hist_2d):
    """[N,360] integer counts (int32/uint32: normalised by the row total) or float32 histograms -> Chi2Operand."""
    torch = _torch()
    n = hist_2d.shape[0]
    ld = padded(n)
    out = torch.empty((NBINS + 1, ld), dtype=torch.float32, device=hist_2d.device)
    mask = torch.empty((ld // CHI2_TILE, 12), dtype=torch.int32, device=hist_2d.device)
    hist_2d = hist_2d.contiguous()
    if hist_2d.dtype == torch.float32:
        check(load().pm_chi2_operand_f32(ptr(hist_2d), n, ptr(out), ld, ptr(mask), stream_ptr()), "pm_chi2_operand_f32")
    else:
        assert hist_2d.dtype in (torch.int32, torch.uint32)
        check(load().pm_chi2_operand(ptr(hist_2d), n, ptr(out), ld, ptr(mask), stream_ptr()), "pm_chi2_operand")
    return Chi2Operand(out, mask, n)


def chi2_cost(a, b, out=None, row_begin=0, row_end=None, out_ptr=None, out_ld=None):
    """cost[row_begin:row_end, :b.n] float32 (ld = b.n rounded up to 4) for two Chi2Operands (rows a, columns b).
    out_ptr / out_ld: raw device address of the first output row and its leading dimension instead of a tensor -
    a peer-mapped window of another rank (PeerWindow): the kernel's stores go over NVLink."""
    torch = _torch()
    n1, n2 = a.n, b.n
    row_end = n1 if row_end is None else row_end
    ldc = (n2 + 3) // 4 * 4
    if out_ptr is not None:
        import ctypes
        check(load().pm_chi2_cost(ptr(a.t), a.ld, ptr(a.mask), n1, ptr(b.t), b.ld, ptr(b.mask), n2, row_begin, row_end,
                                  ctypes.c_void_p(int(out_ptr)), int(out_ld if out_ld is not None else ldc), stream_ptr()),
              "pm_chi2_cost")
        return None
    if out is None:
        out = torch.empty((row_end - row_begin, ldc), dtype=torch.float32, device=a.t.device)
    assert out.stride(-1) == 1 and out.shape[-1] >= n2
    check(load().pm_chi2_cost(ptr(a.t), a.ld, ptr(a.mask), n1, ptr(b.t), b.ld, ptr(b.mask), n2, row_begin, row_end,
                              ptr(out), out.stride(-2), stream_ptr()), "pm_chi2_cost")
    return out


def lap_solve(cost, nr, nc, max_bid_rounds=2048, algorithm=0, out=None):
    """cost [batch, nr, ldc] float32 (nr <= nc) -> col4row [batch, nr] int32, total [batch] f64, stats [batch, 16] i64.
    out = (col4row, total, stats) writes into caller-owned tensors (views of a larger batch are fine)."""
    torch = _torch()
    if cost.dim() == 2:
        cost = cost.unsqueeze(0)
    batch, ldc = cost.shape[0], cost.stride(1)
    assert cost.stride(2) == 1 and (batch == 1 or cost.stride(0) == nr * ldc), "cost batch must be densely stacked"
    if out is None:
        col4row = torch.empty((batch, nr), dtype=torch.int32, device=cost.device)
        total = torch.empty(batch, dtype=torch.float64, device=cost.device)
        stats = torch.empty((batch, LAP_STATS), dtype=torch.int64, device=cost.device)     # zeroed by the init kernel
    else:
        col4row, total, stats = out
        assert col4row.is_contiguous() and total.is_contiguous() and stats.is_contiguous()
    nbytes = load().pm_lap_workspace_bytes(batch, nr, nc)
    ws = torch.empty(nbytes // 8 + 1, dtype=torch.float64, device=cost.device)
    check(load().pm_lap_solve(ptr(cost), batch, nr, nc, ldc, int(max_bid_rounds), int(algorithm), ptr(col4row), ptr(total), ptr(stats),
                              ptr(ws), nbytes, stream_ptr()), "pm_lap_solve")
    return col4row, total, stats


def ransac(moving_k, fixed_k, trials, error, min_samples=4, sample_idx=None, seed=0, want_per_trial=False,
           transform='Affine', out=None):
    """moving_k / fixed_k [K,3] in correspondence order -> (A [16], inliers [1] i32, trial [1] i32, per_trial|None).
    out = (A [16] f64, inliers [1] i32) writes the first two results into caller-owned tensors."""
    torch = _torch()
    k = moving_k.shape[0]
    dev = moving_k.device
    if out is None:
        best_a = torch.empty(16, dtype=torch.float64, device=dev)
        best_inl = torch.empty(1, dtype=torch.int32, device=dev)
    else:
        best_a, best_inl = out
    best_trial = torch.empty(1, dtype=torch.int32, device=dev)
    per_trial = torch.empty(trials, dtype=torch.int32, device=dev) if want_per_trial else None
    if sample_idx is not None:
        sample_idx = sample_idx.to(device=dev, dtype=torch.int32).contiguous()
        assert tuple(sample_idx.shape) == (trials, min_samples)
    nbytes = load().pm_ransac_workspace_bytes(trials)
    ws = torch.empty(nbytes // 8 + 1, dtype=torch.float64, device=dev)
    check(load().pm_ransac(ptr(moving_k), ptr(fixed_k), k, ptr(sample_idx), trials, min_samples, float(error),
                           int(seed) & (2 ** 64 - 1), transform_code(transform), ptr(best_a), ptr(best_inl),
                           ptr(best_trial), ptr(per_trial), ptr(ws), nbytes, stream_ptr()), "pm_ransac")
    return best_a, best_inl, best_trial, per_trial


def icp(moving, fixed, iterations=50, want_nn=False, transform='Affine'):
    """-> (A_icp [16] f64, residuals [iterations] f64, nn [N1] i32 | None)."""
    torch = _torch()
    n1, n2, dev = moving.shape[0], fixed.shape[0], moving.device
    a_icp = torch.empty(16, dtype=torch.float64, device=dev)
    resid = torch.empty(max(iterations, 1), dtype=torch.float64, device=dev)
    nn = torch.empty(n1, dtype=torch.int32, device=dev) if want_nn else None
    nbytes = load().pm_icp_workspace_bytes2(n1, n2)
    ws = torch.empty(nbytes // 8 + 1, dtype=torch.float64, device=dev)
    check(load().pm_icp(ptr(moving), n1, ptr(fixed), n2, int(iterations), transform_code(transform), ptr(a_icp),
                        ptr(resid), ptr(nn), ptr(ws), nbytes, stream_ptr()), "pm_icp")
    return a_icp, resid[:iterations], nn


def fit_transform(moving_k, fixed_k, transform='Affine'):
    """get_affine_transform / get_similar_transform (find_transform.py:4-17, :21-99) on [K,3] pairs -> [16] f64."""
    torch = _torch()
    a = torch.empty(16, dtype=torch.float64, device=moving_k.device)
    if transform_code(transform) == TRANSFORMS['Similar']:
        check(load().pm_fit_similar(ptr(moving_k), ptr(fixed_k), moving_k.shape[0], ptr(a), stream_ptr()), "pm_fit_similar")
    else:
        check(load().pm_fit_affine(ptr(moving_k), ptr(fixed_k), moving_k.shape[0], ptr(a), stream_ptr()), "pm_fit_affine")
    return a


def select_best(inliers, a_all):
    """np.argmax(inliers) on the device (_dock_widget.py:683): -> (best [1] i32, A_best [16] f64)."""
    torch = _torch()
    n = inliers.numel()
    assert inliers.dtype == torch.int32 and a_all.is_contiguous() and a_all.numel() == 16 * n
    best = torch.empty(1, dtype=torch.int32, device=inliers.device)
    a = torch.empty(16, dtype=torch.float64, device=inliers.device)
    check(load().pm_select_best(ptr(inliers), ptr(a_all), n, ptr(best), ptr(a), stream_ptr()), "pm_select_best")
    return best, a


def apply_affine(pts, a16):
    torch = _torch()
    out = torch.empty_like(pts)
    check(load().pm_apply_affine(ptr(pts), pts.shape[0], ptr(a16), ptr(out), stream_ptr()), "pm_apply_affine")
    return out


def gather_points(pts, index_i32):
    torch = _torch()
    k = index_i32.numel()
    out = torch.empty((k, 3), dtype=torch.float64, device=pts.device)
    check(load().pm_gather_points(ptr(pts), ptr(index_i32), k, ptr(out), stream_ptr()), "pm_gather_points")
    return out


def compose(a16, b16):
    torch = _torch()
    c = torch.empty(16, dtype=torch.float64, device=a16.device)
    check(load().pm_compose(ptr(a16), ptr(b16), ptr(c), stream_ptr()), "pm_compose")
    return c


def label_centroids(labels, anisotropy=1.0, table_size=None, sync=True):
    """Label volume [nz, ny, nx] (CUDA int32 or uint16 tensor) -> (ids [n] i32, centroids [n,3] f64 zyx, sizes [n] f64),
    ids ascending (np.unique order, 0 / negatives = background).  One streaming pass (pm_label_centroids)."""
    torch = _torch()
    assert labels.dim() == 3 and labels.is_cuda
    labels = labels.contiguous()
    if labels.dtype == torch.int32:
        dtype = 0
    elif labels.dtype == torch.uint16:
        dtype = 1
    else:
        raise ValueError("label volume must be int32 or uint16, got %s" % labels.dtype)
    nz, ny, nx = labels.shape
    dev = labels.device
    if table_size is None:
        mx = torch.zeros(1, dtype=torch.int32, device=dev)
        check(load().pm_label_max_id(ptr(labels), dtype, labels.numel(), ptr(mx), stream_ptr()), "pm_label_max_id")
        table_size = int(mx.item()) + 1
    cap = max(table_size - 1, 1)
    ids = torch.empty(cap, dtype=torch.int32, device=dev)
    cen = torch.empty((cap, 3), dtype=torch.float64, device=dev)
    sizes = torch.empty(cap, dtype=torch.float64, device=dev)
    n_out = torch.empty(1, dtype=torch.int32, device=dev)            # (always written by the finalize kernel)
    nbytes = load().pm_label_workspace_bytes(table_size)
    ws = torch.empty(nbytes // 8 + 1, dtype=torch.int64, device=dev)
    check(load().pm_label_centroids(ptr(labels), dtype, nz, ny, nx, table_size, float(anisotropy), cap, ptr(ids), ptr(cen),
                                    ptr(sizes), ptr(n_out), ptr(ws), nbytes, stream_ptr()), "pm_label_centroids")
    if not sync:                      # everything is enqueued; the caller reads n_out later
        return ids, cen, sizes, n_out
    n = min(int(n_out.item()), cap)
    return ids[:n], cen[:n], sizes[:n]


def resample_affine(src, M, out_shape, order=0, cval=0.0, out=None):
    """Volume src [sz, sy, sx] (CUDA int32, uint16 or float32 tensor) resampled into out_shape (dz, dy, dx), same dtype.
    M: 4 x 4 float64 (CUDA tensor, or host array copied over) mapping an output voxel index (z, y, x, 1) to a source
    index; order 0 (nearest) or 1 (trilinear); voxels that map outside the source get cval.  Equal to
    scipy.ndimage.affine_transform(src, M[:3, :3], offset=M[:3, 3], output_shape, order, mode='constant', cval)
    (pm_resample_affine).  out: a caller-owned contiguous tensor of that shape and dtype."""
    torch = _torch()
    name = str(src.dtype).replace("torch.", "")
    if name not in _lib.VOLUME_DTYPES:
        raise ValueError("volume must be int32, uint16 or float32, got %s" % src.dtype)
    if not src.is_cuda or (out is not None and (not out.is_cuda or out.device != src.device)):
        raise ValueError("src and out must be CUDA tensors on the same device")
    if src.dim() != 3 or len(out_shape) != 3:
        raise ValueError("expected a 3-D volume and a 3-D output shape")
    if order not in (0, 1):
        raise ValueError("order must be 0 or 1, got %r" % (order,))
    src = src.contiguous()
    m = torch.as_tensor(M, dtype=torch.float64, device=src.device).reshape(16).contiguous()
    out_shape = tuple(int(s) for s in out_shape)
    if out is None:
        out = torch.empty(out_shape, dtype=src.dtype, device=src.device)
    assert out.dtype == src.dtype and tuple(out.shape) == out_shape and out.is_contiguous()
    sz, sy, sx = src.shape
    check(load().pm_resample_affine(ptr(src), _lib.VOLUME_DTYPES[name], sz, sy, sx, ptr(m), int(order), float(cval),
                                    ptr(out), *out_shape, stream_ptr()), "pm_resample_affine")
    return out


def cdist(a, b):
    """[n1,3], [n2,3] f64 -> [n1, ld] f32 Euclidean distances (ld = n2 rounded up to 4), as the LAP kernel wants them."""
    torch = _torch()
    n1, n2 = a.shape[0], b.shape[0]
    ld = (n2 + 3) // 4 * 4
    out = torch.zeros((n1, ld), dtype=torch.float32, device=a.device)
    check(load().pm_cdist(ptr(a), n1, ptr(b), n2, ptr(out), ld, stream_ptr()), "pm_cdist")
    return out


class PeerWindow:
    """A per-rank device buffer that every rank of the box can store into (CUDA IPC over NVLink; pm_peer.cu).
    `local` is this rank's buffer as a uint8 torch tensor view; `remote[r]` is the address at which rank r's buffer
    is mapped in this process (remote[rank] = the local address).  Collective: every rank of `group` constructs it
    with the same `nbytes`."""

    def __init__(self, nbytes, group=None):
        import ctypes
        import torch.distributed as dist
        torch = _torch()
        self.nbytes, self.group = int(nbytes), group
        self.rank, self.world = dist.get_rank(group), dist.get_world_size(group)
        self.ptr, self.remote, self._opened = None, [], []
        # every step that can fail is followed by a collective in which ALL ranks learn about it and raise together
        handle = (ctypes.c_ubyte * 64)()
        err = None
        try:
            p = ctypes.c_void_p()
            check(load().pm_peer_alloc(self.nbytes, ctypes.byref(p)), "pm_peer_alloc")
            self.ptr = p.value
            check(load().pm_peer_export(ctypes.c_void_p(self.ptr), handle), "pm_peer_export")
        except Exception as e:
            err = e
        mine = torch.tensor(list(handle) + [0 if err is None else 1], dtype=torch.uint8, device="cuda")
        everyone = torch.empty((self.world, 65), dtype=torch.uint8, device="cuda")
        dist.all_gather_into_tensor(everyone, mine, group=group)
        handles = everyone.cpu().numpy()
        if handles[:, 64].any():
            self.close()
            raise _lib.PlatyMatchError("peer window: allocation / export failed on a rank (%s)" % (err,))
        for r in range(self.world):
            if r == self.rank:
                self.remote.append(self.ptr)
                continue
            q = ctypes.c_void_p()
            buf = (ctypes.c_ubyte * 64)(*handles[r, :64].tolist())
            try:
                check(load().pm_peer_open(buf, ctypes.byref(q)), "pm_peer_open")
                self._opened.append(q.value)
            except Exception as e:
                err = e
            self.remote.append(q.value)
        flag = torch.tensor([0 if err is None else 1], dtype=torch.int32, device="cuda")
        dist.all_reduce(flag, op=dist.ReduceOp.MAX, group=group)
        if int(flag.item()):
            self.close()
            raise _lib.PlatyMatchError("peer window: cudaIpcOpenMemHandle failed on a rank (%s)" % (err,))

    def tensor(self, shape, dtype, offset_bytes=0):
        """A torch view of (part of) the local buffer."""
        torch = _torch()
        n = int(np.prod(shape))
        itemsize = torch.empty(0, dtype=dtype).element_size()
        assert offset_bytes + n * itemsize <= self.nbytes
        iface = {"shape": tuple(int(x) for x in shape), "typestr": np.dtype(str(dtype).replace("torch.", "")).str,
                 "data": (self.ptr + offset_bytes, False), "version": 2}
        holder = type("_Win", (), {"__cuda_array_interface__": iface})()
        return torch.as_tensor(holder, device="cuda")

    def close(self):
        import ctypes
        torch = _torch()
        torch.cuda.synchronize()
        for q in self._opened:
            load().pm_peer_close(ctypes.c_void_p(q))
        self._opened = []
        if self.ptr:
            load().pm_peer_free(ctypes.c_void_p(self.ptr))
            self.ptr = None


def detect_pass(src, axis, weights, out=None, t0=None, t1=None, scale=1.0):
    """One separable 1-D correlation of a float32 CUDA volume along `axis` (pm_detect_pass): weights = the symmetric
    float64 half-kernel w[0..lw] (centre first, CUDA tensor), mode 'reflect', float32 result.  t0 / t1 given:
    out = scale * ((t0 + t1) + pass) in float32."""
    torch = _torch()
    assert src.dtype == torch.float32 and src.dim() == 3 and src.is_cuda and src.is_contiguous()
    assert weights.dtype == torch.float64 and weights.is_cuda and weights.is_contiguous()
    if out is None:
        out = torch.empty_like(src)
    nz, ny, nx = src.shape
    check(load().pm_detect_pass(ptr(src), nz, ny, nx, int(axis), ptr(weights), weights.numel() - 1, ptr(t0), ptr(t1),
                                float(scale), ptr(out), stream_ptr()), "pm_detect_pass")
    return out


def detect_otsu(img, factor=1.0):
    """[2] float64 device tensor: (threshold_otsu(img, 256), factor * threshold) of a float32 CUDA tensor."""
    torch = _torch()
    assert img.dtype == torch.float32 and img.is_cuda and img.is_contiguous()
    out = torch.empty(2, dtype=torch.float64, device=img.device)
    nbytes = load().pm_detect_otsu_workspace_bytes()
    ws = torch.empty(nbytes // 8 + 1, dtype=torch.int64, device=img.device)
    check(load().pm_detect_otsu(ptr(img), img.numel(), float(factor), ptr(out), ptr(ws), nbytes, stream_ptr()),
          "pm_detect_otsu")
    return out


def detect_minima(l_prev, l_cur, l_next, k, threshold, keys, values, count):
    """Append scale k's candidates (pm_detect_minima) to keys [cap] int64 / values [cap] float32; count [1] int64."""
    nz, ny, nx = l_cur.shape
    check(load().pm_detect_minima(ptr(l_prev), ptr(l_cur), ptr(l_next), nz, ny, nx, int(k), ptr(threshold),
                                  keys.numel(), ptr(keys), ptr(values), ptr(count), stream_ptr()), "pm_detect_minima")


def detect_suppress(keys, count, shape, radii, max_radius, anisotropy, overlap):
    """Greedy suppression of the priority-sorted candidates keys [cap] (the first min(count, cap)); radii: CUDA float64
    per scale.  -> state [cap] uint8 (1 kept, 2 dropped; entries past the count are undefined)."""
    torch = _torch()
    cap = keys.numel()
    nz, ny, nx = shape
    state = torch.empty(cap, dtype=torch.uint8, device=keys.device)
    nbytes = load().pm_detect_suppress_workspace_bytes(cap, nz, ny, nx, float(max_radius), float(anisotropy))
    ws = torch.empty(nbytes // 8 + 1, dtype=torch.int64, device=keys.device)
    check(load().pm_detect_suppress(ptr(keys), ptr(count), cap, nz, ny, nx, ptr(radii), float(max_radius),
                                    float(anisotropy), float(overlap), ptr(state), ptr(ws), nbytes, stream_ptr()),
          "pm_detect_suppress")
    return state
