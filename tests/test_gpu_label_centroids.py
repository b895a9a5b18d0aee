"""DESIGN §8 row 2 — the label-centroid pass (pm_label_centroids) against an exact integer reference, bit for bit: ids,
all three centroid coordinates, sizes and the number of ids.  Both accumulation kernels run on the same data: the
streaming kernel reads 16-byte-aligned volumes, the round-1 kernel reads views offset by 1-3 elements and volumes whose
planes hold 2^32 voxels or more.  Volumes past 2^32 voxels are built on the device with closed-form sums.  Sparse ids
are compacted before the pass where a table sized by the largest id would cost more, at every volume size."""
import os
import sys
from fractions import Fraction

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))

gpu = pytest.mark.gpu
DTYPES = [np.int32, np.uint16]
OFFSETS = [0, 1, 2, 3]                 # elements: 0 -> the streaming kernel, 1-3 -> the round-1 kernel
PAD = 4


# ---- reference ------------------------------------------------------------------------------------------------------
def _result(ids, count, sums, anisotropy):
    """ids and Python-int counts / (z, y, x) index sums -> (ids int64, centroids [n, 3], sizes); each centroid is the
    correctly rounded quotient, as np.mean of integer indices is."""
    cen = np.array([[float(Fraction(s[h], c)) for h in range(3)] for c, s in zip(count, sums)],
                   dtype=np.float64).reshape(-1, 3)
    sizes = np.array([anisotropy * c for c in count], dtype=np.float64)
    return np.asarray(ids, dtype=np.int64), cen, sizes


def reference(vol, anisotropy=1.0, table_size=None):
    """Ids > 0 (below table_size when given) in ascending order, their centroids (zyx) and sizes, from exact integer
    index sums."""
    v = np.asarray(vol).astype(np.int64).reshape(-1)
    keep = v > 0
    if table_size is not None:
        keep &= v < table_size
    lin = np.flatnonzero(keep)
    ids, inv = np.unique(v[lin], return_inverse=True)
    z, rem = np.divmod(lin, vol.shape[1] * vol.shape[2])
    y, x = np.divmod(rem, vol.shape[2])
    count = np.bincount(inv, minlength=ids.size)
    # float64 bincount sums of integers below 2^53 are exact
    assert lin.size == 0 or int(lin.max()) * lin.size < 2 ** 53
    sums = np.stack([np.bincount(inv, weights=c, minlength=ids.size) for c in (z, y, x)], axis=1)
    return _result(ids, [int(c) for c in count], [[int(s) for s in row] for row in sums], anisotropy)


def _series(a, b):
    """sum(range(a, b))"""
    return (a + b - 1) * (b - a) // 2


def box_sums(z0, z1, y0, y1, x0, x1):
    """(count, [sum z, sum y, sum x]) of the box [z0, z1) x [y0, y1) x [x0, x1), as Python ints."""
    nz, ny, nx = z1 - z0, y1 - y0, x1 - x0
    return nz * ny * nx, [_series(z0, z1) * ny * nx, _series(y0, y1) * nz * nx, _series(x0, x1) * nz * ny]


def closed_form(boxes, anisotropy=1.0):
    """Reference of a volume of disjoint boxes [(id, (z0, z1, y0, y1, x0, x1)), ...] on background."""
    acc = {}
    for i, b in boxes:
        c, s = box_sums(*b)
        a = acc.setdefault(i, [0, [0, 0, 0]])
        a[0] += c
        a[1] = [p + q for p, q in zip(a[1], s)]
    ids = sorted(acc)
    return _result(ids, [acc[i][0] for i in ids], [acc[i][1] for i in ids], anisotropy)


def assert_same(got, want):
    ids, cen, sizes = (np.asarray(x) for x in got)
    wids, wcen, wsizes = want
    assert np.array_equal(ids.astype(np.int64), wids), (ids[:8], wids[:8])
    assert cen.shape == wcen.shape and np.array_equal(cen, wcen)
    assert np.array_equal(sizes, wsizes)


def test_reference_matches_oracle():
    """The reference equals the oracle's per-id np.where / np.mean walk bit for bit (CPU only)."""
    import oracle as O
    from platymatch_b200.synthetic import make_label_volume
    rng = np.random.default_rng(5)
    vols = [make_label_volume((17, 19, 23), 30, radius=(1.0, 4.0), seed=3),
            make_label_volume((9, 31, 5), 12, seed=4, dtype=np.uint16, sparse_ids=True),
            rng.integers(0, 9, size=(7, 11, 13)).astype(np.int32),
            np.zeros((2, 3, 4), np.int32)]
    vols[2][-1, -1, -1] = 2 ** 31 - 1
    for vol in vols:
        det, sizes, ids = O.detections_from_labels(vol, anisotropy=1.7)
        wids, wcen, wsizes = reference(vol, 1.7)
        assert np.array_equal(ids.astype(np.int64), wids)
        assert np.array_equal(det.T.reshape(-1, 3), wcen) and np.array_equal(sizes, wsizes)
    want = closed_form([(3, (1, 3, 0, 2, 4, 7)), (5, (0, 1, 1, 4, 0, 1)), (3, (2, 3, 3, 4, 0, 2))], 0.5)
    vol = np.zeros((3, 4, 7), np.int32)
    vol[1:3, 0:2, 4:7], vol[0:1, 1:4, 0:1], vol[2:3, 3:4, 0:2] = 3, 5, 3
    for x, y in zip(want, reference(vol, 0.5)):
        assert np.array_equal(x, y)


# ---- device helpers -------------------------------------------------------------------------------------------------
def _torch():
    from platymatch_b200 import device as D
    return D._torch()


def device_view(vol, offset):
    """vol in a flat device buffer of PAD more elements, at `offset` elements: a contiguous [nz, ny, nx] view whose
    data pointer is 16-byte aligned only for offset 0."""
    from platymatch_b200 import device as D
    flat = np.zeros(vol.size + PAD, dtype=vol.dtype)
    flat[offset:offset + vol.size] = vol.reshape(-1)
    buf = D.to_device_volume(flat)
    view = buf[offset:offset + vol.size].view(vol.shape)
    assert view.is_contiguous() and (view.data_ptr() % 16 == 0) == (offset == 0)
    return view


def centroids(view, **kw):
    from platymatch_b200 import device as D
    return [x.cpu().numpy() for x in D.label_centroids(view, **kw)]


def assert_both_kernels(vol, anisotropy=1.0, table_size=None):
    want = reference(vol, anisotropy, table_size)
    for off in OFFSETS:
        assert_same(centroids(device_view(vol, off), anisotropy=anisotropy, table_size=table_size), want)
    return want


# ---- both kernels on the same data ----------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("shape", [(1, 1, 1), (1, 1, 7), (3, 5, 7), (7, 1, 1001), (33, 31, 29)])
@pytest.mark.parametrize("dtype", DTYPES, ids=["i32", "u16"])
def test_tail_shapes(shape, dtype):
    """Voxel counts that are not multiples of 4 or 8: the tail after the last full chunk, and the very last voxel."""
    rng = np.random.default_rng(int(np.prod(shape)))
    vol = (rng.integers(1, 6, size=shape) * (rng.random(shape) < 0.6)).astype(dtype)
    vol.reshape(-1)[-1] = 9
    assert_both_kernels(vol, anisotropy=1.3)


@gpu
@pytest.mark.parametrize("dtype", DTYPES, ids=["i32", "u16"])
def test_crowded_touching_nuclei(dtype):
    """500 balls of radius 2-7 in 70 x 83 x 101: nuclei touch along rows, so chunks hold several ids and runs."""
    from platymatch_b200.synthetic import make_label_volume
    vol = make_label_volume((70, 83, 101), 500, radius=(2.0, 7.0), seed=4, dtype=dtype)
    want = assert_both_kernels(vol, anisotropy=2.5)
    assert want[0].size > 300


@gpu
@pytest.mark.parametrize("dtype", DTYPES, ids=["i32", "u16"])
def test_rows_shorter_than_a_load(dtype):
    """Rows of 3 voxels: every 16-byte chunk spans several rows (and planes)."""
    from platymatch_b200.synthetic import make_label_volume
    vol = make_label_volume((40, 50, 3), 25, seed=7, dtype=dtype, sparse_ids=True)
    vol[1, 2, :] = 17
    assert_both_kernels(vol)


# ---- finalize and table edges ---------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("dtype", DTYPES, ids=["i32", "u16"])
def test_ids_at_finalize_cta_boundaries(dtype):
    """Each finalize CTA compacts 1024 ids (1..1024, 1025..2048, ...) and counts the non-empty ids before its own: ids on
    both sides of those boundaries, with the ids between them absent, and the largest id alone in its CTA."""
    rng = np.random.default_rng(11)
    ids = np.array([1023, 1024, 1025, 2047, 2048, 2049, 3072, 4097], dtype=np.int64)
    shape = (11, 13, 17)
    vol = (ids[rng.integers(0, ids.size, size=shape)] * (rng.random(shape) < 0.5)).astype(dtype)
    want = assert_both_kernels(vol)
    assert np.array_equal(want[0], ids)


@gpu
def test_uint16_largest_id():
    rng = np.random.default_rng(2)
    shape = (9, 10, 21)
    vol = (rng.choice(np.array([1, 2, 65534, 65535]), size=shape) * (rng.random(shape) < 0.3)).astype(np.uint16)
    vol[-1, -1, -3:] = 65535
    want = assert_both_kernels(vol)
    assert want[0][-1] == 65535


@gpu
@pytest.mark.parametrize("dtype", DTYPES, ids=["i32", "u16"])
def test_ids_only_in_the_tail(dtype):
    """75 voxels: 18 full int32 or 9 full uint16 chunks, then a tail of 3 that alone holds ids 40 and 41 (the largest)."""
    vol = np.zeros((5, 3, 5), dtype=dtype)
    vol[0, 1, 2:4] = 6
    flat = vol.reshape(-1)
    flat[-3], flat[-2], flat[-1] = 40, 41, 40
    want = assert_both_kernels(vol, anisotropy=0.75)
    assert want[0].tolist() == [6, 40, 41]


@gpu
def test_negative_int32_ids_are_background():
    rng = np.random.default_rng(9)
    shape = (13, 17, 19)
    vol = rng.choice(np.array([-(2 ** 31), -70000, -1, 0, 0, 1, 5, 70000], dtype=np.int32), size=shape)
    want = assert_both_kernels(vol)
    assert want[0].tolist() == [1, 5, 70000]


@gpu
@pytest.mark.parametrize("dtype", DTYPES, ids=["i32", "u16"])
def test_explicit_table_size_drops_larger_ids(dtype):
    """ids >= table_size are ignored: table_size 501 keeps 500, table_size 500 drops it."""
    rng = np.random.default_rng(6)
    shape = (12, 14, 31)
    vol = (rng.choice(np.array([3, 10, 500, 1025, 40000]), size=shape) * (rng.random(shape) < 0.4)).astype(dtype)
    for table_size, kept in ((501, [3, 10, 500]), (500, [3, 10]), (1026, [3, 10, 500, 1025])):
        want = assert_both_kernels(vol, table_size=table_size)
        assert want[0].tolist() == kept


@gpu
@pytest.mark.parametrize("dtype", DTYPES, ids=["i32", "u16"])
def test_capacity_contract(dtype):
    """The C ABI with fewer output slots than ids: n_out reports every id, the first `capacity` entries are written,
    the others keep what they held."""
    from platymatch_b200 import device as D
    from platymatch_b200._lib import check, load, ptr, stream_ptr
    torch = _torch()
    rng = np.random.default_rng(8)
    shape = (10, 12, 14)
    vol = (rng.integers(1, 8, size=shape) * (rng.random(shape) < 0.5)).astype(dtype)
    wids, wcen, wsizes = reference(vol, 1.5)
    assert wids.size == 7
    table_size = 8
    nbytes = load().pm_label_workspace_bytes(table_size)
    for off in OFFSETS:
        view = device_view(vol, off)
        for capacity in (0, 3):
            ids = torch.full((8,), -7, dtype=torch.int32, device="cuda")
            cen = torch.full((8, 3), -2.5, dtype=torch.float64, device="cuda")
            sizes = torch.full((8,), -3.5, dtype=torch.float64, device="cuda")
            n_out = torch.full((1,), -1, dtype=torch.int32, device="cuda")
            ws = torch.empty(nbytes // 8, dtype=torch.int64, device="cuda")
            check(load().pm_label_centroids(ptr(view), D._dtype_code(view), *shape, table_size, 1.5, capacity, ptr(ids),
                                            ptr(cen), ptr(sizes), ptr(n_out), ptr(ws), nbytes, stream_ptr()),
                  "pm_label_centroids")
            ids, cen, sizes = ids.cpu().numpy(), cen.cpu().numpy(), sizes.cpu().numpy()
            assert int(n_out.item()) == 7
            k = capacity
            assert np.array_equal(ids[:k], wids[:k]) and np.array_equal(cen[:k], wcen[:k])
            assert np.array_equal(sizes[:k], wsizes[:k])
            assert np.all(ids[k:] == -7) and np.all(cen[k:] == -2.5) and np.all(sizes[k:] == -3.5)


@gpu
def test_side_stream():
    """A pass enqueued on a side stream right after the upload, with no host synchronisation, gives the default-stream
    result."""
    from platymatch_b200 import device as D
    from platymatch_b200.synthetic import make_label_volume
    torch = _torch()
    vol = make_label_volume((96, 128, 160), 300, radius=(2.0, 6.0), seed=13)
    torch.cuda.synchronize()
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        t = torch.from_numpy(vol).cuda()
        ids, cen, sizes, n_out = D.label_centroids(t, 1.25, table_size=301, sync=False)
    side.synchronize()
    n = int(n_out.item())
    base = D.label_centroids(t, 1.25)
    assert n == base[0].numel()
    for x, y in zip((ids[:n], cen[:n], sizes[:n]), base):
        assert torch.equal(x, y)
    assert_same([x.cpu().numpy() for x in base], reference(vol, 1.25))


# ---- beyond 2^32 voxels ---------------------------------------------------------------------------------------------
BIG = (1026, 2047, 2047)               # 4 299 154 434 voxels; tail of 2 for both dtypes; a plane holds 4.19e6
BIG_N = BIG[0] * BIG[1] * BIG[2]


def _need(nbytes):
    torch = _torch()
    free, _ = torch.cuda.mem_get_info()
    if free < nbytes + (2 << 30):
        pytest.skip("needs %.1f GB of free device memory, %.1f GB free" % ((nbytes + (2 << 30)) / 1e9, free / 1e9))


def _write_boxes(buf, offset, shape, boxes):
    n = shape[0] * shape[1] * shape[2]
    vol = buf[offset:offset + n].view(shape)
    for i, (z0, z1, y0, y1, x0, x1) in boxes:
        vol[z0:z1, y0:y1, x0:x1] = i if buf.dtype == _torch().int32 or i < 2 ** 15 else i - 2 ** 16
    return vol


def big_results(dtype, shape, boxes, offsets, fill=0):
    """Results of the pass on a volume of `boxes` on `fill`, built on the device in a flat buffer of PAD more elements
    (uint16 as int16, viewed as uint16 for the pass), read at each of `offsets`.  The buffer is released on return, so
    a failing comparison afterwards does not keep it."""
    torch = _torch()
    n = shape[0] * shape[1] * shape[2]
    buf = torch.full((n + PAD,), fill, dtype=torch.int32 if dtype == np.int32 else torch.int16, device="cuda")
    out = []
    for off in offsets:
        if off:
            buf.fill_(fill)
        vol = _write_boxes(buf, off, shape, boxes)
        assert vol.is_contiguous() and (vol.data_ptr() % 16 == 0) == (off == 0)
        out.append(centroids(vol.view(torch.uint16) if dtype == np.uint16 else vol))
    del vol, buf
    torch.cuda.empty_cache()
    return out


def _linear(v):
    z, rem = divmod(v, BIG[1] * BIG[2])
    return z, rem // BIG[2], rem % BIG[2]


def _voxel_box(v):
    z, y, x = _linear(v)
    return z, z + 1, y, y + 1, x, x + 1


def big_boxes(top):
    """Disjoint boxes around linear index 2^32 (z = 1025, y = 1, x = 1024) and at both ends of the volume."""
    assert _linear(2 ** 32) == (1025, 1, 1024)
    return [(5, (0, 2, 0, 3, 0, 5)),                               # the first voxels
            (7, (1000, 1026, 0, 2047, 1030, 1040)),                # z slabs reaching past 2^32: both sides
            (9, (1024, 1026, 0, 3, 1000, 1010)),                   # straddles: rows below and above 2^32
            (11, _voxel_box(2 ** 32 - 1)),
            (12, _voxel_box(2 ** 32)),
            (13, (1025, 1026, 1, 2, 1025, 1029)),                  # the voxels right after 2^32
            (7, (1025, 1026, 500, 509, 1040, 2000)),
            (top, (1025, 1026, 2000, 2010, 100, 113)),             # the largest id: only past 2^32
            (14, _voxel_box(BIG_N - 1))]                           # the last voxel: in the tail


@gpu
@pytest.mark.parametrize("dtype,top", [(np.int32, 2 ** 20 + 1), (np.int32, 2 ** 31 - 1), (np.uint16, 65535)],
                         ids=["i32-direct", "i32-compacted", "u16"])
def test_beyond_2_32_voxels(dtype, top):
    """4.3e9 voxels through the aligned view (streaming kernel, 64-bit chunk positions past 2^32, the tail loop) and a
    view offset by one element (round-1 kernel), against closed-form sums; pm_label_max_id scans past 2^32 for the
    largest id.  int32 runs once with a directly sized table and once with ids compacted first (slab by slab: more
    voxels than one torch.unique call takes), whose 4-byte compacted volume is read by the streaming kernel."""
    from platymatch_b200 import device as D
    compacted = D._compact_pays(top, BIG_N)
    assert compacted == (top == 2 ** 31 - 1)
    _need((BIG_N + PAD) * np.dtype(dtype).itemsize + (BIG_N * 4 + (4 << 30) if compacted else 0))
    boxes = big_boxes(top)
    want = closed_form(boxes)
    assert want[0][-1] == top
    for got in big_results(dtype, BIG, boxes, (0, 1)):
        assert_same(got, want)


@gpu
def test_one_id_beyond_2_32_voxels():
    """Id 1 fills a uint16 volume of 4.3e9 voxels except for a few boxes: its count, and the sums of its indices, pass
    2^32 (64-bit counts, float64 sums of up to 4.4e12), and its centroid is still the correctly rounded mean."""
    _need((BIG_N + PAD) * 2)
    holes = [(0, (0, 1, 0, 3, 0, 2047)), (2, (400, 402, 7, 90, 33, 1500)), (3, _voxel_box(2 ** 32)),
             (0, (1025, 1026, 2046, 2047, 2000, 2047))]
    count, sums = box_sums(0, BIG[0], 0, BIG[1], 0, BIG[2])
    for _, b in holes:
        c, s = box_sums(*b)
        count -= c
        sums = [p - q for p, q in zip(sums, s)]
    assert count > 2 ** 32
    want = tuple(np.concatenate(x) for x in zip(_result([1], [count], [sums], 1.0), closed_form([h for h in holes if h[0]])))
    (got,) = big_results(np.uint16, BIG, holes, (0,), fill=1)
    assert_same(got, want)


@gpu
def test_plane_of_2_32_voxels():
    """uint16 at (1, 65536, 65537): ny * nx >= 2^32, so the 16-byte-aligned volume goes to the round-1 kernel."""
    shape = (1, 65536, 65537)
    _need((shape[1] * shape[2] + PAD) * 2)
    boxes = [(4, (0, 1, 0, 2, 0, 9)), (6, (0, 1, 3, 4, 65530, 65537)), (8, (0, 1, 65533, 65535, 65500, 65537)),
             (9, (0, 1, 65535, 65536, 65536, 65537))]
    (got,) = big_results(np.uint16, shape, boxes, (0,))
    assert_same(got, closed_form(boxes))


# ---- sparse ids do not size the table -------------------------------------------------------------------------------
@gpu
def test_sparse_ids_peak_memory():
    """ids {1, 2^22 + 1} in a 32^3 int32 volume: the device memory of detections_from_labels stays a small multiple of
    the volume: the upload, the 4-byte compacted volume and one slab's scratch, 13.0 bytes per voxel in all on one B200,
    where a table sized by the largest id would take 128 MiB and its outputs 151 MB more."""
    from platymatch_b200.utils.labels import detections_from_labels
    torch = _torch()
    vol = np.zeros((32, 32, 32), np.int32)
    vol[3:9, 4:7, 5:20] = 1
    vol[20:30, 1:31, 30:32] = 2 ** 22 + 1
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    det, sizes, ids = detections_from_labels(vol, 1.5)
    peak = torch.cuda.max_memory_allocated() - base
    print("peak %d bytes = %.2f bytes per voxel" % (peak, peak / vol.size))
    assert peak < 4 * vol.nbytes, "peak %d bytes for a %d-byte volume" % (peak, vol.nbytes)
    assert_same((ids, det.T, sizes), reference(vol, 1.5))


@gpu
def test_sparse_ids_up_to_2_31():
    """The id set of the overlap table's large-id test (up to 2^31 - 1, with negatives) through detections_from_labels,
    in int32, int64 and uint32 volumes: ids come back in the caller's dtype."""
    from platymatch_b200.utils.labels import detections_from_labels
    rng = np.random.default_rng(12)
    shape = (9, 23, 41)
    top = 2 ** 31 - 1
    a = rng.choice(np.array([-(2 ** 31), -5, -1, 0, 1, top, top - 1, top - 7], dtype=np.int32), size=shape)
    want = reference(a, 2.0)
    assert want[0].tolist() == [1, top - 7, top - 1, top]
    for v in (a, a.astype(np.int64), np.maximum(a, 0).astype(np.uint32)):
        det, sizes, ids = detections_from_labels(v, 2.0)
        assert ids.dtype == v.dtype
        assert_same((ids, det.T, sizes), want)


@gpu
@pytest.mark.parametrize("shape", [(15, 17, 19), (128, 128, 257)], ids=["floor", "ratio"])
def test_compaction_bound(shape, monkeypatch):
    """The smallest largest id that is compacted: 2^19 in a small volume, sqrt(LABEL_COMPACT_RATIO * voxels) in a larger
    one.  One id below it takes the direct table, it and above are compacted; on the same data the other path gives
    identical output.  Each volume is read aligned and at an offset of one element, so the direct pass runs both
    kernels; the compacted volume is a new aligned tensor, always read by the streaming kernel."""
    import math
    from platymatch_b200 import device as D
    n = shape[0] * shape[1] * shape[2]
    bound = max(D.LABEL_COMPACT_MIN_ID, math.isqrt(D.LABEL_COMPACT_RATIO * n - 1) + 1)
    assert (bound == D.LABEL_COMPACT_MIN_ID) == (shape == (15, 17, 19))
    calls = []
    real_compact, real_pays = D._compact_label_ids, D._compact_pays

    def counted(labels):
        calls.append(tuple(labels.shape))
        return real_compact(labels)
    monkeypatch.setattr(D, "_compact_label_ids", counted)
    rng = np.random.default_rng(14)
    for top, compacted in ((bound - 1, False), (bound, True), (bound + 1, True)):
        assert real_pays(top, n) == compacted
        vol = (rng.choice(np.array([2, 1025, 40000, top]), size=shape) * (rng.random(shape) < 0.5)).astype(np.int32)
        want = reference(vol, 1.5)
        assert want[0][-1] == top
        for off in (0, 1):
            view = device_view(vol, off)
            for forced in (None, not compacted):
                if forced is not None:
                    monkeypatch.setattr(D, "_compact_pays", lambda m, v: forced)
                del calls[:]
                assert_same(centroids(view, anisotropy=1.5), want)
                assert calls == ([shape] if (compacted if forced is None else forced) else [])
                monkeypatch.setattr(D, "_compact_pays", real_pays)
