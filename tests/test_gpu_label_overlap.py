"""DESIGN §8 row 7 — two label volumes compared on the GPU: the overlap table (pm_label_overlap) against np.unique of the
pair keys, and instance matching (`match_labels`) against scipy's linear_sum_assignment on the same float32 matrix."""
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

pytestmark = pytest.mark.gpu


# ---- oracle ---------------------------------------------------------------------------------------------------------
def oracle_table(a, b):
    """np.unique of the keys a << 32 | b (ids <= 0 as 0), the (0, 0) entry removed."""
    ka = np.where(a > 0, a, 0).astype(np.int64)
    kb = np.where(b > 0, b, 0).astype(np.int64)
    keys, cnt = np.unique((ka << 32) | kb, return_counts=True)
    keep = keys != 0
    return keys[keep] >> 32, keys[keep] & 0xFFFFFFFF, cnt[keep].astype(np.int64)


def oracle_match(a, b, thresholds, table=None):
    """The matching contract restated with numpy and scipy on the same float32 matrix (table: oracle_table(a, b) when
    already computed)."""
    from scipy.optimize import linear_sum_assignment
    ia, ib, n = oracle_table(a, b) if table is None else table
    size_a = {k: 0 for k in ia}
    size_b = {k: 0 for k in ib}
    for x, y, c in zip(ia, ib, n):
        size_a[x] += int(c)
        size_b[y] += int(c)
    fg = (ia > 0) & (ib > 0)
    n_fg = int(n[fg].sum())
    a_fg, b_fg = int(n[ia > 0].sum()), int(n[ib > 0].sum())
    n_true, n_pred = len({int(x) for x in ia if x > 0}), len({int(y) for y in ib if y > 0})
    t, p, c = ia[fg], ib[fg], n[fg]
    iou = c / np.array([size_a[x] + size_b[y] - k for x, y, k in zip(t, p, c)], dtype=np.float64)
    res = {"dice": 2 * n_fg / (a_fg + b_fg) if a_fg + b_fg else 0.0,
           "jaccard": n_fg / (a_fg + b_fg - n_fg) if a_fg + b_fg - n_fg else 0.0,
           "n_true": n_true, "n_pred": n_pred, "per_threshold": []}
    for th in thresholds:
        adm = iou >= th
        if not adm.any():
            res["per_threshold"].append({"tp": 0, "cost": 0.0, "pairs": set(), "unique_costs": True})
            continue
        ut, up = np.unique(t[adm]), np.unique(p[adm])
        K = min(ut.size, up.size)
        C = np.zeros((ut.size, up.size), dtype=np.float32)
        vals = (-(1.0 + iou[adm] / (2.0 * K))).astype(np.float32)
        C[np.searchsorted(ut, t[adm]), np.searchsorted(up, p[adm])] = vals
        r, q = linear_sum_assignment(C.astype(np.float64))
        ok = C[r, q] != 0
        pairs = {(int(ut[i]), int(up[j])) for i, j in zip(r[ok], q[ok])}
        res["per_threshold"].append({"tp": int(ok.sum()), "cost": float(C[r, q].astype(np.float64).sum()),
                                     "pairs": pairs, "unique_costs": np.unique(vals).size == vals.size})
    return res


def assert_match_equals_oracle(got, want, exact_pairs=True):
    assert got["n_true"] == want["n_true"] and got["n_pred"] == want["n_pred"]
    assert got["dice"] == want["dice"] and got["jaccard"] == want["jaccard"]
    for g, w in zip(got["per_threshold"], want["per_threshold"]):
        assert g["tp"] == w["tp"], (g["threshold"], g["tp"], w["tp"])
        assert g["fp"] == got["n_pred"] - w["tp"] and g["fn"] == got["n_true"] - w["tp"]
        assert abs(g["cost"] - w["cost"]) <= 1e-9 * max(1.0, abs(w["cost"])), (g["cost"], w["cost"])
        pairs = set(zip(g["matched"][0].tolist(), g["matched"][1].tolist()))
        if exact_pairs and w["unique_costs"]:
            assert pairs == w["pairs"], g["threshold"]


def _table(a, b):
    from platymatch_b200.evaluate_metrics import label_contingency
    return label_contingency(a, b)


def assert_table(a, b):
    got, want = _table(a, b), oracle_table(a, b)
    for g, w in zip(got, want):
        assert g.dtype == np.int64 and np.array_equal(g, w)
    return got


# ---- fixtures -------------------------------------------------------------------------------------------------------
def _pair(shape=(40, 56, 72), n=60, sparse=False, seed=0):
    from platymatch_b200.synthetic import make_label_volume
    a = make_label_volume(shape, n, radius=(3.0, 6.0), seed=seed, sparse_ids=sparse)
    b = make_label_volume(shape, n, radius=(3.0, 6.0), seed=seed + 100, sparse_ids=sparse)
    return a, b


def _perturbed(a, seed):
    """a with its ids permuted, shifted by a voxel along y and x, and every tenth nucleus removed."""
    rng = np.random.default_rng(seed)
    ids = np.unique(a[a > 0])
    perm = np.zeros(int(a.max()) + 1, dtype=np.int64)
    perm[ids] = rng.permutation(ids) + 1000
    perm[ids[::10]] = 0
    return np.roll(perm[a], (1, -1), axis=(1, 2)).astype(np.int32)


DTYPES = [(np.int32, np.int32), (np.int32, np.uint16), (np.uint16, np.int32), (np.uint16, np.uint16)]


# ---- the table ------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("sparse", [False, True])
@pytest.mark.parametrize("dtypes", DTYPES, ids=lambda d: "%s-%s" % (np.dtype(d[0]).name, np.dtype(d[1]).name))
def test_table_matches_unique(dtypes, sparse):
    a, b = _pair(sparse=sparse)
    assert_table(a.astype(dtypes[0]), b.astype(dtypes[1]))


@pytest.mark.parametrize("shape", [(1, 1, 1), (1, 1, 7), (3, 5, 7), (13, 17, 19), (7, 1, 1001), (33, 31, 29)])
@pytest.mark.parametrize("dtypes", DTYPES[:2], ids=["i32-i32", "i32-u16"])
def test_table_tails(shape, dtypes):
    """Voxel counts that are not multiples of 4 or 8: the tail voxels after the last full chunk are counted."""
    rng = np.random.default_rng(int(np.prod(shape)))
    a = (rng.integers(0, 4, size=shape) * (rng.random(shape) < 0.6)).astype(dtypes[0])
    b = (rng.integers(0, 5, size=shape) * (rng.random(shape) < 0.6)).astype(dtypes[1])
    a.reshape(-1)[-1], b.reshape(-1)[-1] = 3, 4                     # (the very last voxel is a pair of its own)
    assert_table(a, b)


@pytest.mark.parametrize("dtypes", DTYPES, ids=lambda d: "%s-%s" % (np.dtype(d[0]).name, np.dtype(d[1]).name))
def test_table_pipelined_steady_state(dtypes):
    """160 x 192 x 192 = 5.9e6 voxels: more chunks than one wave of resident CTAs covers in one grid-stride step (148 SMs
    x 3 CTAs x 256 threads x 1 or 2 chunks of 8 voxels = 0.9e6 / 1.8e6 voxels), so every dtype pair runs the software
    pipeline through both register buffers and several queue flushes per warp."""
    from platymatch_b200.synthetic import make_label_volume
    shape = (160, 192, 192)
    a = make_label_volume(shape, 500, radius=(3.0, 7.0), seed=21, sparse_ids=dtypes[0] == np.int32)
    b = make_label_volume(shape, 500, radius=(3.0, 7.0), seed=22)
    assert a.size > 2 * 148 * 3 * 256 * 2 * 8
    assert_table(a.astype(dtypes[0]), b.astype(dtypes[1]))


def test_table_background_cases():
    a, _ = _pair()
    z = np.zeros_like(a)
    ia, ib, n = assert_table(a, z)
    assert np.all(ib == 0) and n.sum() == np.count_nonzero(a)
    ia, ib, n = assert_table(z, a.astype(np.uint16))
    assert np.all(ia == 0)
    for x in assert_table(z, z):
        assert x.size == 0


def test_table_self_diagonal_and_shift():
    a, _ = _pair(sparse=True, seed=4)
    ia, ib, n = assert_table(a, a)
    assert np.array_equal(ia, ib)                                    # the diagonal
    ids, cnt = np.unique(a[a > 0], return_counts=True)
    assert np.array_equal(ia, ids) and np.array_equal(n, cnt)
    b = np.zeros_like(a)
    b.reshape(-1)[1:] = a.reshape(-1)[:-1]                           # shifted by one voxel (linear order)
    ia, ib, n = assert_table(a, b)
    assert np.count_nonzero(ia != ib) > 0


def test_table_negative_and_large_ids():
    rng = np.random.default_rng(12)
    shape = (9, 23, 41)
    top = 2 ** 31 - 1
    a = rng.choice(np.array([-(2 ** 31), -5, -1, 0, 1, top, top - 1, top - 7], dtype=np.int32), size=shape)
    b = rng.choice(np.array([0, -3, 2, top, top - 2], dtype=np.int32), size=shape)
    ia, ib, _ = assert_table(a, b)
    assert ia.max() == top and ib.max() == top and ia.min() == 0
    assert_table(a, rng.integers(0, 65536, size=shape).astype(np.uint16))


def test_table_overflow_reruns(monkeypatch):
    """A noise pair with ~40k distinct pairs against a first capacity of 2048 slots: reruns until nothing is dropped."""
    from platymatch_b200 import device as D
    rng = np.random.default_rng(3)
    shape = (40, 50, 61)
    a = rng.integers(0, 200, size=shape).astype(np.int32)
    b = rng.integers(0, 200, size=shape).astype(np.uint16)
    calls = []
    real = D.label_overlap

    def counted(x, y, capacity):
        calls.append(capacity)
        return real(x, y, capacity)
    monkeypatch.setattr(D, "label_overlap", counted)
    ia, _, _ = assert_table(a, b)
    assert ia.size > 30000 and len(calls) >= 3 and calls[0] == 2048, calls
    # the device call reports the overflow itself: pairs written <= capacity, dropped voxels > 0
    keys, counts, n_out = real(D.to_device_volume(a), D.to_device_volume(b), 1024)
    n_pairs, dropped = n_out.cpu().tolist()
    assert n_pairs <= 1024 and dropped > 0
    assert int(counts[:n_pairs].sum()) + dropped == np.count_nonzero((a > 0) | (b > 0))


def test_table_beyond_2_31_voxels():
    """4120 x 1024 x 1024 = 4.3e9 voxels, int32 z-slab ids against uint16 y-slab ids, built on the device: the table is
    the product of the slab sizes, and the pair (1, 1) covers 4.30e9 > 2^32 voxels."""
    from platymatch_b200 import device as D
    torch = D._torch()
    nz, ny, nx = 4120, 1024, 1024
    a = torch.ones((nz, ny, nx), dtype=torch.int32, device="cuda")
    a[0] = 0
    a[-8:] = 2
    b16 = torch.ones((nz, ny, nx), dtype=torch.int16, device="cuda")
    b16[:, 0] = 0
    b16[:, -1] = 3
    keys, counts, n_out = D.label_overlap(a, b16.view(torch.uint16), 1024)
    n_pairs, dropped = n_out.cpu().tolist()
    del a, b16
    torch.cuda.empty_cache()
    assert dropped == 0
    got = dict(zip(keys[:n_pairs].cpu().tolist(), counts[:n_pairs].cpu().tolist()))
    cz, cy = {0: 1, 1: nz - 9, 2: 8}, {0: 1, 1: ny - 2, 3: 1}
    want = {(za << 32) | yb: cz[za] * cy[yb] * nx for za in cz for yb in cy if (za, yb) != (0, 0)}
    assert got == want
    assert want[(1 << 32) | 1] > 2 ** 32


def test_table_on_side_stream():
    """A table pass enqueued on a side stream right after the upload, with no host synchronisation, gives the same table
    as on the default stream."""
    from platymatch_b200 import device as D
    torch = D._torch()
    a, b = _pair(seed=7)
    torch.cuda.synchronize()
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        ta, tb = torch.from_numpy(a).cuda(), torch.from_numpy(b).cuda()
        keys, counts, n_out = D.label_overlap(ta, tb, 4096)
        n = n_out[0]
        s, order = torch.sort(torch.where(torch.arange(keys.numel(), device="cuda") < n, keys, torch.iinfo(torch.int64).max))
        side_res = torch.stack([s, counts[order]])
    side.synchronize()
    n_side = int(n.item())
    k2, c2, n2 = D.label_overlap(ta, tb, 4096)
    m = int(n2[0].item())
    s2, o2 = torch.sort(k2[:m])
    assert n_side == m and int(n_out[1]) == 0
    assert torch.equal(side_res[0, :m], s2) and torch.equal(side_res[1, :m], c2[:m][o2])


# ---- matching -------------------------------------------------------------------------------------------------------
THRESHOLDS = (0.1, 0.3, 0.5, 0.9, 1.0)


@pytest.mark.parametrize("case", ["shifted_relabelled", "independent_radii", "self_permuted"])
def test_match_labels_against_oracle(case):
    from platymatch_b200.evaluate_metrics import match_labels
    from platymatch_b200.synthetic import make_label_volume
    shape = (40, 56, 72)
    a = make_label_volume(shape, 70, radius=(3.0, 6.0), seed=5)
    if case == "shifted_relabelled":
        b = _perturbed(a, 1)
    elif case == "independent_radii":                # a's centres (replaying its rng stream), other radii and order
        rng = np.random.default_rng(5)
        centres = []
        for _ in range(70):
            centres.append(rng.random(3) * np.array(shape))
            rng.uniform(3.0, 6.0)
        b = make_label_volume(shape, radius=(2.5, 6.5), seed=9, centers=np.array(centres)[::-1]).astype(np.uint16)
    else:
        perm = np.zeros(int(a.max()) + 1, dtype=np.int64)
        perm[1:] = np.random.default_rng(2).permutation(int(a.max())) + 1
        b = perm[a].astype(np.int32)
    got = match_labels(a, b, THRESHOLDS)
    want = oracle_match(a, b, THRESHOLDS)
    assert_match_equals_oracle(got, want)
    tps = [r["tp"] for r in got["per_threshold"]]
    assert tps == sorted(tps, reverse=True)
    if case == "self_permuted":
        assert all(r["tp"] == got["n_true"] for r in got["per_threshold"])    # IoU 1 everywhere
        assert got["dice"] == 1.0 and got["jaccard"] == 1.0
    else:
        assert tps[0] > tps[-1]                                             # thresholds matter here


def test_match_labels_split_nucleus_tie():
    """A nucleus split exactly into two halves: IoU 0.5 with each half, a tie.  Whichever half is chosen, tp / fp / fn
    are right."""
    from platymatch_b200.evaluate_metrics import match_labels
    a = np.zeros((8, 12, 16), np.int32)
    b = np.zeros_like(a)
    a[1:5, 2:6, 2:10] = 1
    b[1:5, 2:6, 2:6], b[1:5, 2:6, 6:10] = 5, 6
    a[5:8, 8:12, 10:16] = 2                                           # a second nucleus found exactly
    b[5:8, 8:12, 10:16] = 9
    got = match_labels(a, b, (0.3, 0.5, 0.51))
    r3, r5, r51 = got["per_threshold"]
    for r in (r3, r5):
        assert (r["tp"], r["fp"], r["fn"]) == (2, 1, 0)
        pairs = set(zip(r["matched"][0].tolist(), r["matched"][1].tolist()))
        assert (2, 9) in pairs and len(pairs & {(1, 5), (1, 6)}) == 1
        assert sorted(r["matched"][2].tolist()) == [0.5, 1.0]
    assert (r51["tp"], r51["fp"], r51["fn"]) == (1, 2, 1)
    want = oracle_match(a, b, (0.3, 0.5, 0.51))
    assert_match_equals_oracle(got, want, exact_pairs=False)


def test_match_labels_stats_fields():
    """The returned ratios restated from their formulas, including zero denominators."""
    from platymatch_b200.evaluate_metrics import match_labels
    a, b = _pair(seed=11)
    got = match_labels(a, _perturbed(a, 3), THRESHOLDS)
    for r in got["per_threshold"]:
        tp, fp, fn = r["tp"], r["fp"], r["fn"]
        assert r["precision"] == tp / (tp + fp) and r["recall"] == tp / (tp + fn)
        assert r["accuracy"] == tp / (tp + fp + fn) and r["f1"] == 2 * tp / (2 * tp + fp + fn)
        mv = r["matched"][2]
        assert mv.size == tp and np.all(mv >= r["threshold"])
        assert r["mean_matched_iou"] == (mv.sum() / tp if tp else 0.0)
        assert np.all(np.diff(r["matched"][0]) > 0)
    z = np.zeros_like(a)
    empty = match_labels(z, z, (0.5,))
    assert empty["dice"] == 0.0 and empty["jaccard"] == 0.0 and empty["n_true"] == 0 and empty["n_pred"] == 0
    r = empty["per_threshold"][0]
    assert (r["tp"], r["fp"], r["fn"], r["precision"], r["recall"], r["f1"], r["mean_matched_iou"]) == (0, 0, 0, 0, 0, 0, 0)
    one_sided = match_labels(a, z, (0.5,))["per_threshold"][0]
    assert one_sided["fn"] == len(np.unique(a[a > 0])) and one_sided["recall"] == 0.0 and one_sided["precision"] == 0.0


# ---- end to end: register, warp, compare ----------------------------------------------------------------------------
def _registration_setup():
    """The two rendered label volumes of tests/test_labels.py::test_registration_from_label_volumes."""
    from platymatch_b200.synthetic import make_label_volume
    rng = np.random.default_rng(8)
    n, shape = 400, (160, 160, 160)
    centre = np.array(shape) / 2.0
    d = rng.normal(size=(n, 3))
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    fixed_c = centre + d * np.array([55.0, 48.0, 42.0]) + rng.normal(0, 1.5, size=(n, 3))
    ang = np.deg2rad(12.0)
    R = np.array([[1, 0, 0], [0, np.cos(ang), -np.sin(ang)], [0, np.sin(ang), np.cos(ang)]])
    shift = np.array([3.0, -5.0, 4.0])
    moving_c = (fixed_c - centre - shift) @ R + centre            # fixed = R (moving - centre) + centre + shift
    fixed_vol = make_label_volume(shape, radius=(2.0, 3.0), seed=1, centers=fixed_c)
    moving_vol = make_label_volume(shape, radius=(2.0, 3.0), seed=2, centers=moving_c, dtype=np.uint16)
    return n, shape, fixed_vol, moving_vol


def _foreground_dice(warped, fixed_vol):
    a, b = warped > 0, fixed_vol > 0
    return 2.0 * np.count_nonzero(a & b) / (np.count_nonzero(a) + np.count_nonzero(b))


def test_registration_then_warp_then_match():
    import platymatch_b200 as pm
    from platymatch_b200.evaluate_metrics import match_labels
    from platymatch_b200.utils.images import transform_image
    from platymatch_b200.utils.labels import detections_from_labels, ransac_error_from_sizes
    n, shape, fixed_vol, moving_vol = _registration_setup()
    fd, fs, _ = detections_from_labels(fixed_vol, 1.0)
    md, ms, _ = detections_from_labels(moving_vol, 1.0)
    res = pm.estimate_transform_unsupervised(md, fd, ransac_trials=4000, ransac_error=ransac_error_from_sizes(ms, fs),
                                             seed=2)
    warped = transform_image(moving_vol, res["transform"], shape, order=0)
    ths = (0.1, 0.5)
    got = match_labels(fixed_vol, warped, ths)
    got0 = match_labels(fixed_vol, moving_vol, ths)
    assert got["dice"] == _foreground_dice(warped, fixed_vol)
    assert got0["dice"] == _foreground_dice(moving_vol, fixed_vol)
    assert_match_equals_oracle(got, oracle_match(fixed_vol, warped, ths))
    assert_match_equals_oracle(got0, oracle_match(fixed_vol, moving_vol, ths))
    for w, u in zip(got["per_threshold"], got0["per_threshold"]):
        print("IoU >= %.1f: warped tp %d (f1 %.3f, mean IoU %.3f), unwarped tp %d; Dice %.4f / %.4f"
              % (w["threshold"], w["tp"], w["f1"], w["mean_matched_iou"], u["tp"], got["dice"], got0["dice"]))
        assert w["tp"] > u["tp"]
