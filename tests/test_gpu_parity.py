"""GPU parity tests: the CUDA path (through the C ABI) against the CPU oracle on the same inputs,
against the golden vectors dumped from the reference, and — at BASELINE.json's full sizes — through
size-independent properties.  Bars (BASELINE.json north_star): integer histograms bit-exact; cost
matrix within 1e-5 relative; equal optimal assignment cost (identical assignment where unique);
final 4x4 within 1e-4.
"""
import numpy as np
import pytest

from conftest import HYP_TAGS, UNARY_KEYS, load_golden

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def torch():
    import torch
    torch.cuda.set_device(0)
    return torch


@pytest.fixture(scope="module")
def D(torch):
    from platymatch_b200 import device
    return device


def _pair(n, seed=None):
    from platymatch_b200.synthetic import make_pair
    return make_pair(n, seed=seed)


# ------------------------------------------------------------------------------ K0 / K1
@pytest.mark.parametrize("n", [2, 3, 31, 257, 3000])
def test_centroid_axis_mean_distance(O, D, torch, n):
    rng = np.random.default_rng(n)
    pts = rng.normal(size=(n, 3)) * np.array([30.0, 20.0, 10.0]) + np.array([300.0, 200.0, 100.0])
    d = torch.from_numpy(pts).cuda()
    stats = D.cloud_stats(d).cpu().numpy()
    assert np.allclose(stats[0:3], pts.mean(0), rtol=1e-13)
    md = D.mean_distance(d).item()
    assert md == pytest.approx(O.get_mean_distance(pts, True), rel=1e-12)
    if n >= 31:
        x0 = O.pca_first_axis(pts)
        assert np.allclose(stats[3:6], x0, atol=1e-10)


def test_api_utils_match_reference_goldens(torch):
    from platymatch_b200.utils.utils import get_centroid, get_mean_distance, get_error
    g = load_golden("asset02")
    assert np.allclose(get_centroid(g["moving"], transposed=False), g["moving_centroid"], rtol=1e-13)
    assert get_centroid(g["moving"].T, transposed=True).shape == (1, 3)
    assert get_mean_distance(g["fixed"], transposed=False) == pytest.approx(float(g["fixed_mean_distance"]), rel=1e-12)
    assert get_error(g["moving"], g["moving"]) == 0.0
    # test_utils.py:5-8 of the reference: centroid of the unit cube
    cube = np.array([[0, 0, 0], [0, 0, 1], [0, 1, 0], [0, 1, 1], [1, 0, 0], [1, 0, 1], [1, 1, 0], [1, 1, 1]], dtype=float)
    assert np.allclose(get_centroid(cube, transposed=True), [[0.5, 0.5, 0.5]])


# ------------------------------------------------------------------------------ K2
def test_shape_context_bit_exact_vs_reference_goldens(torch, golden):
    """get_unary on the reference's assets: integer histograms of all 6 descriptor sets bit-exact."""
    from platymatch_b200.estimate_transform.shape_context import get_unary, get_unary_counts
    for cloud, typ, keys in (("moving", "moving", ["u11", "u12"]), ("fixed", "fixed", ["u21", "u22", "u23", "u24"])):
        counts, dropped, ties, x0 = get_unary_counts(golden[cloud + "_centroid"], float(golden[cloud + "_mean_distance"]),
                                                     golden[cloud], typ)
        for v, k in enumerate(keys):
            assert np.array_equal(counts[v], golden["counts_" + k].astype(np.uint32)), (golden["name"], k)
            assert np.array_equal(dropped[v], golden[cloud].shape[1] - 1 - golden["totals_" + k])
        sc = get_unary(golden[cloud + "_centroid"], float(golden[cloud + "_mean_distance"]), golden[cloud], typ)
        assert len(sc) == 4 and sc[0].shape == (golden[cloud].shape[1], 360)
        if typ == "moving":
            assert sc[2].size == 0 and sc[3].size == 0
        for v, k in enumerate(keys):
            assert np.array_equal(sc[v][:8], golden["sc_rows_" + k])      # float64 rows, bit for bit


@pytest.mark.parametrize("n", [2, 5, 33, 1000, 3000])
def test_shape_context_bit_exact_vs_oracle(O, torch, n):
    from platymatch_b200.estimate_transform.shape_context import get_unary_counts
    p = _pair(max(n, 4), seed=100 + n)
    pts = p["fixed"][:, :n]
    c, md = O.get_centroid(pts, False), (O.get_mean_distance(pts, False) if n > 1 else 1.0)
    counts, dropped, ties, x0 = get_unary_counts(c, md, pts, "fixed")
    for v in range(4):
        oc, od = O.shape_context_counts(pts.T, c, md, x0, v + 1)
        assert np.array_equal(counts[v], oc), (n, v, int(np.abs(counts[v].astype(int) - oc.astype(int)).sum()))
        assert np.array_equal(dropped[v], od)
    assert np.allclose(x0, O.pca_first_axis(pts.T), atol=1e-9) or n < 10


def test_shape_context_edge_cases(O, torch):
    """Coincident nuclei (NaN -> dropped), theta == pi and theta == 0 neighbours, integer coordinates."""
    from platymatch_b200.estimate_transform.shape_context import get_unary_counts
    rng = np.random.default_rng(5)
    pts = np.round(rng.normal(size=(3, 200)) * 40 + 200)          # integer grid -> many exact ties
    pts[:, 10] = pts[:, 11]                                       # coincident pair
    c = O.get_centroid(pts, False)
    pts[:, 20] = c[:, 0] + 2.0 * (pts[:, 21] - c[:, 0])           # collinear with the centroid: theta = 0 / pi
    md = O.get_mean_distance(pts, False)
    counts, dropped, ties, x0 = get_unary_counts(c, md, pts, "fixed")
    for v in range(4):
        oc, od = O.shape_context_counts(pts.T, c, md, x0, v + 1)
        assert np.array_equal(counts[v], oc)
        assert np.array_equal(dropped[v], od)
    assert dropped[0][10] >= 1 and dropped[0][11] >= 1


def test_variants_are_phi_permutations(torch):
    """SURVEY §2.1: sc2/sc3/sc4 are phi-bin permutations of sc (no ties on generic float data)."""
    from platymatch_b200.estimate_transform.shape_context import get_unary_counts
    g = load_golden("synth400")
    counts, _, _, _ = get_unary_counts(g["fixed_centroid"], float(g["fixed_mean_distance"]), g["fixed"], "fixed")
    h = counts.reshape(4, -1, 30, 12)
    k = np.arange(12)
    assert np.array_equal(h[1][:, :, (k + 6) % 12], h[0])
    assert np.array_equal(h[2][:, :, 11 - k], h[0])
    assert np.array_equal(h[3][:, :, (5 - k) % 12], h[0])


def test_host_entry_points_match_device_path(torch):
    """pm_host_mean_distance / pm_host_shape_context (the numpy callers' entry points, INTEGRATION.md §2) return
    exactly what get_mean_distance / get_unary_counts return."""
    import ctypes
    from platymatch_b200 import _lib
    from platymatch_b200.device import R_EDGES
    from platymatch_b200.estimate_transform.shape_context import get_unary_counts
    from platymatch_b200.utils.utils import get_mean_distance
    lib, vp = _lib.load(), ctypes.c_void_p
    g = load_golden("asset02")
    pts = np.ascontiguousarray(g["fixed"].T[:, :3], dtype=np.float64)
    n = pts.shape[0]
    md = ctypes.c_double()
    _lib.check(lib.pm_host_mean_distance(pts.ctypes.data_as(vp), n, 0, ctypes.byref(md)), "pm_host_mean_distance")
    assert md.value == get_mean_distance(g["fixed"], transposed=False)
    c = np.ascontiguousarray(g["fixed_centroid"], dtype=np.float64).reshape(-1)[:3]
    mean_dist = float(g["fixed_mean_distance"])
    edges = np.ascontiguousarray(R_EDGES, dtype=np.float64)
    counts = np.empty((4, n, 360), dtype=np.uint32)
    dropped = np.empty((4, n), dtype=np.uint32)
    x0 = np.empty(3, dtype=np.float64)
    ties = ctypes.c_ulonglong()
    _lib.check(lib.pm_host_shape_context(pts.ctypes.data_as(vp), n, c.ctypes.data_as(vp), mean_dist,
                                         edges.ctypes.data_as(vp), edges.size, 4, 0, counts.ctypes.data_as(vp),
                                         dropped.ctypes.data_as(vp), x0.ctypes.data_as(vp), ctypes.byref(ties)),
               "pm_host_shape_context")
    d_counts, d_dropped, d_ties, d_x0 = get_unary_counts(c, mean_dist, g["fixed"], "fixed")
    assert np.array_equal(counts, d_counts) and np.array_equal(dropped, d_dropped)
    assert np.array_equal(x0, d_x0) and ties.value == d_ties


# ------------------------------------------------------------------------------ K3
def _unaries(get_unary, g):
    um = get_unary(g["moving_centroid"], float(g["moving_mean_distance"]), g["moving"], "moving")
    uf = get_unary(g["fixed_centroid"], float(g["fixed_mean_distance"]), g["fixed"], "fixed")
    return {"u11": um[0], "u12": um[1], "u21": uf[0], "u22": uf[1], "u23": uf[2], "u24": uf[3]}


def test_chi2_vs_reference_goldens(O, torch, golden):
    """cost matrix within 1e-5 relative of the reference's float64 matrices: the rows and sampled entries the golden
    keeps, and every entry of the oracle's matrix (pinned to the reference's by tests/test_oracle_golden.py)."""
    from platymatch_b200.estimate_transform.shape_context import unary_distance_matrix, get_unary
    u, uo = _unaries(get_unary, golden), _unaries(O.get_unary, golden)
    worst = 0.0
    for tag in HYP_TAGS:
        ka, kb = UNARY_KEYS[tag]
        U = unary_distance_matrix(u[ka], u[kb])
        sub = golden["cost_sub_" + tag]
        checks = [(U[:sub.shape[0]], sub), (U, O.unary_distance_matrix(uo[ka], uo[kb]))]
        if "cost_pick_" + tag in golden:
            checks.append((U.ravel()[golden["cost_pick_idx_" + tag]], golden["cost_pick_" + tag]))
        for got, ref in checks:
            nz = ref > 0
            worst = max(worst, float((np.abs(got - ref)[nz] / ref[nz]).max()))
            assert np.all(got[~nz] == 0.0)                  # identical histograms -> exactly 0, like the reference
    assert worst < 1e-5, worst


@pytest.mark.parametrize("n1,n2", [(1, 1), (3, 130), (129, 127), (700, 900)])
def test_chi2_vs_oracle_shapes(O, torch, n1, n2):
    from platymatch_b200.estimate_transform.shape_context import unary_distance_matrix, get_unary_distance
    rng = np.random.default_rng(n1 * 1000 + n2)
    def hist(n):
        c = rng.poisson(0.6, size=(n, 360)).astype(np.float64) * (rng.random((n, 360)) < 0.4)
        c[:, 0] += 1
        return c / c.sum(1, keepdims=True)
    a, b = hist(n1), hist(n2)
    U, ref = unary_distance_matrix(a, b), O.unary_distance_matrix(a, b)
    assert U.shape == (n1, n2)
    assert np.allclose(U, ref, rtol=1e-5, atol=0)
    assert get_unary_distance(a[0], b[0]) == pytest.approx(ref[0, 0], rel=1e-5)
    assert get_unary_distance(a[0], a[0]) == 0.0


@pytest.mark.parametrize("case", ["disjoint", "one_shared", "odd_shared", "blocks_differ", "dense", "row_only_extra"])
def test_chi2_structured_sparsity(O, torch, case):
    """The kernel skips bins that are empty for a whole 128-block on both sides and folds one-sided bins
    into row / column sums: exercise every list shape (no shared bin, odd counts, per-block differences)."""
    from platymatch_b200.estimate_transform.shape_context import unary_distance_matrix
    rng = np.random.default_rng(len(case))
    n1, n2 = 300, 391

    def hist(n, bins_of_block):
        c = np.zeros((n, 360))
        for blk in range((n + 127) // 128):
            rows = slice(blk * 128, min(n, blk * 128 + 128))
            bins = np.asarray(bins_of_block(blk))
            m = rows.stop - rows.start
            vals = rng.integers(0, 5, size=(m, len(bins))).astype(np.float64)
            vals[np.arange(m), rng.integers(0, len(bins), size=m)] += 1       # no empty histogram
            c[rows][:, bins] = vals
        return c / c.sum(1, keepdims=True)

    if case == "disjoint":
        a, b = hist(n1, lambda q: np.arange(0, 40)), hist(n2, lambda q: np.arange(100, 171))
    elif case == "one_shared":
        a, b = hist(n1, lambda q: np.arange(0, 40)), hist(n2, lambda q: np.arange(39, 90))
    elif case == "odd_shared":
        a, b = hist(n1, lambda q: np.arange(5, 76)), hist(n2, lambda q: np.arange(31, 64))          # 33 shared
    elif case == "blocks_differ":
        a = hist(n1, lambda q: np.arange(q * 50, q * 50 + 97))
        b = hist(n2, lambda q: np.arange(300 - q * 70, 360 - q * 70 + (q % 2)))
    elif case == "dense":
        a, b = hist(n1, lambda q: np.arange(360)), hist(n2, lambda q: np.arange(360))
    else:
        a, b = hist(n1, lambda q: np.arange(0, 359)), hist(n2, lambda q: np.arange(8, 24))
    U, ref = unary_distance_matrix(a, b), O.unary_distance_matrix(a, b)
    assert np.allclose(U, ref, rtol=1e-5, atol=0), float(np.abs(U / ref - 1).max())
    V = unary_distance_matrix(a, a)
    assert np.all(np.diag(V) == 0.0) and np.allclose(V, O.unary_distance_matrix(a, a), rtol=1e-5, atol=0)


# ------------------------------------------------------------------------------ K4
def _check_lap(O, cost, **kw):
    from platymatch_b200.lap import linear_sum_assignment
    from scipy.optimize import linear_sum_assignment as scipy_lsa
    c32 = np.asarray(cost, dtype=np.float32).astype(np.float64)          # the values the GPU solves
    r, c, st = linear_sum_assignment(cost, return_stats=True, **kw)
    ro, co = O.linear_sum_assignment(c32)
    rs, cs = scipy_lsa(c32)
    assert np.array_equal(ro, rs) and np.array_equal(co, cs)             # oracle == scipy on the same matrix
    assert len(np.unique(c)) == len(c) == min(cost.shape) and np.array_equal(r, np.sort(r))
    got, ref = c32[r, c].sum(), c32[ro, co].sum()
    assert got == pytest.approx(ref, rel=1e-12, abs=1e-12), (got, ref, st)
    assert st["total"] == pytest.approx(ref, rel=1e-12, abs=1e-12)
    return (r, c), (ro, co), st


@pytest.mark.parametrize("shape", [(1, 1), (1, 7), (2, 2), (5, 9), (9, 5), (64, 64), (100, 257), (300, 300), (500, 1200)])
@pytest.mark.parametrize("rounds,algo", [(0, 0), (3, 1), (128, 1), (3, 2), (128, 2)])
def test_lap_random_matrices(O, torch, shape, rounds, algo):
    rng = np.random.default_rng(shape[0] * 7 + shape[1])
    cost = rng.random(shape)
    (r, c), (ro, co), st = _check_lap(O, cost, max_bid_rounds=rounds, algorithm=algo)
    assert np.array_equal(c, co)              # continuous random costs: the optimum is unique


@pytest.mark.parametrize("algo", [1, 2])
def test_lap_ties_and_structure(O, torch, algo):
    """Integer costs (many equal-cost optima), constant matrix, permuted diagonal, negative entries."""
    rng = np.random.default_rng(3)
    _check_lap(O, rng.integers(0, 5, size=(60, 80)).astype(float), algorithm=algo)
    _check_lap(O, rng.integers(0, 3, size=(300, 700)).astype(float), algorithm=algo)
    _check_lap(O, np.ones((17, 17)), algorithm=algo)
    perm = rng.permutation(200)
    cost = np.ones((200, 200)); cost[np.arange(200), perm] = 0.0
    (r, c), _, _ = _check_lap(O, cost, algorithm=algo)
    assert np.array_equal(c, perm)
    _check_lap(O, rng.normal(size=(50, 70)), algorithm=algo)
    # all rows want the same few columns: long price wars, list refreshes
    cost = rng.random((400, 900)) + 5.0
    cost[:, :20] -= 5.0
    _check_lap(O, cost, algorithm=algo)


def test_lap_sparse_auction_stats(O, torch):
    """The sparse auction leaves (almost) nothing to the augmenting-path phase on a shape-context-like matrix."""
    rng = np.random.default_rng(11)
    a, b = rng.random((600, 40)), rng.random((800, 40))
    cost = ((a[:, None, :] - b[None, :, :]) ** 2).sum(-1)
    (r, c), (ro, co), st = _check_lap(O, cost, algorithm=1)
    assert np.array_equal(c, co)
    assert st["bids"] >= 600 and st["augmentations"] <= 30, st


def test_lap_on_reference_cost_matrices(O, torch):
    """The assignment scipy produced inside the reference run (golden) is reproduced on the same matrix: the oracle's,
    which tests/test_oracle_golden.py pins to the reference's (it equals the reference's full matrices bit for bit)."""
    from platymatch_b200.lap import linear_sum_assignment
    g = load_golden("synth400")
    u = _unaries(O.get_unary, g)
    for tag in ["11", "12", "13", "14"]:
        ka, kb = UNARY_KEYS[tag]
        U = O.unary_distance_matrix(u[ka], u[kb])
        r, c = linear_sum_assignment(U)
        c32 = U.astype(np.float32).astype(np.float64)
        assert c32[r, c].sum() == pytest.approx(c32[g["lap_row_" + tag], g["lap_col_" + tag]].sum(), rel=1e-9)
        assert U[r, c].sum() == pytest.approx(float(g["lap_cost_" + tag]), rel=1e-6)
        assert np.mean(c == g["lap_col_" + tag]) > 0.98      # float32 rounding may move near-ties only


def test_lap_3k_pair_equal_cost(O, torch):
    """Config 1 size (2700 x 3000): equal optimal cost and identical assignment vs the oracle on the GPU's matrix."""
    import platymatch_b200 as pm
    p = _pair(3000)
    dm, df = pm.describe_cloud(p["moving"], 1), pm.describe_cloud(p["fixed"], 4)
    res = pm.register_described(dm, df, ransac_trials=64, icp_iterations=1, keep_cost=True)
    cost = res["cost"].cpu().numpy()[:, :, :3000].astype(np.float64)
    for q in range(4):
        ro, co = O.linear_sum_assignment(cost[q])
        got = res["assignments"][q][1].cpu().numpy()
        assert res["lap_cost"][q].item() == pytest.approx(cost[q][ro, co].sum(), rel=1e-12)
        assert np.array_equal(got, co), q


# ------------------------------------------------------------------------------ K5
def test_ransac_vs_reference_goldens(O, torch, golden):
    from platymatch_b200.estimate_transform.shape_context import do_ransac
    m, f = golden["moving"], golden["fixed"]
    rs = np.random.RandomState(int(golden["seed"]))
    trials = int(golden["trials"])
    for q, tag in enumerate(HYP_TAGS):
        r, c = golden["lap_row_" + tag], golden["lap_col_" + tag]
        idx = np.stack([rs.choice(len(r), 4, replace=False) for _ in range(trials)])
        A, inl = do_ransac(m[:, r], f[:, c], 4, trials, 16, 'Affine', sample_indices=idx)
        assert inl == int(golden["ransac_inliers"][q]), tag
        assert np.allclose(A, golden["ransac_A"][q], rtol=1e-7, atol=1e-7), tag


def test_ransac_affine_per_trial_counts_and_device_rng(O, D, torch):
    p = _pair(800, seed=8)
    k = p["moving"].shape[1]
    m, f = p["moving"], p["fixed"][:, p["gt_fixed_index"]]
    idx = O.ransac_sample_indices(k, 4, 300, seed=4)
    _, _, inl_o, mats = O.do_ransac(m, f, 4, 300, 16, sample_indices=idx, return_all=True)
    md, fd = D.to_device_points(m), D.to_device_points(f)
    a, inl, trial, per = D.ransac(md, fd, 300, 16.0, 4, torch.from_numpy(idx).cuda(), want_per_trial=True)
    assert np.array_equal(per.cpu().numpy(), inl_o)
    assert trial.item() == int(np.argmax(inl_o))
    # device Philox sampling: deterministic per seed, indices distinct, finds the true affine on clean matches
    a1, i1, _, _ = D.ransac(md, fd, 500, 16.0, 4, None, seed=123)
    a2, i2, _, _ = D.ransac(md, fd, 500, 16.0, 4, None, seed=123)
    assert i1.item() == i2.item() and torch.equal(a1, a2) and i1.item() > 0.9 * k
    # no inliers at all (negative threshold) -> all-ones matrix and 0, as the reference (shape_context.py:120)
    a0, i0, t0, _ = D.ransac(md, fd, 20, -1.0, 4, None, seed=1)
    assert i0.item() == 0 and torch.all(a0 == 1.0) and t0.item() == -1
    # coplanar (degenerate) samples: numpy's pinv still answers (minimum-norm affine), so does the kernel; never NaN
    mflat = m.copy(); mflat[2] = 5.0
    idx3 = O.ransac_sample_indices(k, 4, 50, seed=2)
    _, i3_o, per3_o, _ = O.do_ransac(mflat, f, 4, 50, 16, sample_indices=idx3, return_all=True)
    a3, i3, _, per3 = D.ransac(D.to_device_points(mflat), fd, 50, 16.0, 4, torch.from_numpy(idx3).cuda(), want_per_trial=True)
    assert i3.item() == i3_o and np.array_equal(per3.cpu().numpy(), per3_o) and torch.all(torch.isfinite(a3))


# ------------------------------------------------------------------------------ K6 + small ops
def test_icp_vs_reference_goldens(torch, golden):
    from platymatch_b200.estimate_transform.apply_transform import apply_affine_transform
    from platymatch_b200.estimate_transform.perform_icp import perform_icp
    moved = apply_affine_transform(golden["moving"], golden["A_sc"])
    a_icp, resid = perform_icp(moved, golden["fixed"], 50, 'Affine', verbose=False, return_residuals=True)
    assert np.allclose(a_icp, golden["A_icp"], rtol=1e-7, atol=1e-7)
    assert np.allclose(resid, golden["icp_residuals"], rtol=1e-6, atol=1e-9)
    assert np.abs(a_icp @ golden["A_sc"] - golden["A_final"]).max() < 1e-4


def test_icp_affine_nearest_neighbour_map(O, D, torch):
    p = _pair(1500, seed=2)
    m = O.apply_affine_transform(p["moving"], p["A_gt"])
    _, _, nn = D.icp(D.to_device_points(m), D.to_device_points(p["fixed"]), 1, want_nn=True)
    nn_o, _ = O.nearest(m, p["fixed"])
    assert np.array_equal(nn.cpu().numpy(), nn_o)


@pytest.mark.parametrize("case", ["shell", "filled", "outliers", "lattice_ties", "identical", "flat"])
def test_icp_affine_grid_search_matches_brute_force(O, D, torch, case, monkeypatch):
    """The uniform-grid search returns exactly the brute-force nearest-neighbour map (first minimum in ascending
    index), also with exact distance ties, queries far outside the fixed cloud's box and degenerate boxes."""
    rng = np.random.default_rng(len(case))
    if case == "shell":
        p = _pair(3000, seed=4); f = p["fixed"]; m = O.apply_affine_transform(p["moving"], p["A_gt"])
    elif case == "filled":
        f = rng.random((3, 2500)) * 300; m = rng.random((3, 2000)) * 300
    elif case == "outliers":
        f = rng.random((3, 1500)) * 100; m = np.concatenate([rng.random((3, 900)) * 100, rng.random((3, 100)) * 5000 - 2500], axis=1)
    elif case == "lattice_ties":
        g = np.stack(np.meshgrid(np.arange(12.0), np.arange(12.0), np.arange(12.0), indexing="ij")).reshape(3, -1)
        f = g[:, rng.permutation(g.shape[1])]; m = g[:, :800] + 0.5            # every query has 8 equidistant neighbours
    elif case == "identical":
        f = rng.random((3, 1200)) * 50; m = f[:, rng.permutation(1200)[:900]].copy()
    else:
        f = rng.random((3, 1000)) * 80; f[0] = 7.0; m = rng.random((3, 700)) * 80          # zero extent along z
    _, _, nn = D.icp(D.to_device_points(m), D.to_device_points(f), 1, want_nn=True)
    nn_o, _ = O.nearest(m, f)
    assert np.array_equal(nn.cpu().numpy(), nn_o)
    monkeypatch.setenv("PM_ICP_BRUTE", "1")
    a_b, r_b, nn_b = D.icp(D.to_device_points(m), D.to_device_points(f), 3, want_nn=True)
    monkeypatch.delenv("PM_ICP_BRUTE")
    monkeypatch.setenv("PM_ICP_MULTI_LAUNCH", "1")          # grid search, three launches per iteration
    a_g, r_g, nn_g = D.icp(D.to_device_points(m), D.to_device_points(f), 3, want_nn=True)
    monkeypatch.delenv("PM_ICP_MULTI_LAUNCH")               # grid search, whole loop in one cooperative launch
    a_p, r_p, nn_p = D.icp(D.to_device_points(m), D.to_device_points(f), 3, want_nn=True)
    assert torch.equal(nn_b, nn_g) and torch.equal(nn_b, nn_p)
    if case != "lattice_ties":                               # (there the fit is rank deficient: NaN rows)
        assert torch.allclose(a_b, a_g, rtol=1e-9, atol=1e-9, equal_nan=True)
        assert torch.allclose(a_b, a_p, rtol=1e-9, atol=1e-9, equal_nan=True)
        assert torch.allclose(r_b, r_p, rtol=1e-9, atol=1e-12, equal_nan=True)


def test_fit_apply_compose(O, torch, golden):
    from platymatch_b200.estimate_transform.find_transform import get_affine_transform
    from platymatch_b200.estimate_transform.apply_transform import apply_affine_transform
    m, f = golden["moving"], golden["fixed"]
    assert np.allclose(get_affine_transform(m[:, :50], f[:, :50]), O.get_affine_transform(m[:, :50], f[:, :50]),
                       rtol=1e-8, atol=1e-8)
    assert np.allclose(apply_affine_transform(m, golden["A_gt"]), O.apply_affine_transform(m, golden["A_gt"]),
                       rtol=1e-14, atol=1e-12)
    m4 = np.vstack([m, np.ones((1, m.shape[1]))])
    assert np.allclose(apply_affine_transform(m4, golden["A_gt"]), O.apply_affine_transform(m, golden["A_gt"]))


# ------------------------------------------------------------------------------ pipeline
def test_pipeline_vs_reference_goldens(O, torch, golden):
    """Full unsupervised registration on the reference's inputs with the reference's RNG stream."""
    import platymatch_b200 as pm
    rs = np.random.RandomState(int(golden["seed"]))
    trials = int(golden["trials"])
    k = min(golden["moving"].shape[1], golden["fixed"].shape[1])
    idx = [np.stack([rs.choice(k, 4, replace=False) for _ in range(trials)]) for _ in range(8)]
    res = pm.estimate_transform_unsupervised(golden["moving"], golden["fixed"], ransac_trials=trials,
                                             sample_indices=idx, as_reference=True)
    assert res["inliers"].tolist() == golden["ransac_inliers"].tolist()
    assert res["best"] == int(golden["best"])
    assert np.abs(res["transform"] - golden["A_final"]).max() < 1e-4
    if golden["name"].startswith("asset"):      # reference's own known-answer assertion
        np.testing.assert_array_almost_equal(golden["A_gt"], res["transform"])
    for q, tag in enumerate(HYP_TAGS):
        assert np.array_equal(res["assignments"][q][1], golden["lap_col_" + tag]), tag


def test_pipeline_supervised_vs_reference_goldens(torch):
    import platymatch_b200 as pm
    for name in ("asset02", "synth400"):
        g = load_golden(name)
        res = pm.estimate_transform_supervised(g["moving"], g["fixed"], g["kp_moving"], g["kp_fixed"])
        assert np.allclose(res["transform_sc"], g["A_kp"], rtol=1e-7, atol=1e-7)
        assert np.abs(res["transform"] - g["A_kp_icp"] @ g["A_kp"]).max() < 1e-4


def test_supervised_8k_keypoints(O, torch):
    """BASELINE config 3 (8k pair, 10 keypoint matches): LS affine on the keypoints + ICP, as the reference's
    supervised branch (_dock_widget.py:707-717).  Checked against the oracle port on the same inputs (the
    init and 3 ICP iterations: the CPU distance matrices of 50 would take minutes) and against the ground truth."""
    import platymatch_b200 as pm
    from platymatch_b200.synthetic import make_keypoints
    p = _pair(8000)
    mk, fk = make_keypoints(p, 10, seed=4)
    res3 = pm.estimate_transform_supervised(p["moving"], p["fixed"], mk, fk, icp_iterations=3)
    a_kp = O.get_affine_transform(mk, fk)
    assert np.allclose(res3["transform_sc"], a_kp, rtol=1e-8, atol=1e-8)
    a_icp = O.perform_icp(O.apply_affine_transform(p["moving"], a_kp), p["fixed"], 3)
    assert np.abs(res3["transform"] - a_icp @ a_kp).max() < 1e-4
    res = pm.estimate_transform_supervised(p["moving"], p["fixed"], mk, fk)           # 50 iterations
    moved = O.apply_affine_transform(p["moving"], res["transform"])
    err = np.linalg.norm(moved - p["fixed"][:, p["gt_fixed_index"]], axis=0)
    assert np.median(err) < 4.0, np.median(err)
    assert res["icp_residuals"][-1] <= res["icp_residuals"][0]


def test_registration_12k(O, torch):
    """Beyond the 8k config: 10800 x 12000, sparse auction (its ring still in shared memory) + DENSE augmenting paths
    (the sparse ones would need 276 KB of shared memory at 12000 columns); the true hypothesis wins and the transform
    maps nuclei onto their partners; the LAP cost does not exceed the ground-truth matching's on the same matrix.
    Optimality against the oracle at this size: tests/test_gpu_lap_paths.py (P3)."""
    import platymatch_b200 as pm
    p = _pair(12000)
    res = pm.estimate_transform_unsupervised(p["moving"], p["fixed"], ransac_trials=2000, keep_cost=True, seed=1)
    best = res["best"]
    n1 = p["moving"].shape[1]
    cost = res["cost"][best][:, :12000].astype(np.float64)
    fix_idx = res["assignments"][best][1]
    assert len(np.unique(fix_idx)) == len(fix_idx) == n1
    assert res["lap_cost"][best] <= cost[np.arange(n1), p["gt_fixed_index"]].sum() + 1e-9
    assert res["lap_cost"][best] == pytest.approx(cost[np.arange(n1), fix_idx].sum(), rel=1e-12)
    moved = O.apply_affine_transform(p["moving"], res["transform"])
    err = np.linalg.norm(moved - p["fixed"][:, p["gt_fixed_index"]], axis=0)
    assert np.median(err) < 4.0, np.median(err)
    assert res["inliers"][best] > 3 * np.delete(res["inliers"], best).max()


def test_pipeline_tall_problem(O, torch):
    """More moving than fixed nuclei: solved through the transpose like scipy, pairs ordered by moving index."""
    import platymatch_b200 as pm
    p = _pair(500, seed=9)
    moving, fixed = p["fixed"], p["moving"]        # swap roles: N1 = 500 > N2 = 450
    idx = [O.ransac_sample_indices(450, 4, 200, seed=q) for q in range(4)]
    res = pm.estimate_transform_unsupervised(moving, fixed, ransac_trials=200, sample_indices=idx)
    ref = O.estimate_transform_unsupervised(moving, fixed, ransac_trials=200, hypotheses=O.HYPOTHESES[:4], sample_indices=idx)
    assert res["best"] == ref["best"]
    assert np.allclose(res["lap_cost"], ref["lap_cost"], rtol=1e-5)
    assert np.abs(res["transform"] - ref["transform"]).max() < 1e-4


def test_full_size_properties_8k(O, torch):
    """BASELINE config 2 (8k x 8k): properties that do not need the reference (27 h on the CPU).

    - histogram rows count N-1-dropped neighbours; variants are phi permutations of each other;
    - the LAP result is a valid assignment whose duals certify optimality is not re-derived here, but its
      cost must not exceed the ground-truth matching's cost and must equal the oracle's on the same matrix
      for the true hypothesis (one 7200 x 8000 CPU solve, a few seconds);
    - the recovered transform maps moving nuclei onto their true partners (median error < jitter scale).
    """
    import platymatch_b200 as pm
    p = _pair(8000)
    res = pm.estimate_transform_unsupervised(p["moving"], p["fixed"], ransac_trials=2000, keep_cost=True, seed=1)
    best = res["best"]
    cost = res["cost"][best][:, :8000].astype(np.float64)
    mov_idx, fix_idx = res["assignments"][best]
    assert len(np.unique(fix_idx)) == len(fix_idx) == 7200
    gt_cost = cost[np.arange(7200), p["gt_fixed_index"]].sum()
    assert res["lap_cost"][best] <= gt_cost + 1e-9
    ro, co = O.linear_sum_assignment(cost)
    assert res["lap_cost"][best] == pytest.approx(cost[ro, co].sum(), rel=1e-12)
    moved = O.apply_affine_transform(p["moving"], res["transform"])
    err = np.linalg.norm(moved - p["fixed"][:, p["gt_fixed_index"]], axis=0)
    assert np.median(err) < 4.0, np.median(err)
    assert res["inliers"][best] > 3 * np.delete(res["inliers"], best).max()
