"""Pins the CPU oracle (oracle/oracle.py + oracle/pm_oracle.c) to the UNMODIFIED reference.

tests/golden/*.npz were dumped by oracle/make_golden.py from /root/reference's own functions
(assets 02 / 04 of the reference's test-suite with the ground truth of
platymatch/_tests/test_estimate_transform.py:88-91, plus a rectangular noisy synthetic pair).
Every oracle stage is compared with what the reference produced on the same inputs.  Of each reference
cost matrix the fixtures keep the first 16 rows, all row and column sums and a seeded sample of the
other entries (`cost_pick_*`), which keeps every fixture under 1 MB.
"""
import numpy as np
import pytest

from conftest import HYP_TAGS, UNARY_KEYS


def _unaries(O, g):
    mc, fc = g["moving_centroid"], g["fixed_centroid"]
    um = O.get_unary(mc, float(g["moving_mean_distance"]), g["moving"], "moving")
    uf = O.get_unary(fc, float(g["fixed_mean_distance"]), g["fixed"], "fixed")
    return {"u11": um[0], "u12": um[1], "u21": uf[0], "u22": uf[1], "u23": uf[2], "u24": uf[3]}


def test_centroid_and_mean_distance(O, golden):
    assert np.allclose(O.get_centroid(golden["moving"], False), golden["moving_centroid"], rtol=1e-14)
    assert np.allclose(O.get_centroid(golden["fixed"], False), golden["fixed_centroid"], rtol=1e-14)
    assert O.get_mean_distance(golden["moving"], False) == pytest.approx(float(golden["moving_mean_distance"]), rel=1e-13)
    assert O.get_mean_distance(golden["fixed"], False) == pytest.approx(float(golden["fixed_mean_distance"]), rel=1e-13)


def test_shape_context_histograms_bit_exact(O, golden):
    """Integer histograms of all 6 descriptor sets equal the reference's, neighbour for neighbour."""
    for cloud, typ, keys in (("moving", "moving", ["u11", "u12"]), ("fixed", "fixed", ["u21", "u22", "u23", "u24"])):
        pts = golden[cloud].T
        x0 = O.pca_first_axis(pts)
        for v, k in enumerate(keys, start=1):
            counts, dropped = O.shape_context_counts(pts, golden[cloud + "_centroid"],
                                                     float(golden[cloud + "_mean_distance"]), x0, v)
            assert np.array_equal(counts, golden["counts_" + k].astype(np.uint32)), (golden["name"], k)
            assert np.array_equal(counts.sum(1), golden["totals_" + k])
            assert np.array_equal(dropped, pts.shape[0] - 1 - golden["totals_" + k])
            sc = O.normalise_counts(counts)
            assert np.array_equal(sc[:8], golden["sc_rows_" + k])          # float64 rows, bit for bit


def test_chi2_cost_matrices(O, golden):
    u = _unaries(O, golden)
    for tag in HYP_TAGS:
        ka, kb = UNARY_KEYS[tag]
        U = O.unary_distance_matrix(u[ka], u[kb])
        sub = golden["cost_sub_" + tag]
        assert np.allclose(U[:sub.shape[0]], sub, rtol=1e-14, atol=0), tag
        assert np.allclose(U.sum(1), golden["cost_rowsum_" + tag], rtol=1e-12)
        assert np.allclose(U.sum(0), golden["cost_colsum_" + tag], rtol=1e-12)
        if "cost_pick_" + tag in golden:        # seeded sample of the reference's entries below those rows
            got = U.ravel()[golden["cost_pick_idx_" + tag]]
            assert np.allclose(got, golden["cost_pick_" + tag], rtol=1e-14, atol=0), tag


def test_lap_matches_scipy_on_reference_matrices(O, golden):
    """Oracle LAP == scipy's result recorded from the reference run (assignment and total cost)."""
    u = _unaries(O, golden)
    for tag in HYP_TAGS:
        ka, kb = UNARY_KEYS[tag]
        U = O.unary_distance_matrix(u[ka], u[kb])
        r, c = O.linear_sum_assignment(U)
        assert U[r, c].sum() == pytest.approx(float(golden["lap_cost_" + tag]), rel=1e-12)
        assert np.array_equal(r, golden["lap_row_" + tag])
        assert np.array_equal(c, golden["lap_col_" + tag]), tag


def test_ransac_with_reference_rng_stream(O, golden):
    """Same seeded numpy stream as the reference run -> same inlier counts and hypotheses."""
    m, f = golden["moving"], golden["fixed"]
    rs = np.random.RandomState(int(golden["seed"]))
    trials = int(golden["trials"])
    for q, tag in enumerate(HYP_TAGS):
        r, c = golden["lap_row_" + tag], golden["lap_col_" + tag]
        idx = np.stack([rs.choice(len(r), 4, replace=False) for _ in range(trials)])
        A, inl = O.do_ransac(m[:, r], f[:, c], 4, trials, 16, sample_indices=idx)
        assert inl == int(golden["ransac_inliers"][q]), tag
        assert np.allclose(A, golden["ransac_A"][q], rtol=1e-9, atol=1e-9), tag


def test_icp_and_final_transform(O, golden):
    moved = O.apply_affine_transform(golden["moving"], golden["A_sc"])
    a_icp, resid = O.perform_icp(moved, golden["fixed"], 50, return_residuals=True)
    assert np.allclose(a_icp, golden["A_icp"], rtol=1e-9, atol=1e-9)
    assert np.allclose(resid, golden["icp_residuals"], rtol=1e-7, atol=1e-12)
    assert np.allclose(a_icp @ golden["A_sc"], golden["A_final"], rtol=1e-9, atol=1e-9)


def test_supervised_branch(O, golden):
    if "kp_moving" not in golden:
        pytest.skip("no keypoints in this fixture")
    res = O.estimate_transform_supervised(golden["moving"], golden["fixed"], golden["kp_moving"], golden["kp_fixed"])
    assert np.allclose(res["transform_sc"], golden["A_kp"], rtol=1e-9, atol=1e-9)
    assert np.allclose(res["transform_icp"], golden["A_kp_icp"], rtol=1e-9, atol=1e-9)


def test_reference_known_answer(golden):
    """The property the reference's own tests assert (test_estimate_transform.py:72,140,208): the
    noise-free assets recover the ground-truth affine to 6 decimals."""
    if golden["name"].startswith("asset"):
        np.testing.assert_array_almost_equal(golden["A_gt"], golden["A_final"])


# ------------------------------------------------------------------------------ transform='Similar' (SURVEY §8f row 1)
FIT_TAGS = ["k4", "k10", "all", "k12n", "alln"]


def test_similar_oracle_vs_reference_goldens(O):
    """oracle.get_similar_transform against tests/golden/similar.npz (oracle/make_golden_similar.py): the corrected
    variant (`q = D[:, 0]`, Horn as published = what the CUDA path implements) against the reference's source with
    that one token changed, and the as-shipped variant (`q = D[0]`) against the unmodified reference."""
    from conftest import load_golden
    g = load_golden("similar")
    for tag in FIT_TAGS:
        m, f = g["fit_m_" + tag], g["fit_f_" + tag]
        assert np.allclose(O.get_similar_transform(m, f), g["fit_fixed_" + tag], rtol=1e-9, atol=1e-9), tag
        # as shipped: the result depends on the signs LAPACK's dgeev gives the eigenvectors; same numpy build -> equal
        assert np.allclose(O.get_similar_transform(m, f, as_shipped=True), g["fit_shipped_" + tag], rtol=1e-7, atol=1e-7), tag
    # the corrected variant recovers an exact similarity; the shipped one does not (documented in DESIGN.md)
    assert np.abs(g["fit_fixed_all"] - g["A_gt"]).max() < 1e-9
    assert np.abs(g["fit_shipped_all"] - g["A_gt"]).max() > 1.0


def test_similar_ransac_and_icp_oracle_vs_reference_goldens(O):
    from conftest import load_golden
    g = load_golden("similar")
    k, trials = g["moving"].shape[1], int(g["ransac_trials"])
    rs = np.random.RandomState(int(g["ransac_seed"]))
    idx = np.stack([rs.choice(k, 4, replace=False) for _ in range(trials)])
    for tag, shipped in (("fixed", False), ("shipped", True)):
        A, inl = O.do_ransac(g["moving"], g["ransac_f"], 4, trials, 16, "Similar", sample_indices=idx, as_shipped=shipped)
        assert inl == int(g["ransac_inliers_" + tag]), tag
        assert np.allclose(A, g["ransac_A_" + tag], rtol=1e-7, atol=1e-7), tag
        if not shipped:     # (as shipped the iteration is chaotic - not a rotation - and amplifies 1e-16 differences)
            a_icp = O.perform_icp(g["icp_start"], g["fixed"], 20, "Similar")
            assert np.allclose(a_icp, g["icp_A_fixed"], rtol=1e-6, atol=1e-6)
