"""Generate golden vectors from the UNMODIFIED reference (runs in the build container only).

TEST INFRASTRUCTURE.  Imports /root/reference through oracle/ref_shim.py, restates the body of
`EstimateTransform._click_run` (`platymatch/_dock_widget.py:526-721`) as a headless driver that
calls the reference's own functions, and writes tests/golden/*.npz.  The fixtures travel to the
GPU box; the reference does not.

    python oracle/make_golden.py [asset02 asset04 synth400]
"""
import contextlib
import io
import os
import re
import sys
import time

import numpy as np
from scipy.optimize import linear_sum_assignment

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, HERE)
sys.path.insert(0, ROOT)
import ref_shim  # noqa: E402

REF = ref_shim.load()
ASSETS = os.path.join(ref_shim.REFERENCE_ROOT, "platymatch", "_tests", "assets")

# ground truth used by the reference's own tests (test_estimate_transform.py:88-91)
A_GT_TEST = np.array([[9.08173020e-01, -2.58092254e-01, 2.21387350e-01, 4.98532315e+00],
                      [-2.85490902e-02, 5.66865806e-01, 7.60292965e-01, -2.13218259e+02],
                      [-2.53059848e-01, -7.49475117e-01, 4.48778146e-01, 5.56203489e+02],
                      [1.73472348e-17, 2.42861287e-17, -4.16333634e-17, 1.00000000e+00]])


def load_asset(name):
    """test_estimate_transform.py:17-21: space-delimited `id x y z`, columns 1:4 flipped to zyx."""
    raw = np.loadtxt(os.path.join(ASSETS, name), delimiter=" ")
    return np.ascontiguousarray(np.flip(raw[:, 1:4], 1).transpose())  # 3 x N


def run_reference(moving, fixed, trials, seed, ransac_error=16, icp_iterations=50, keypoints=None):
    """Headless restatement of _dock_widget.py:526-721 calling the reference's functions."""
    out, t = {}, {}
    tic = time.perf_counter()
    mc = REF.get_centroid(moving, transposed=False)                      # :526
    fc = REF.get_centroid(fixed, transposed=False)                       # :527
    md = REF.get_mean_distance(moving, transposed=False)                 # :531
    fd = REF.get_mean_distance(fixed, transposed=False)                  # :532
    t["mean_distance"] = time.perf_counter() - tic
    out.update(moving_centroid=mc, fixed_centroid=fc, moving_mean_distance=md, fixed_mean_distance=fd)
    mcopy, fcopy = moving.copy(), fixed.copy()                           # :533-534

    tic = time.perf_counter()
    u11, u12, _, _ = REF.get_unary(mc, mean_distance=md, detections=moving, type="moving", transposed=False)
    t["unary_moving"] = time.perf_counter() - tic
    tic = time.perf_counter()
    u21, u22, u23, u24 = REF.get_unary(fc, mean_distance=fd, detections=fixed, type="fixed", transposed=False)
    t["unary_fixed"] = time.perf_counter() - tic
    out["unaries"] = dict(u11=u11, u12=u12, u21=u21, u22=u22, u23=u23, u24=u24)

    tic = time.perf_counter()
    mats = []
    for ua in (u11, u12):                                                # order 11,12,13,14,21,22,23,24 (:556-602)
        for ub in (u21, u22, u23, u24):
            U = np.zeros((moving.shape[1], fixed.shape[1]))
            for i in range(U.shape[0]):
                for j in range(U.shape[1]):
                    U[i, j] = REF.get_unary_distance(ua[i], ub[j])
            mats.append(U)
    t["cost_matrices"] = time.perf_counter() - tic
    out["cost"] = mats

    tic = time.perf_counter()
    assign = [linear_sum_assignment(U) for U in mats]                    # :604-611
    t["lap"] = time.perf_counter() - tic
    out["assign"] = assign

    np.random.seed(seed)                                                 # reference is unseeded; pinned here
    tic = time.perf_counter()
    rs = []
    for (r, c) in assign:                                                # :622-675
        rs.append(REF.do_ransac(mcopy[:, r], fcopy[:, c], min_samples=4, trials=trials,
                                error=ransac_error, transform="Affine"))
    t["ransac"] = time.perf_counter() - tic
    inliers = np.array([x[1] for x in rs])
    best = int(np.argmax(inliers))                                       # :683-703 first max
    a_sc = rs[best][0]
    out.update(ransac_A=np.stack([x[0] for x in rs]), ransac_inliers=inliers, best=best, A_sc=a_sc)

    tic = time.perf_counter()
    buf = io.StringIO()
    with contextlib.redirect_stdout(buf):
        moved = REF.apply_affine_transform(mcopy, a_sc)                  # :714
        a_icp = REF.perform_icp(moved, fcopy, icp_iterations, "Affine")  # :715-717
    t["icp"] = time.perf_counter() - tic
    out["icp_residuals"] = np.array([float(x) for x in re.findall(r"is ([0-9.eE+-]+|nan)", buf.getvalue())])
    out.update(A_icp=a_icp, A_final=a_icp @ a_sc, timing=t)              # :428
    if keypoints is not None:                                            # supervised branch :707-717
        mk, fk = keypoints
        a_kp = REF.get_affine_transform(mk, fk)
        with contextlib.redirect_stdout(io.StringIO()):
            a_kicp = REF.perform_icp(REF.apply_affine_transform(mcopy, a_kp), fcopy, icp_iterations, "Affine")
        out.update(kp_moving=mk, kp_fixed=fk, A_kp=a_kp, A_kp_icp=a_kicp)
    return out


def counts_of(sc):
    """Reference rows are count/sum(count) (shape_context.py:41); recover the integer counts.

    The row sum is the number of counted neighbours; it is N-1 unless a neighbour fell outside
    bins 0..359 (un-clamped index) or was NaN.  Find the integer total that makes every entry integral.
    """
    n = sc.shape[0]
    counts = np.zeros(sc.shape, dtype=np.uint16)
    totals = np.zeros(n, dtype=np.int32)
    for i in range(n):
        for tot in range(n - 1, 0, -1):
            c = sc[i] * tot
            if np.abs(c - np.round(c)).max() < 1e-6 and abs(np.round(c).sum() - tot) < 0.5:
                counts[i] = np.round(c).astype(np.uint16)
                totals[i] = tot
                break
        else:
            raise RuntimeError("could not recover counts for row %d" % i)
    return counts, totals


def save_case(name, moving, fixed, res, trials, seed, sub_rows=16, picks=4000, extra=None):
    d = dict(moving=moving, fixed=fixed, trials=trials, seed=seed,
             moving_centroid=res["moving_centroid"], fixed_centroid=res["fixed_centroid"],
             moving_mean_distance=res["moving_mean_distance"], fixed_mean_distance=res["fixed_mean_distance"],
             ransac_A=res["ransac_A"], ransac_inliers=res["ransac_inliers"], best=res["best"],
             A_sc=res["A_sc"], A_icp=res["A_icp"], A_final=res["A_final"], icp_residuals=res["icp_residuals"],
             timing_keys=np.array(list(res["timing"].keys())), timing_vals=np.array(list(res["timing"].values())))
    for k, sc in res["unaries"].items():
        c, tot = counts_of(sc)
        d["counts_" + k], d["totals_" + k] = c, tot
        d["rowsum_" + k] = sc.sum(1)
        d["sc_rows_" + k] = sc[:8]                       # a few raw float64 rows (normalisation check)
    names = ["11", "12", "13", "14", "21", "22", "23", "24"]
    for q, (U, (r, c)) in enumerate(zip(res["cost"], res["assign"])):
        tag = names[q]
        d["lap_row_" + tag], d["lap_col_" + tag] = r.astype(np.int32), c.astype(np.int32)
        d["lap_cost_" + tag] = U[r, c].sum()
        d["cost_rowsum_" + tag], d["cost_colsum_" + tag] = U.sum(1), U.sum(0)
        d["cost_sub_" + tag] = U[:sub_rows]
        # a seeded sample of the remaining entries instead of the whole matrix keeps the fixture under 1 MB
        pool = np.arange(sub_rows * U.shape[1], U.size)
        idx = np.sort(np.random.default_rng(q).choice(pool, min(picks, pool.size), replace=False)).astype(np.int32)
        d["cost_pick_idx_" + tag], d["cost_pick_" + tag] = idx, U.ravel()[idx]
    if extra:
        d.update(extra)
    for k in ("kp_moving", "kp_fixed", "A_kp", "A_kp_icp"):
        if k in res:
            d[k] = res[k]
    path = os.path.join(ROOT, "tests", "golden", name + ".npz")
    np.savez_compressed(path, **d)
    print(name, "->", path, "%.1f MB" % (os.path.getsize(path) / 1e6), "timing", res["timing"],
          "inliers", res["ransac_inliers"], "max|A_final-A_gt|",
          np.abs(res["A_final"] - extra["A_gt"]).max() if extra and "A_gt" in extra else None, flush=True)


def main(which):
    if "asset02" in which:   # test_shape_context_2 (test_estimate_transform.py:75-140), current 8-matrix pipeline
        m = load_asset("02-insitu.csv")
        f = REF.apply_affine_transform(m, A_GT_TEST)
        rng = np.random.default_rng(7)
        sel = rng.choice(m.shape[1], 10, replace=False)
        res = run_reference(m, f, trials=2000, seed=0, keypoints=(m[:, sel], f[:, sel]))
        save_case("asset02", m, f, res, 2000, 0, extra=dict(A_gt=A_GT_TEST))
    if "asset04" in which:   # test_shape_context_3 uses asset 04 with the same ground truth
        m = load_asset("04-insitu.csv")
        f = REF.apply_affine_transform(m, A_GT_TEST)
        res = run_reference(m, f, trials=500, seed=1)
        save_case("asset04", m, f, res, 500, 1, extra=dict(A_gt=A_GT_TEST))
    if "synth400" in which:  # rectangular, noisy: SURVEY §8d generator (jitter 2 px, 10 % dropout)
        from platymatch_b200.synthetic import make_pair, make_keypoints
        p = make_pair(400, seed=400)
        res = run_reference(p["moving"], p["fixed"], trials=1000, seed=2, keypoints=make_keypoints(p, 10, seed=3))
        save_case("synth400", p["moving"], p["fixed"], res, 1000, 2,
                  extra=dict(A_gt=p["A_gt"], gt_fixed_index=p["gt_fixed_index"]))


if __name__ == "__main__":
    main(sys.argv[1:] or ["asset02", "asset04", "synth400"])
