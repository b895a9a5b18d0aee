"""DESIGN §8 row 8 — the thin-plate spline deformation.  Contract: scipy.interpolate.RBFInterpolator(kernel='linear',
degree=1, smoothing) for the fit and the point warp, map_coordinates(src, RBFInterpolator(...)(grid), order,
mode='constant', cval) for the volume warp.  The system matrix is bit-equal to its numpy restatement; fits within 1e-7
voxel of scipy; the volume warp samples exactly at the coordinates pm_spline_eval gives and matches the scipy oracle to
the row-5 bars, away from voxels whose oracle coordinate lies within 1e-6 of a rounding or domain boundary."""
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import spline_oracle as SO  # noqa: E402

pytestmark = pytest.mark.gpu

NEAR = 1e-6                 # oracle coordinates this close to a rounding or domain boundary may round either way


def _shell(k, seed):
    """k nuclei-like centres (3, k) of a make_fixed_cloud shell and a smooth displacement of them as the targets."""
    from platymatch_b200.synthetic import make_deformed_pair
    rng = np.random.default_rng(seed)
    p = make_deformed_pair(max(k, 40), seed=seed, dropout=0.0)
    y = p["fixed"][:, rng.permutation(p["fixed"].shape[1])[:k]]
    if k < 40:                                              # a handful of points: spread, not on a shell
        y = rng.uniform(0, 300, size=(3, k))
    from platymatch_b200.synthetic import deformation_field
    d = y + deformation_field(y, p["field"]) + rng.normal(0, 1.0, size=y.shape)
    return y, d


@pytest.mark.parametrize("k", [4, 5, 300, 3000])
def test_system_matrix_bit_equal(k):
    import torch
    from platymatch_b200 import device as D
    from platymatch_b200.estimate_transform.deformable import shift_scale
    y, _ = _shell(k, seed=k)
    y = np.ascontiguousarray(y.T)
    shift, scale = shift_scale(y)
    for lam in (0.0, 2.5):
        lhs = D.spline_system(torch.from_numpy(y).cuda(), torch.from_numpy(np.r_[shift, scale]).cuda(), lam)
        got, want = lhs.cpu().numpy(), SO.system_matrix(y, shift, scale, lam)
        assert np.array_equal(got.view(np.uint64), want.view(np.uint64)), (k, lam)
    # a padded leading dimension leaves the pad untouched
    out = torch.full((k + 4, k + 9), 7.0, dtype=torch.float64, device="cuda")
    D.spline_system(torch.from_numpy(y).cuda(), torch.from_numpy(np.r_[shift, scale]).cuda(), 1.0, out=out)
    o = out.cpu().numpy()
    assert np.array_equal(o[:, :k + 4], SO.system_matrix(y, shift, scale, 1.0)) and np.all(o[:, k + 4:] == 7.0)


@pytest.mark.parametrize("lam", [0.0, 1.0, 100.0])
@pytest.mark.parametrize("k", [4, 10, 300, 3000, 8000])
def test_fit_and_apply_match_scipy(k, lam):
    from platymatch_b200.estimate_transform.deformable import apply_spline, fit_spline
    y, d = _shell(k, seed=100 + k)
    sp = fit_spline(y, d, smoothing=lam)
    ref = SO.rbf(y, d, lam)
    rng = np.random.default_rng(k)
    lo, hi = y.min(axis=1), y.max(axis=1)
    q = rng.uniform(lo - 0.1 * (hi - lo), hi + 0.1 * (hi - lo), size=(2000, 3)).T
    for pts in (y, q):
        got = apply_spline(sp, pts)
        err = np.abs(got - ref(pts.T).T).max()
        assert err <= 1e-7, (k, lam, err)
    if lam == 0.0:
        assert np.abs(apply_spline(sp, y) - d).max() <= 1e-7
    host = sp.to_numpy()
    assert np.array_equal(host["shift"], ref._shift) and np.array_equal(host["scale"], ref._scale)
    assert np.abs(host["coeffs"] - ref._coeffs).max() <= 1e-6 * max(1.0, np.abs(ref._coeffs).max())


def _spline_case(name):
    """(source shape, output shape, source points (3, K), target points (3, K), smoothing, cval) of the warp tests.
    A spline maps OUTPUT voxel indices to SOURCE coordinates, so it is fitted from output-grid points to source ones."""
    rng = np.random.default_rng(len(name))

    def warp_points(k, out_shape, src_shape, amp):
        o = np.array(out_shape, dtype=np.float64)[:, None]
        s = np.array(src_shape, dtype=np.float64)[:, None]
        y = rng.uniform(-0.1, 1.1, size=(3, k)) * (o - 1)
        t = (y / np.maximum(o - 1, 1)) * (s - 1) + amp * np.sin(y / 7.0 + rng.uniform(0, 6, size=(3, 1)))
        return y, t
    if name == "k5_larger_out":
        s, o = (19, 23, 37), (21, 26, 35)
        y, t = warp_points(5, o, s, 1.5)
        return s, o, y, t, 0.0, 0.0
    if name == "k400_larger_out":
        s, o = (19, 23, 37), (22, 29, 41)
        y, t = warp_points(400, o, s, 1.5)
        return s, o, y, t, 1.0, 0.0
    if name == "k400_smaller_out":
        s, o = (30, 41, 45), (17, 19, 22)
        y, t = warp_points(400, o, s, 2.0)
        return s, o, y, t, 1.0, -7.5
    if name == "identity_like":
        s = o = (13, 17, 21)
        y = rng.uniform(0, 1, size=(3, 40)) * (np.array(o)[:, None] - 1)
        return s, o, y, y.copy(), 0.0, 0.0
    if name == "all_outside":
        s, o = (8, 9, 10), (5, 6, 7)
        y, t = warp_points(5, o, s, 0.5)
        return s, o, y, t + np.array([[1000.0], [0.0], [0.0]]), 0.0, 3.0
    raise KeyError(name)


CASES = ["k5_larger_out", "k400_larger_out", "k400_smaller_out", "identity_like", "all_outside"]


def _source(shape, dtype, seed):
    rng = np.random.default_rng(seed)
    if dtype == np.uint16:
        return rng.integers(0, 65536, size=shape).astype(np.uint16)
    if dtype == np.int32:
        return rng.integers(-100000, 100000, size=shape).astype(np.int32)
    return rng.uniform(-50.0, 50.0, size=shape).astype(np.float32)


def _near_boundary(c, shape):
    """(N,) voxels whose coordinate (3, N) lies within NEAR of a rounding (.5) or domain (0, n - 1) boundary."""
    n = np.array(shape, dtype=np.float64)[:, None]
    frac = c - np.floor(c)
    near = (np.abs(frac - 0.5) < NEAR) | (np.abs(c) < NEAR) | (np.abs(c - (n - 1)) < NEAR)
    return np.any(near, axis=0)


@pytest.mark.parametrize("order", [0, 1])
@pytest.mark.parametrize("dtype", [np.int32, np.uint16, np.float32], ids=["int32", "uint16", "float32"])
@pytest.mark.parametrize("case", CASES)
def test_warp_matches_scipy_oracle(case, dtype, order):
    import scipy.ndimage as nd
    import torch
    from platymatch_b200 import device as D
    from platymatch_b200.estimate_transform.deformable import fit_spline
    sshape, oshape, y, t, lam, cval = _spline_case(case)
    src = _source(sshape, dtype, seed=len(case) + order)
    sp = fit_spline(y, t, smoothing=lam)
    out = D.to_host_volume(D.resample_spline(D.to_device_volume(src), sp.centres, sp.coeffs, sp.shift_scale, oshape,
                                             order, cval))
    g = SO.grid(oshape)
    c_ref = SO.rbf(y, t, lam)(g).T                                            # the oracle's coordinates
    c_gpu = D.spline_eval(sp.centres, sp.coeffs, sp.shift_scale, torch.from_numpy(g).cuda()).cpu().numpy().T
    assert np.abs(c_gpu - c_ref).max() <= 1e-7
    ref = nd.map_coordinates(src, c_ref, order=order, mode="constant", cval=cval).reshape(oshape)
    near = _near_boundary(c_ref, sshape).reshape(oshape)
    got = out
    if order == 0:
        diff = got != ref
        assert not np.any(diff & ~near), int(np.count_nonzero(diff & ~near))
        print("%s %s order 0: %d voxels near a boundary, %d of them differ" %
              (case, np.dtype(dtype).name, np.count_nonzero(near), np.count_nonzero(diff)))
    else:
        exact_ref = nd.map_coordinates(src.astype(np.float64), c_ref, order=1, mode="constant", cval=cval).reshape(oshape)
        exact_gpu = nd.map_coordinates(src.astype(np.float64), c_gpu, order=1, mode="constant", cval=cval).reshape(oshape)
        slack = np.abs(exact_gpu - exact_ref)                                 # the coordinate-induced difference
        ok = ~near
        if dtype == np.float32:
            bound = np.spacing(np.abs(ref)).astype(np.float64) + slack
            assert np.all(np.abs(got.astype(np.float64) - ref)[ok] <= bound[ok])
        else:
            tie = np.abs(np.abs(exact_ref - np.trunc(exact_ref)) - 0.5) < 1e-9 + slack
            d = got.astype(np.int64) - ref.astype(np.int64)
            assert np.all(np.abs(d[ok]) <= 1) and not np.any(d[ok & ~tie])
    if case == "identity_like":
        inner = ~near
        assert np.array_equal(got[inner], src[inner]) if order == 0 else True
    if case == "all_outside":
        assert np.all(got == np.asarray(cval).astype(dtype))


@pytest.mark.parametrize("dtype", [np.int32, np.uint16, np.float32], ids=["int32", "uint16", "float32"])
def test_warp_samples_at_eval_coordinates(dtype):
    """pm_spline_eval on every voxel gives the coordinates: the numpy order-0 sampler at them equals pm_resample_spline
    bit for bit (no boundary exception: the two kernels share the evaluation routine)."""
    import torch
    from platymatch_b200 import device as D
    from platymatch_b200.estimate_transform.deformable import fit_spline
    sshape, oshape, y, t, lam, cval = _spline_case("k400_larger_out")
    oshape = (13, 37, 45)
    sp = fit_spline(y, t, smoothing=lam)
    src = _source(sshape, dtype, seed=3)
    out = D.to_host_volume(D.resample_spline(D.to_device_volume(src), sp.centres, sp.coeffs, sp.shift_scale, oshape,
                                             0, -2.0))
    c = D.spline_eval(sp.centres, sp.coeffs, sp.shift_scale, torch.from_numpy(SO.grid(oshape)).cuda()).cpu().numpy().T
    want = SO.sample_order0(src, c, -2.0).reshape(oshape)
    assert np.array_equal(out.view(np.uint8), want.view(np.uint8))
    assert np.count_nonzero(want != np.asarray(-2.0).astype(dtype)) > want.size // 2


def test_warp_beyond_2_31_voxels():
    """An int32 source of 2048 x 1024 x 1040 = 2.18e9 voxels built from its linear index, warped (order 0) through a
    K = 8 spline into a small grid that spans it; 1e5 output voxels checked against the index pattern at the
    coordinates pm_spline_eval gives."""
    import torch
    from platymatch_b200 import device as D
    from platymatch_b200.estimate_transform.deformable import fit_spline
    P = 2147483629
    sshape = (2048, 1024, 1040)
    plane = sshape[1] * sshape[2]
    lin = torch.arange(plane, dtype=torch.int64, device="cuda")
    src = torch.empty(sshape, dtype=torch.int32, device="cuda")
    for z in range(sshape[0]):
        src[z] = torch.remainder(lin + z * plane, P).to(torch.int32).view(sshape[1], sshape[2])
    del lin
    oshape = (128, 64, 65)
    rng = np.random.default_rng(1)
    y = rng.uniform(0, 1, size=(3, 8)) * (np.array(oshape)[:, None] - 1)
    y[:, :4] = np.array([[0, 0, 0], [127, 0, 0], [0, 63, 0], [0, 0, 64]], dtype=np.float64).T
    scale = (np.array(sshape, dtype=np.float64) - 1.5) / (np.array(oshape) - 1)
    t = y * scale[:, None] + 0.3 + rng.normal(0, 0.5, size=y.shape)
    sp = fit_spline(y, t, smoothing=0.0)
    out = D.to_host_volume(D.resample_spline(src, sp.centres, sp.coeffs, sp.shift_scale, oshape, 0, -1.0))
    del src
    torch.cuda.empty_cache()
    flat = rng.choice(out.size, 100000, replace=False)
    g = np.stack(np.unravel_index(flat, oshape), axis=1).astype(np.float64)
    c = D.spline_eval(sp.centres, sp.coeffs, sp.shift_scale, torch.from_numpy(g).cuda()).cpu().numpy().T
    inside = np.all((c >= 0) & (c <= np.array(sshape)[:, None] - 1), axis=0)
    idx = np.floor(np.where(inside, c, 0) + 0.5).astype(np.int64)
    lin_src = (idx[0] * sshape[1] + idx[1]) * sshape[2] + idx[2]
    want = np.where(inside, lin_src % P, -1)
    assert inside.mean() > 0.9 and lin_src[inside].max() >= 2 ** 31
    assert np.array_equal(out.reshape(-1)[flat], want)


def test_warp_on_side_stream():
    """A fit and a warp enqueued on a side stream give the same bytes as on the default stream."""
    import torch
    from platymatch_b200 import device as D
    from platymatch_b200.estimate_transform.deformable import fit_spline
    sshape, oshape, y, t, lam, cval = _spline_case("k400_smaller_out")
    src = D.to_device_volume(_source(sshape, np.float32, seed=9))
    torch.cuda.synchronize()
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        sp = fit_spline(y, t, smoothing=lam)
        got = D.resample_spline(src, sp.centres, sp.coeffs, sp.shift_scale, oshape, 1, cval)
    side.synchronize()
    sp0 = fit_spline(y, t, smoothing=lam)
    ref = D.resample_spline(src, sp0.centres, sp0.coeffs, sp0.shift_scale, oshape, 1, cval)
    assert np.array_equal(D.to_host_volume(got).view(np.uint32), D.to_host_volume(ref).view(np.uint32))


def _held_out_errors(moving, fixed, gt, T, held, smoothing):
    """Refit without the held-out moving nuclei, then (spline, affine) errors at them against their true partners."""
    from platymatch_b200.estimate_transform.deformable import apply_spline, estimate_deformation
    train = np.flatnonzero(~held)
    dfm = estimate_deformation(moving[:, train], fixed, T, smoothing=smoothing)
    truth = fixed[:, gt[held]]
    e_spline = np.linalg.norm(apply_spline(dfm["forward"], moving[:, held]) - truth, axis=0)
    e_affine = np.linalg.norm(T[:3, :3] @ moving[:, held] + T[:3, 3:4] - truth, axis=0)
    return dfm, train, e_spline, e_affine


def test_registration_then_deformation():
    """make_deformed_pair -> unsupervised registration -> estimate_deformation.  On held-out nuclei (refit without them)
    the spline's median error is at most half the affine's; fit, residuals and held-out errors equal the scipy oracle
    on the same pairs within 1e-6."""
    import platymatch_b200 as pm
    from platymatch_b200.estimate_transform.deformable import DEFAULT_SMOOTHING, apply_spline, estimate_deformation
    from platymatch_b200.synthetic import make_deformed_pair
    p = make_deformed_pair(1500, seed=5)
    m, f, gt = p["moving"], p["fixed"], p["gt_fixed_index"]
    res = pm.estimate_transform_unsupervised(m, f, ransac_trials=4000, seed=1)
    T = res["transform"]
    dfm = estimate_deformation(m, f, T)
    assert np.mean(gt[dfm["moving_index"]] == dfm["fixed_index"]) > 0.9
    assert dfm["median_residual_spline"] < dfm["median_residual_affine"]
    mi, fi = dfm["moving_index"], dfm["fixed_index"]
    fwd = SO.rbf(m[:, mi], f[:, fi], DEFAULT_SMOOTHING)
    r_spline = np.median(np.linalg.norm(fwd(m[:, mi].T).T - f[:, fi], axis=0))
    assert abs(dfm["median_residual_spline"] - r_spline) <= 1e-6
    inv = SO.rbf(f[:, fi], m[:, mi], DEFAULT_SMOOTHING)
    assert np.abs(apply_spline(dfm["inverse"], f) - inv(f.T).T).max() <= 1e-6
    held = np.random.default_rng(0).random(m.shape[1]) < 0.2
    d2, train, e_spline, e_affine = _held_out_errors(m, f, gt, T, held, DEFAULT_SMOOTHING)
    ref = SO.rbf(m[:, train[d2["moving_index"]]], f[:, d2["fixed_index"]], DEFAULT_SMOOTHING)
    e_ref = np.linalg.norm(ref(m[:, held].T).T - f[:, gt[held]], axis=0)
    assert np.abs(e_spline - e_ref).max() <= 1e-6
    print("held-out median error: affine %.3f, spline %.3f (%d nuclei, %d pairs); pair residual affine %.3f spline %.3f"
          % (np.median(e_affine), np.median(e_spline), held.sum(), d2["moving_index"].size,
             dfm["median_residual_affine"], dfm["median_residual_spline"]))
    assert np.median(e_spline) <= 0.5 * np.median(e_affine)


def test_deformable_warp_of_label_volumes():
    """Label volumes of ~400 nuclei rendered at a deformed pair's centres: the moving one warped into the fixed grid with
    the best affine (least squares on the true pairs) and with the spline of estimate_deformation.  match_labels at IoU
    0.5 finds strictly more true positives, and Dice is higher, for the spline warp."""
    from platymatch_b200.estimate_transform.deformable import estimate_deformation
    from platymatch_b200.evaluate_metrics import match_labels
    from platymatch_b200.synthetic import make_deformed_pair, make_label_volume
    from platymatch_b200.utils.images import transform_image, transform_image_deformable
    p = make_deformed_pair(445, seed=3)
    m, f, gt = p["moving"], p["fixed"], p["gt_fixed_index"]
    f = f[:, gt]                                            # fixed nuclei in the moving order: nucleus i is id i + 1 in both
    f = f - f.min(axis=1, keepdims=True) + 8.0
    m = m - m.min(axis=1, keepdims=True) + 8.0
    fshape = tuple(int(v) for v in np.ceil(f.max(axis=1) + 9.0))
    mshape = tuple(int(v) for v in np.ceil(m.max(axis=1) + 9.0))
    fixed_vol = make_label_volume(fshape, radius=(4.0, 6.0), seed=1, centers=f.T)
    moving_vol = make_label_volume(mshape, radius=(4.0, 6.0), seed=1, centers=m.T, dtype=np.uint16)
    mh = np.vstack([m, np.ones(m.shape[1])])
    T = np.vstack([f @ np.linalg.pinv(mh), [0.0, 0.0, 0.0, 1.0]])
    dfm = estimate_deformation(m, f, T)
    w_affine = transform_image(moving_vol, T, fshape, order=0)
    w_spline = transform_image_deformable(moving_vol, dfm, fshape, order=0)
    assert w_spline.dtype == np.uint16
    r_affine = match_labels(fixed_vol, w_affine, (0.5,))
    r_spline = match_labels(fixed_vol, w_spline, (0.5,))
    tp_a, tp_s = r_affine["per_threshold"][0]["tp"], r_spline["per_threshold"][0]["tp"]
    print("%d nuclei, %s grid: affine Dice %.4f tp %d / spline Dice %.4f tp %d at IoU 0.5 (%d pairs)" %
          (m.shape[1], fshape, r_affine["dice"], tp_a, r_spline["dice"], tp_s, dfm["moving_index"].size))
    assert tp_s > tp_a and r_spline["dice"] > r_affine["dice"]


def test_resample_spline_refuses_host_tensors():
    import torch
    from platymatch_b200 import device as D
    c = torch.zeros((8, 3), dtype=torch.float64, device="cuda")
    co = torch.zeros((12, 3), dtype=torch.float64, device="cuda")
    ss = torch.ones(6, dtype=torch.float64, device="cuda")
    with pytest.raises(ValueError):
        D.resample_spline(torch.zeros((4, 5, 6), dtype=torch.int32), c, co, ss, (4, 5, 6))
    with pytest.raises(ValueError):
        D.resample_spline(torch.zeros((4, 5, 6), dtype=torch.int32, device="cuda"), c.cpu(), co, ss, (4, 5, 6))
    with pytest.raises(ValueError):
        D.resample_spline(torch.zeros((4, 5, 6), dtype=torch.int32, device="cuda"), c, co[:11], ss, (4, 5, 6))
