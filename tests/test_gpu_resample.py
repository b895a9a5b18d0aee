"""SURVEY §8(f) row 5 — the moving volume resampled into the fixed frame (reference _dock_widget.py:1095-1130,
`_export_transformed_image`).  Contract: scipy.ndimage.affine_transform(src, M[:3, :3], offset=M[:3, 3], output_shape,
order, mode='constant', cval).  Order 0 is bit-identical for every dtype; order 1 is within 1 ulp for float32 and
identical for integers except +-1 where scipy's float64 value lies within 1e-9 of a .5 rounding boundary."""
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

pytestmark = pytest.mark.gpu


def _scipy(src, M, shape, order, cval):
    import scipy.ndimage as nd
    return nd.affine_transform(src, M[:3, :3], offset=M[:3, 3], output_shape=shape, order=order, mode="constant",
                               cval=cval)


def _to_device(a):
    import torch
    if a.dtype == np.uint16:
        return torch.from_numpy(np.ascontiguousarray(a).view(np.int16)).cuda().view(torch.uint16)
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _to_host(t):
    import torch
    if t.dtype == torch.uint16:
        return t.view(torch.int16).cpu().numpy().view(np.uint16)
    return t.cpu().numpy()


def _gpu(src, M, shape, order, cval):
    import torch
    from platymatch_b200 import device as D
    out = D.resample_affine(_to_device(src), torch.from_numpy(np.ascontiguousarray(M, dtype=np.float64)).cuda(), shape,
                            order, cval)
    return _to_host(out)


def _rotation(angles):
    a, b, c = angles
    rx = np.array([[1, 0, 0], [0, np.cos(a), -np.sin(a)], [0, np.sin(a), np.cos(a)]])
    ry = np.array([[np.cos(b), 0, np.sin(b)], [0, 1, 0], [-np.sin(b), 0, np.cos(b)]])
    rz = np.array([[np.cos(c), -np.sin(c), 0], [np.sin(c), np.cos(c), 0], [0, 0, 1]])
    return rx @ ry @ rz


def _affine(lin, off):
    M = np.eye(4)
    M[:3, :3], M[:3, 3] = lin, off
    return M


def _cases():
    rng = np.random.default_rng(5)
    near = _affine(_rotation(rng.uniform(-0.25, 0.25, 3)) * rng.uniform(0.9, 1.1, 3) + rng.normal(0, 0.02, (3, 3)),
                   rng.uniform(-4, 4, 3))
    perm = np.zeros((3, 3))
    perm[0, 2] = perm[1, 0] = perm[2, 1] = 1                  # source (z, y, x) = output (x, z, y)
    rot90 = _affine(np.array([[1, 0, 0], [0, 0, 1], [0, -1, 0]]), [0, 0, 9])       # source (z, x, 9 - y)
    nan = np.full((4, 4), np.nan)
    nan[3] = [0, 0, 0, 1]
    return [  # id, source shape, output shape, M, cval
        ("identity", (13, 17, 21), (13, 17, 21), np.eye(4), 0.0),
        ("int_shift_larger_out", (9, 33, 35), (11, 30, 37), _affine(np.eye(3), [2, -3, 5]), 0.0),
        ("half_voxel_shift", (7, 10, 19), (7, 10, 19), _affine(np.eye(3), [0.5, -0.5, 1.5]), 0.0),
        ("half_voxel_grid", (6, 9, 13), (11, 17, 25), _affine(np.eye(3) * 0.5, [0.25, 0, -0.5]), 0.0),
        ("permutation", (5, 7, 9), (7, 9, 5), _affine(perm, [0, 0, 0]), 0.0),
        ("rot90_yx", (6, 14, 10), (6, 10, 14), rot90, 0.0),
        ("scale2_axis_len1", (1, 9, 11), (3, 18, 22), _affine(np.eye(3) * 0.5, [0, 0, 0]), 0.0),
        ("scale_half_smaller_out", (20, 31, 45), (10, 16, 23), _affine(np.eye(3) * 2.0, [0, 0, 0]), 0.0),
        ("near_rigid", (37, 41, 43), (40, 39, 50), near, 0.0),
        ("near_rigid_x_len1", (15, 12, 1), (17, 13, 3), _affine(_rotation([0.2, 0, 0]), [0.3, -1, 0]), 0.0),
        ("all_outside", (8, 9, 10), (5, 6, 7), _affine(np.eye(3), [1000, 0, 0]), 3.0),
        ("nan_matrix", (8, 9, 10), (5, 6, 7), nan, 2.0),
        ("negative_cval", (37, 41, 43), (40, 39, 50), near, -7.5),
    ]


CASES = _cases()


def _source(shape, dtype, seed):
    rng = np.random.default_rng(seed)
    if dtype == np.uint16:
        return rng.integers(0, 65536, size=shape).astype(np.uint16)
    if dtype == np.int32:
        return rng.integers(-100000, 100000, size=shape).astype(np.int32)
    return rng.uniform(-50.0, 50.0, size=shape).astype(np.float32)


def _assert_matches(out, src, M, shape, order, cval):
    ref = _scipy(src, M, shape, order, cval)
    assert out.dtype == ref.dtype and out.shape == ref.shape
    if order == 0:
        assert np.array_equal(out.view(np.uint8), ref.view(np.uint8))          # bit-identical
        return 0
    if out.dtype == np.float32:
        assert np.all(np.abs(out.astype(np.float64) - ref) <= np.spacing(np.abs(ref)).astype(np.float64))
        return 0
    # integers: differences only where scipy's float64 value sits within 1e-9 of a .5 boundary, and only by 1
    exact = _scipy(src.astype(np.float64), M, shape, order, cval)
    tie = np.abs(np.abs(exact - np.trunc(exact)) - 0.5) < 1e-9
    diff = out.astype(np.int64) - ref.astype(np.int64)
    assert np.all(np.abs(diff) <= 1)
    assert not np.any(diff[~tie]), int(np.count_nonzero(diff[~tie]))
    return int(np.count_nonzero(diff))


@pytest.mark.parametrize("order", [0, 1])
@pytest.mark.parametrize("dtype", [np.int32, np.uint16, np.float32], ids=["int32", "uint16", "float32"])
@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_resample_matches_scipy(case, dtype, order):
    name, sshape, oshape, M, cval = case
    src = _source(sshape, dtype, seed=len(name))
    out = _gpu(src, M, oshape, order, cval)
    _assert_matches(out, src, M, oshape, order, cval)
    if name == "identity":
        assert np.array_equal(out, src)
    if name in ("all_outside", "nan_matrix"):
        assert np.all(out == np.asarray(cval).astype(dtype))


def test_resample_label_like_values_and_ties():
    """Integer order 1 on small values: many exact .5 results (weights 0.5 from the half-voxel shift), where the
    round-half-away-from-zero rule decides, for both signs."""
    rng = np.random.default_rng(2)
    M = _affine(np.eye(3), [0.5, 0.5, 0.5])
    for dtype, lo in ((np.int32, -9), (np.uint16, 0)):
        src = rng.integers(lo, 10, size=(12, 13, 14)).astype(dtype)
        out = _gpu(src, M, (12, 13, 14), 1, 0.0)
        _assert_matches(out, src, M, (12, 13, 14), 1, 0.0)
    tiny = np.array([[[-5, 4]]], dtype=np.int32)
    assert _gpu(tiny, _affine(np.eye(3), [0, 0, 0.5]), (1, 1, 1), 1, 0.0)[0, 0, 0] == -1
    assert _gpu(tiny, _affine(np.eye(3), [0, 0, 0.25]), (1, 1, 1), 1, 0.0)[0, 0, 0] == -3
    assert _gpu(np.array([[[0, 10]]], dtype=np.uint16), _affine(np.eye(3), [0, 0, 0.25]), (1, 1, 1), 1, 0.0)[0, 0, 0] == 3


def test_resample_boundaries():
    """-1e-9 is outside, n - 1 is inside (and reads the last voxel with order 1), n - 1 + 1e-7 is outside."""
    src = np.arange(1, 6, dtype=np.float32).reshape(1, 1, 5)
    for off, want in ((-1e-9, -1.0), (0.0, 1.0), (4.0, 5.0), (4.0000001, -1.0)):
        M = _affine(np.eye(3), [0, 0, off])
        for order in (0, 1):
            assert _gpu(src, M, (1, 1, 1), order, -1.0)[0, 0, 0] == want, (off, order)


def test_resample_unaligned_and_out_buffer():
    """Views whose rows start off a 16-byte boundary take the scalar store path; `out` is written in place."""
    import torch
    from platymatch_b200 import device as D
    src = _source((9, 10, 23), np.int32, seed=4)
    M = _affine(_rotation([0.1, -0.05, 0.2]), [1.0, -2.0, 0.5])
    ref = _scipy(src, M, (7, 11, 21), 0, 0.0)
    big = torch.zeros(7 * 11 * 21 + 1, dtype=torch.int32, device="cuda")
    out = big[1:].view(7, 11, 21)
    res = D.resample_affine(_to_device(src), torch.from_numpy(M).cuda(), (7, 11, 21), 0, 0.0, out=out)
    assert res.data_ptr() == out.data_ptr()
    assert np.array_equal(out.cpu().numpy(), ref) and int(big[0]) == 0


def test_resample_beyond_2_31_voxels():
    """An int32 source of 2048 x 1024 x 1040 = 2.18e9 voxels (8.7 GB), built on the device from its linear index,
    resampled (order 0) into a small grid that spans it; 1e5 output voxels checked against the index pattern."""
    import torch
    from platymatch_b200 import device as D
    P = 2147483629                                        # (prime: a 32-bit wrapped offset gives a different value)
    sshape = (2048, 1024, 1040)
    plane = sshape[1] * sshape[2]
    lin = torch.arange(plane, dtype=torch.int64, device="cuda")
    src = torch.empty(sshape, dtype=torch.int32, device="cuda")
    for z in range(sshape[0]):
        src[z] = torch.remainder(lin + z * plane, P).to(torch.int32).view(sshape[1], sshape[2])
    del lin
    oshape = (128, 64, 65)
    lin3 = _rotation([0.01, -0.008, 0.012]) @ np.diag([2047 / 128, 1023 / 64, 1039 / 65])
    M = _affine(lin3, [3.0, 2.5, 1.0])
    out = _to_host(D.resample_affine(src, torch.from_numpy(M).cuda(), oshape, 0, -1.0))
    del src
    torch.cuda.empty_cache()
    rng = np.random.default_rng(0)
    flat = rng.choice(out.size, 100000, replace=False)
    z, y, x = (a.astype(np.float64) for a in np.unravel_index(flat, oshape))
    c = [((z * M[h, 0] + y * M[h, 1]) + x * M[h, 2]) + M[h, 3] for h in range(3)]
    inside = np.ones(flat.size, dtype=bool)
    for h in range(3):
        inside &= (c[h] >= 0) & (c[h] <= sshape[h] - 1)
    idx = [np.floor(c[h] + 0.5).astype(np.int64) for h in range(3)]
    lin_src = (idx[0] * sshape[1] + idx[1]) * sshape[2] + idx[2]
    want = np.where(inside, lin_src % P, -1)
    assert inside.mean() > 0.9 and lin_src[inside].max() >= 2 ** 31
    assert np.array_equal(out.reshape(-1)[flat], want)


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


def _overlap(warped, fixed_vol, n):
    a, b = warped > 0, fixed_vol > 0
    dice = 2.0 * np.count_nonzero(a & b) / (np.count_nonzero(a) + np.count_nonzero(b))
    same = 0
    for k in range(1, n + 1):                     # the majority fixed label (background included) under nucleus k
        f = fixed_vol[warped == k]
        if f.size:
            v, cnt = np.unique(f, return_counts=True)
            same += int(v[np.argmax(cnt)] == k)
    return dice, same


def test_registration_then_warp_labels():
    """Register two label volumes, then warp the moving one into the fixed grid: bit-identical to scipy with the same
    recovered transform, and it overlays the fixed volume (with the true transform: Dice 0.788, 362 of 400)."""
    import platymatch_b200 as pm
    from platymatch_b200.utils.images import transform_image
    from platymatch_b200.utils.labels import detections_from_labels, ransac_error_from_sizes
    n, shape, fixed_vol, moving_vol = _registration_setup()
    fd, fs, _ = detections_from_labels(fixed_vol, 1.0)
    md, ms, _ = detections_from_labels(moving_vol, 1.0)
    res = pm.estimate_transform_unsupervised(md, fd, ransac_trials=4000, ransac_error=ransac_error_from_sizes(ms, fs),
                                             seed=2)
    T = res["transform"]
    warped = transform_image(moving_vol, T, shape, order=0)
    assert warped.dtype == np.uint16
    M = np.linalg.inv(T)
    assert np.array_equal(warped, _scipy(moving_vol, M, shape, 0, 0))
    dice, same = _overlap(warped, fixed_vol, n)
    dice0, _ = _overlap(moving_vol, fixed_vol, n)
    print("recovered transform: Dice %.4f, %d of %d nuclei on their fixed label (identity: Dice %.4f)" %
          (dice, same, n, dice0))
    assert dice >= 0.7 and same >= 340, (dice, same, T)
    assert dice0 < 0.1


def test_transform_image_dtypes():
    """uint16 / int32 / float32 straight through; other integer dtypes through int32 and back in their own dtype."""
    from platymatch_b200.utils.images import transform_image
    rng = np.random.default_rng(6)
    T = _affine(_rotation([0.1, 0.05, -0.1]) * 1.02, [1.5, -0.5, 2.0])
    M = np.linalg.inv(T)
    for dtype in (np.uint8, np.int8, np.int16, np.uint32, np.int64, np.uint16, np.int32, np.float32):
        if np.issubdtype(dtype, np.integer):
            info = np.iinfo(dtype)
            src = rng.integers(max(info.min, -1000), min(info.max, 1000) + 1, size=(11, 12, 13)).astype(dtype)
        else:
            src = rng.normal(size=(11, 12, 13)).astype(dtype)
        for order in (0, 1):
            out = transform_image(src, T, (10, 13, 12), order=order)
            assert out.dtype == src.dtype
            if dtype in (np.uint16, np.int32, np.float32):
                _assert_matches(out, src, M, (10, 13, 12), order, 0)
            else:
                _assert_matches(out.astype(np.int32), src.astype(np.int32), M, (10, 13, 12), order, 0)


def test_resample_on_side_stream_after_registration():
    """A resample enqueued on a side stream after the registration's last kernel, with no host synchronisation in
    between, gives the same bytes as on the default stream."""
    import torch
    from platymatch_b200 import device as D
    from platymatch_b200.pipeline import describe_pair, register_described
    from platymatch_b200.synthetic import make_pair
    pair = make_pair(600, seed=11)
    vol = _source((64, 80, 96), np.float32, seed=9)
    dev_vol = _to_device(vol)
    centre = torch.tensor([31.5, 39.5, 47.5], dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        dm, df = describe_pair(pair["moving"], pair["fixed"], 1, 4)
        res = register_described(dm, df, ransac_trials=500, seed=3)
        # the registration's linear part about the volume centre, built on the device from its last kernel's output
        m = res["transform"].view(4, 4).clone()
        m[:3, 3] = centre - m[:3, :3] @ centre
        out = D.resample_affine(dev_vol, m, (70, 75, 90), 1, -1.0)
    side.synchronize()
    got = _to_host(out)
    ref = _to_host(D.resample_affine(dev_vol, m, (70, 75, 90), 1, -1.0))
    assert np.array_equal(got.view(np.uint32), ref.view(np.uint32))
    assert np.count_nonzero(ref != -1.0) > ref.size // 3           # (0.68 of the grid maps inside with A_gt)


def test_resample_refuses_host_tensors():
    """A host src or out, or an out on another device, is refused before any pointer reaches the kernel."""
    import torch
    from platymatch_b200 import device as D
    src = torch.zeros((4, 5, 6), dtype=torch.int32)
    M = torch.eye(4, dtype=torch.float64, device="cuda")
    with pytest.raises(ValueError):
        D.resample_affine(src, M, (4, 5, 6))
    with pytest.raises(ValueError):
        D.resample_affine(src.cuda(), M, (4, 5, 6), out=torch.zeros((4, 5, 6), dtype=torch.int32))
