"""DESIGN §8 row 8 — the thin-plate spline deformation: argument checks that run on the host before any CUDA call or
device transfer, scipy's polynomial domain, and the numpy restatement of the sampler the GPU tests compare against
(no GPU needed)."""
import ctypes
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from spline_oracle import sample_order0, sample_order1  # noqa: E402


def _lib():
    from platymatch_b200 import _lib
    return _lib.load()


# 16-byte-aligned stand-ins for device buffers; never dereferenced, because every call below is refused first
A, B, C, E, F = (ctypes.c_void_p(v) for v in (1 << 12, 1 << 20, 1 << 24, 1 << 28, 1 << 32))


def test_spline_system_refusals():
    lib = _lib()

    def call(y=A, k=10, ss=B, lam=0.0, lhs=C, ld=14):
        return lib.pm_spline_system(y, k, ss, lam, lhs, ld, None)

    for kw in ({"y": None}, {"ss": None}, {"lhs": None}):
        assert call(**kw) == -1 and b"null pointer" in lib.pm_last_error_string()
    assert call(k=0) == -1 and b"k must be" in lib.pm_last_error_string()
    assert call(k=-3) == -1
    assert call(ld=13) == -1 and b"ld" in lib.pm_last_error_string()
    for lam in (-1.0, float("nan"), float("inf")):
        assert call(lam=lam) == -1 and b"smoothing" in lib.pm_last_error_string()
    assert call(lhs=ctypes.c_void_p((1 << 12) + 64)) == -1 and b"overlap" in lib.pm_last_error_string()


def test_spline_eval_refusals():
    lib = _lib()

    def call(y=A, c=B, k=10, ss=C, pts=E, n=100, out=F):
        return lib.pm_spline_eval(y, c, k, ss, pts, n, out, None)

    for kw in ({"y": None}, {"c": None}, {"ss": None}, {"pts": None}, {"out": None}):
        assert call(**kw) == -1 and b"null pointer" in lib.pm_last_error_string()
    assert call(k=0) == -1 and b"k must be" in lib.pm_last_error_string()
    assert call(n=0) == -1 and b"n must be" in lib.pm_last_error_string()
    assert call(out=ctypes.c_void_p((1 << 28) + 8 * 3 * 99)) == -1 and b"overlap" in lib.pm_last_error_string()
    assert call(out=ctypes.c_void_p((1 << 20) + 8 * 3 * 13)) == -1           # the last coefficient row
    assert call(out=ctypes.c_void_p((1 << 24) + 40)) == -1                   # the last scale


def test_resample_spline_refusals():
    lib = _lib()

    def call(src=A, dtype=0, s=(4, 5, 6), y=B, c=C, k=10, ss=E, order=0, dst=F, d=(3, 4, 5)):
        return lib.pm_resample_spline(src, dtype, *s, y, c, k, ss, order, 0.0, dst, *d, None)

    for kw in ({"src": None}, {"y": None}, {"c": None}, {"ss": None}, {"dst": None}):
        assert call(**kw) == -1 and b"null pointer" in lib.pm_last_error_string()
    assert call(dtype=3) == -1 and b"dtype" in lib.pm_last_error_string()
    assert call(order=2) == -1 and b"order" in lib.pm_last_error_string()
    assert call(order=-1) == -1
    assert call(k=0) == -1 and b"k must be" in lib.pm_last_error_string()
    for s, d in (((0, 5, 6), (3, 4, 5)), ((4, 5, 6), (3, 0, 5)), ((4, -5, 6), (3, 4, 5)), ((4, 5, 6), (3, 4, -1))):
        assert call(s=s, d=d) == -1 and b"extent" in lib.pm_last_error_string()
    assert call(dst=ctypes.c_void_p((1 << 12) + 16)) == -1 and b"overlap" in lib.pm_last_error_string()
    assert call(dst=ctypes.c_void_p((1 << 12) + 4 * 4 * 5 * 6 - 4)) == -1                      # last int32 of src
    assert call(dtype=1, dst=ctypes.c_void_p((1 << 12) + 2 * 4 * 5 * 6 - 2)) == -1             # last uint16 of src
    assert call(dst=ctypes.c_void_p((1 << 20) + 8)) == -1 and b"spline" in lib.pm_last_error_string()


def _no_device(monkeypatch):
    from platymatch_b200 import device as D

    def no_device():
        raise AssertionError("the device was touched")
    monkeypatch.setattr(D, "_torch", no_device)


def test_fit_spline_refusals_before_device(monkeypatch):
    from platymatch_b200.estimate_transform.deformable import fit_spline
    _no_device(monkeypatch)
    rng = np.random.default_rng(0)
    y = rng.normal(size=(3, 20)) * 10
    d = rng.normal(size=(3, 20))
    cases = [
        ((y[:2], d[:2]), {}, "3 x N"),                                # not 3 x K
        ((y, d[:, :19]), {}, "differ in size"),
        ((y[:, :3], d[:, :3]), {}, "at least 4"),
        ((np.where(np.arange(20) == 5, np.nan, y), d), {}, "finite"),
        ((y, np.where(np.arange(20) == 7, np.inf, d)), {}, "finite"),
        ((y, d), {"smoothing": -1.0}, "smoothing"),
        ((y, d), {"smoothing": float("nan")}, "smoothing"),
    ]
    flat = y.copy()
    flat[2] = 0.25 * flat[0] - 2.0 * flat[1] + 3.0                    # coplanar: rank 3
    cases.append(((flat, d), {}, "rank 3"))
    line = np.outer([1.0, 2.0, -1.0], np.arange(20.0))                # collinear: rank 2
    cases.append(((line, d), {}, "rank 2"))
    dup = y.copy()
    dup[:, 11] = dup[:, 3]
    cases.append(((dup, d), {"smoothing": 0.0}, "equal"))
    for args, kw, msg in cases:
        with pytest.raises(ValueError, match=msg):
            fit_spline(*args, **kw)
    big = rng.normal(size=(3, 16385))
    with pytest.raises(ValueError, match="16384"):
        fit_spline(big, big)


def test_duplicates_with_smoothing_pass_the_host_checks(monkeypatch):
    """Equal source points are fine once smoothing > 0 (scipy solves that system too): the call reaches the device."""
    from platymatch_b200.estimate_transform.deformable import fit_spline
    _no_device(monkeypatch)
    rng = np.random.default_rng(1)
    y = rng.normal(size=(3, 20)) * 10
    y[:, 11] = y[:, 3]
    with pytest.raises(AssertionError, match="device was touched"):
        fit_spline(y, y, smoothing=1.0)


def test_deformation_entry_points_refuse_before_device(monkeypatch):
    from platymatch_b200.estimate_transform.deformable import match_nuclei
    from platymatch_b200.utils.images import transform_image_deformable
    _no_device(monkeypatch)
    pts = np.zeros((3, 5))
    with pytest.raises(ValueError):
        match_nuclei(pts, pts, np.eye(3))
    with pytest.raises(ValueError):
        match_nuclei(pts, pts, np.eye(4), max_distance=-1.0)
    with pytest.raises(ValueError):
        match_nuclei(pts[:2], pts, np.eye(4))
    vol = np.zeros((2, 3, 4), dtype=np.int32)
    for args, kw in (((vol[0], {}, (2, 3, 4)), {}), ((vol, {}, (2, 0, 4)), {}), ((vol, {}, (2, 3)), {}),
                     ((vol, {}, (2, 3, 4)), {"order": 2}), ((vol.astype(np.float64), {}, (2, 3, 4)), {}),
                     ((np.full((2, 3, 4), 2 ** 40, dtype=np.int64), {}, (2, 3, 4)), {}),
                     ((vol, {"forward": None}, (2, 3, 4)), {})):
        with pytest.raises((ValueError, KeyError)):
            transform_image_deformable(*args, **kw)


@pytest.mark.parametrize("seed", range(3))
def test_shift_scale_equal_scipy(seed):
    from scipy.interpolate import RBFInterpolator
    from platymatch_b200.estimate_transform.deformable import shift_scale
    rng = np.random.default_rng(seed)
    y = rng.normal(size=(40, 3)) * rng.uniform(1, 300, 3) + rng.uniform(-500, 500, 3)
    ref = RBFInterpolator(y, np.zeros((40, 1)), kernel="linear", degree=1)
    shift, scale = shift_scale(y)
    assert np.array_equal(shift, ref._shift) and np.array_equal(scale, ref._scale)


def test_shift_scale_flat_axis():
    """scipy replaces a zero scale by 1 (such a set is then refused for its rank, by scipy and by fit_spline)."""
    from platymatch_b200.estimate_transform.deformable import shift_scale
    y = np.c_[np.arange(5.0), np.full(5, 7.25), np.arange(5.0) ** 2]
    shift, scale = shift_scale(y)
    assert scale[1] == 1.0 and shift[1] == 7.25 and scale[0] == 2.0 and shift[2] == 8.0


@pytest.mark.parametrize("order", [0, 1])
@pytest.mark.parametrize("dtype", [np.int32, np.uint16, np.float32], ids=["int32", "uint16", "float32"])
def test_sampler_restatement_equals_map_coordinates(dtype, order):
    """The numpy sampler (tests/spline_oracle.py) equals scipy.ndimage.map_coordinates(order, mode='constant') on random
    coordinates away from rounding and domain boundaries, and gives cval outside and for NaN."""
    import scipy.ndimage as nd
    rng = np.random.default_rng(order * 7 + np.dtype(dtype).itemsize)
    shape = (9, 11, 14)
    if dtype == np.float32:
        src = rng.uniform(-50, 50, size=shape).astype(dtype)
    else:
        src = rng.integers(0 if dtype == np.uint16 else -1000, 1000, size=shape).astype(dtype)
    c = rng.uniform(-1.5, np.array(shape)[:, None] + 0.5, size=(3, 20000))
    frac = c - np.floor(c)
    away = np.all(np.abs(frac - 0.5) > 1e-6, axis=0) & np.all((np.abs(c) > 1e-6) &
                                                              (np.abs(c - (np.array(shape)[:, None] - 1)) > 1e-6), axis=0)
    c = c[:, away]
    c[:, :5] = np.nan
    cval = 3.0
    got = (sample_order0 if order == 0 else sample_order1)(src, c, cval)
    ref = nd.map_coordinates(src, c, order=order, mode="constant", cval=cval)
    assert got.dtype == src.dtype
    if order == 0 or dtype == np.float32:
        if dtype == np.float32 and order == 1:
            assert np.all(np.abs(got.astype(np.float64) - ref) <= np.spacing(np.abs(ref)))
        else:
            assert np.array_equal(got, ref)
    else:
        exact = nd.map_coordinates(src.astype(np.float64), c, order=1, mode="constant", cval=cval)
        tie = np.abs(np.abs(exact - np.trunc(exact)) - 0.5) < 1e-9
        diff = got.astype(np.int64) - ref.astype(np.int64)
        assert not np.any(diff[~tie]) and np.all(np.abs(diff) <= 1)
    assert np.all(got[:5] == np.asarray(cval).astype(dtype))
