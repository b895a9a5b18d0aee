"""Nuclei detection (SURVEY §2 row 10, reference platymatch/detect_nuclei/ss_log.py): the host-side pieces of the
contract and the argument checks, without a GPU."""
import math
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import detect_oracle as DO  # noqa: E402


def _pass(a, w_half, axis):
    """One pass as pm_detect_pass computes it: reflect, centre first, tap pairs outermost first, float64 -> float32."""
    lw = w_half.size - 1
    b = np.moveaxis(np.asarray(a, dtype=np.float32), axis, -1).astype(np.float64)
    p = np.pad(b, [(0, 0)] * (b.ndim - 1) + [(lw, lw)], mode="symmetric")
    n = b.shape[-1]
    acc = p[..., lw:lw + n] * w_half[0]
    for j in range(lw, 0, -1):
        acc = acc + (p[..., lw - j:lw - j + n] + p[..., lw + j:lw + j + n]) * w_half[j]
    return np.ascontiguousarray(np.moveaxis(acc.astype(np.float32), -1, axis))


def _log8(img, sig):
    from platymatch_b200.detect_nuclei.ss_log import log_weights
    w = [[log_weights(s, 0), log_weights(s, 2)] for s in sig]
    gz = _pass(img, w[0][0], 0)
    t0 = _pass(_pass(_pass(img, w[0][1], 0), w[1][0], 1), w[2][0], 2)
    t1 = _pass(_pass(gz, w[1][1], 1), w[2][0], 2)
    t2 = _pass(_pass(gz, w[1][0], 1), w[2][1], 2)
    return (t0 + t1) + t2


def test_weights_bit_equal_scipy():
    from scipy.ndimage._filters import _gaussian_kernel1d
    from platymatch_b200.detect_nuclei.ss_log import gaussian_kernel1d, log_weights
    for sigma in np.concatenate([np.linspace(0.1, 12.0, 97), [1 / math.sqrt(3), 8 / math.sqrt(3) / 2.0]]):
        for order in (0, 2):
            lw = int(4.0 * sigma + 0.5)
            ref = _gaussian_kernel1d(sigma, order, lw)
            assert np.array_equal(gaussian_kernel1d(sigma, order, lw), ref)
            assert np.array_equal(log_weights(sigma, order), ref[::-1][lw:])


@pytest.mark.parametrize("shape", [(20, 23, 41), (3, 30, 17), (1, 25, 25), (7, 1, 9)])
def test_eight_pass_schedule_bit_equal_gaussian_laplace(shape):
    import scipy.ndimage as nd
    img = (np.random.default_rng(sum(shape)).random(shape) * 1000).astype(np.float32)
    for sig in [(1.0, 2.0, 2.0), (3.7, 3.7, 3.7), (0.8, 2.5, 2.5), (4.6, 4.6, 4.6)]:
        ref = nd.gaussian_laplace(img, sig)
        assert np.array_equal(_log8(img, sig).view(np.uint32), ref.view(np.uint32)), sig


def test_single_pass_bit_equal_gaussian_filter1d():
    import scipy.ndimage as nd
    from platymatch_b200.detect_nuclei.ss_log import log_weights
    img = (np.random.default_rng(4).normal(size=(5, 13, 40)) * 50).astype(np.float32)
    for sigma in (0.5, 1.3, 2.9, 6.0):
        for order in (0, 2):
            for axis in range(3):
                ref = nd.gaussian_filter1d(img, sigma, axis=axis, order=order)
                assert np.array_equal(_pass(img, log_weights(sigma, order), axis), ref)


def test_restated_histogram_equals_numpy():
    rng = np.random.default_rng(7)
    cases = [rng.normal(size=5000).astype(np.float32),
             (rng.integers(0, 257, size=4000) * np.float32(0.37)).astype(np.float32),     # many values on edges
             np.array([0.0, 1.0, 1.0, 1.0], dtype=np.float32),                              # the max value repeated
             np.array([-3.0, 1e-7, 2e7], dtype=np.float32),
             rng.uniform(1000.0, 1000.1, size=3000).astype(np.float32)]                      # edges a few ulp apart
    lo, hi = np.float32(-1.5), np.float32(2.25)
    edges = np.linspace(lo, hi, 257, dtype=np.float32)
    cases.append(np.concatenate([edges, edges, [hi, hi]]).astype(np.float32))               # every edge exactly
    for a in cases:
        c, e = DO.otsu_histogram(a)
        rc, re = np.histogram(a, 256, range=(a.min(), a.max()))
        assert re.dtype == np.float32 and np.array_equal(e, re) and np.array_equal(c, rc)


def test_otsu_known_answers():
    assert DO.otsu(np.full((2, 3, 4), 7.25, dtype=np.float32)) == 7.25
    two = np.concatenate([np.zeros(100), np.full(100, 10.0)]).astype(np.float32)
    t = DO.otsu(two)
    assert 0.0 < t < 10.0
    assert t == 10.0 / 256 / 2                   # the centre of the first bin: the first maximum wins
    rng = np.random.default_rng(1)
    bimodal = np.concatenate([rng.normal(20, 2, 4000), rng.normal(80, 2, 4000)]).astype(np.float32)
    t = DO.otsu(bimodal)                          # every threshold in the gap is a maximum: the first one wins
    assert bimodal[bimodal < 50].max() - 0.25 < t < 50


def test_sphere_intersection_identities():
    from platymatch_b200.detect_nuclei.ss_log import sphere_intersection as si
    vol = lambda r: 4.0 / 3.0 * math.pi * r * r * r
    assert si((0, 0, 0), 2, (0, 0, 5), 3) == 0.0                 # touching
    assert si((0, 0, 0), 2, (9, 0, 0), 3) == 0.0
    assert si((0, 0, 0), 2, (0, 1, 0), 3) == vol(2)               # contained
    assert si((1, 2, 3), 4, (1, 2, 3), 4) == vol(4)               # identical
    rng = np.random.default_rng(0)
    for _ in range(50):
        c1, c2 = rng.uniform(-3, 3, 3), rng.uniform(-3, 3, 3)
        r1, r2 = rng.uniform(1, 4, 2)
        assert si(c1, r1, c2, r2) == si(c2, r2, c1, r1)
    # numeric integration of a lens
    c1, r1, c2, r2 = np.zeros(3), 3.0, np.array([0.0, 1.5, 2.0]), 2.0
    g = np.linspace(-3.5, 3.5, 281)
    h = g[1] - g[0]
    Z, Y, X = np.meshgrid(g, g, g, indexing="ij", sparse=True)
    inside = ((Z ** 2 + Y ** 2 + X ** 2) <= r1 ** 2) & (((Z - c2[0]) ** 2 + (Y - c2[1]) ** 2 + (X - c2[2]) ** 2) <= r2 ** 2)
    assert abs(inside.sum() * h ** 3 - si(c1, r1, c2, r2)) < 0.02 * si(c1, r1, c2, r2)


def test_oracle_suppression_chains():
    # unit spheres 1.2 apart in a row: each overlaps its neighbours by more than half, so keep / drop alternates
    n = 9
    c = np.stack([np.zeros(n), np.zeros(n), 1.2 * np.arange(n)], axis=1)
    assert DO.suppress_spheres(c, np.ones(n), 0.1).tolist() == [i % 2 == 0 for i in range(n)]
    # reversed priority: the same alternation counted from the other end
    assert DO.suppress_spheres(c[::-1], np.ones(n), 0.1).tolist() == [i % 2 == 0 for i in range(n)]
    # overlap = 1 keeps everything, overlap = 0 keeps only non-touching spheres
    assert DO.suppress_spheres(c, np.ones(n), 1.0).all()
    c2 = np.stack([np.zeros(4), np.zeros(4), np.array([0.0, 2.0, 3.9, 10.0])], axis=1)
    assert DO.suppress_spheres(c2, np.ones(4), 0.0).tolist() == [True, True, False, True]


@pytest.mark.parametrize("kw", [
    dict(image=np.zeros((4, 5, 6), dtype=np.bool_)),
    dict(image=np.zeros((4, 5, 6), dtype=np.complex64)),
    dict(image=np.zeros((5, 6), dtype=np.float32)),
    dict(image=np.zeros((2, 4, 5, 6), dtype=np.float32)),
    dict(image=np.zeros((0, 5, 6), dtype=np.float32)),
    dict(radii=[]),
    dict(radii=[3, 2]),
    dict(radii=[2, 2]),
    dict(radii=[0, 2]),
    dict(radii=[-1.0]),
    dict(radii=[2000.0]),
    dict(anisotropy=0.0),
    dict(anisotropy=-1.0),
    dict(overlap=-0.1),
    dict(overlap=1.5),
])
def test_find_spheres_refuses_before_device(kw, monkeypatch):
    from platymatch_b200 import device as D
    from platymatch_b200.detect_nuclei import find_spheres

    def no_device():
        raise AssertionError("the device was touched")
    monkeypatch.setattr(D, "_torch", no_device)
    args = dict(image=np.zeros((4, 5, 6), dtype=np.float32), radii=[2.0, 3.0])
    args.update(kw)
    with pytest.raises(ValueError):
        find_spheres(args.pop("image"), args.pop("radii"), **args)


def test_detect_entry_points_refuse_on_host():
    import ctypes
    from platymatch_b200 import _lib
    lib = _lib.load()
    p, q = ctypes.c_void_p(1 << 12), ctypes.c_void_p(1 << 30)
    assert lib.pm_detect_pass(None, 2, 3, 4, 0, p, 1, None, None, 1.0, q, None) == -1
    assert lib.pm_detect_pass(p, 2, 3, 4, 3, p, 1, None, None, 1.0, q, None) == -1
    assert b"axis" in lib.pm_last_error_string()
    assert lib.pm_detect_pass(p, 2, 0, 4, 0, p, 1, None, None, 1.0, q, None) == -1
    assert lib.pm_detect_pass(p, 2, 3, 4, 0, p, 385, None, None, 1.0, q, None) == -1
    assert lib.pm_detect_pass(p, 2, 3, 4, 0, p, 1, p, None, 1.0, q, None) == -1
    assert lib.pm_detect_pass(p, 2, 3, 4, 0, p, 1, None, None, 1.0, ctypes.c_void_p((1 << 12) + 8), None) == -1
    assert b"overlap" in lib.pm_last_error_string()
    assert lib.pm_detect_otsu(p, 0, 0.2, q, p, 1 << 20, None) == -1
    assert lib.pm_detect_otsu(p, 10, 0.2, q, p, 8, None) == -3
    assert lib.pm_detect_minima(p, None, None, 2, 3, 4, 0, p, 10, p, p, p, None) == -1
    assert lib.pm_detect_minima(None, p, None, 2, 3, 4, -1, p, 10, p, p, p, None) == -1
    assert lib.pm_detect_suppress_workspace_bytes(100, 10, 10, 10, 2.0, 1.0) >= 2 * 100 * 4
    for args in ((p, p, 0, 4, 4, 4, p, 2.0, 1.0, 0.5), (p, p, 10, 4, 4, 4, p, 0.0, 1.0, 0.5),
                 (p, p, 10, 4, 4, 4, p, 2.0, 0.0, 0.5), (p, p, 10, 4, 4, 4, p, 2.0, 1.0, 1.5)):
        assert lib.pm_detect_suppress(*args, p, p, 1 << 30, None) == -1
    assert lib.pm_detect_suppress(p, p, 10, 4, 4, 4, p, 2.0, 1.0, 0.5, p, p, 4, None) == -3
