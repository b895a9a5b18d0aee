"""Nuclei detection on the GPU (SURVEY §2 row 10, reference platymatch/detect_nuclei/ss_log.py) against the project's
contract restated with scipy in tests/detect_oracle.py: passes and L_k bit-identical, Otsu, candidates and the greedy
keep-set equal, and the end-to-end image -> detections -> registration row."""
import math
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.dirname(os.path.abspath(__file__))]
import detect_oracle as DO  # noqa: E402

pytestmark = pytest.mark.gpu


def _dev(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _w(sigma, order):
    from platymatch_b200.detect_nuclei.ss_log import log_weights
    return _dev(log_weights(sigma, order))


PASS_SHAPES = [(5, 13, 40), (3, 30, 17), (1, 25, 25), (40, 1, 3), (33, 70, 129), (2, 3, 1)]


@pytest.mark.parametrize("shape", PASS_SHAPES, ids=["x".join(map(str, s)) for s in PASS_SHAPES])
def test_pass_bit_identical_to_gaussian_filter1d(shape):
    import scipy.ndimage as nd
    from platymatch_b200 import device as D
    img = (np.random.default_rng(sum(shape)).normal(size=shape) * 100).astype(np.float32)
    x = _dev(img)
    for sigma in (0.5, 1.3, 2.9, 4.62, 6.0):
        for order in (0, 2):
            for axis in range(3):
                out = D.detect_pass(x, axis, _w(sigma, order)).cpu().numpy()
                ref = nd.gaussian_filter1d(img, sigma, axis=axis, order=order)
                assert np.array_equal(out.view(np.uint32), ref.view(np.uint32)), (sigma, order, axis)


def _device_log(x, sigma_zyx, scale):
    from platymatch_b200 import device as D
    sz, sy, sx = sigma_zyx
    gz = D.detect_pass(x, 0, _w(sz, 0))
    acc = D.detect_pass(D.detect_pass(D.detect_pass(x, 0, _w(sz, 2)), 1, _w(sy, 0)), 2, _w(sx, 0))
    t1 = D.detect_pass(D.detect_pass(gz, 1, _w(sy, 2)), 2, _w(sx, 0))
    return D.detect_pass(D.detect_pass(gz, 1, _w(sy, 0)), 2, _w(sx, 2), t0=acc, t1=t1, scale=scale)


@pytest.mark.parametrize("anisotropy", [1.0, 2.0, 3.3])
def test_scale_space_bit_identical(anisotropy):
    img = (np.random.default_rng(3).random((24, 37, 50)) * 500).astype(np.float32)
    radii = [1.5, 3.0, 5.0, 8.0]
    ref = DO.scale_space_log(img, radii, anisotropy)
    for r, L in zip(radii, ref):
        s = r / math.sqrt(3.0)
        out = _device_log(_dev(img), (s / anisotropy, s, s), float(np.float32(s ** 2))).cpu().numpy()
        assert np.array_equal(out.view(np.uint32), L.view(np.uint32)), r


@pytest.mark.parametrize("kind", ["normal", "uniform_int", "constant", "zeros", "two_values", "nuclei"])
def test_otsu_equals_oracle(kind):
    from platymatch_b200 import device as D
    from platymatch_b200.synthetic import make_nuclei_image
    rng = np.random.default_rng(9)
    img = {"normal": lambda: rng.normal(size=(31, 40, 57)),
           "uniform_int": lambda: rng.integers(0, 256, size=(20, 30, 40)) * 0.37,
           "constant": lambda: np.full((5, 6, 7), 3.5),
           "zeros": lambda: np.zeros((5, 6, 7)),
           "two_values": lambda: np.where(rng.random((9, 9, 9)) < 0.3, -2.0, 7.0),
           "nuclei": lambda: make_nuclei_image((48, 64, 64), rng.uniform(4, 44, (40, 3)), 3.0, seed=2)}[kind]()
    img = np.asarray(img, dtype=np.float32)
    out = D.detect_otsu(_dev(img), 0.2).cpu().numpy()
    t = DO.otsu(img)
    assert out[0] == t and out[1] == 0.2 * t


def _device_candidates(L, threshold, cap=1 << 16):
    import torch
    from platymatch_b200 import device as D
    K = len(L)
    Ld = [_dev(a) for a in L]
    thr = torch.tensor([0.0, threshold], dtype=torch.float64, device="cuda")
    keys = torch.empty(cap, dtype=torch.int64, device="cuda")
    vals = torch.empty(cap, dtype=torch.float32, device="cuda")
    count = torch.zeros(1, dtype=torch.int64, device="cuda")
    for k in range(K):
        D.detect_minima(Ld[k - 1] if k else None, Ld[k], Ld[k + 1] if k + 1 < K else None, k, thr, keys, vals, count)
    n = int(count.item())
    assert n <= cap
    k, v = keys[:n].cpu().numpy(), vals[:n].cpu().numpy()
    o = np.argsort(k)
    return k[o], v[o]


def test_candidates_equal_oracle_with_ties():
    from platymatch_b200.synthetic import make_nuclei_image
    # blobs centred between voxels (exact ties along x, or x and y), plus a noisy field
    img = make_nuclei_image((30, 40, 44), [(10, 12, 10.5), (20, 27.5, 30.5), (15, 30, 12)], 4.0, noise=0.0)
    noisy = make_nuclei_image((30, 40, 44), np.random.default_rng(1).uniform(3, 27, (12, 3)), 3.0, noise=3.0, seed=4)
    for im in (img, noisy, np.round(noisy / 8) * 8):                 # the last one: plateaus and ties everywhere
        L = DO.scale_space_log(im, [2.0, 3.0, 4.0], 1.0)
        for t in (0.2 * DO.otsu(im), -1e30):
            keys, vals = _device_candidates(L, t, cap=1 << 20)
            rk, rv = DO.scale_space_minima(np.stack(L), t)
            assert np.array_equal(keys, rk) and np.array_equal(vals, rv)
    L = DO.scale_space_log(img, [2.0, 3.0, 4.0], 1.0)
    keys, _ = _device_candidates(L, 0.2 * DO.otsu(img))
    assert len(keys) == 3                                            # one candidate per tie group


@pytest.mark.parametrize("value", [0.0, 5.0])
def test_constant_image_has_no_candidates(value):
    from platymatch_b200.detect_nuclei import find_spheres
    det, r, resp = find_spheres(np.full((12, 13, 14), value, dtype=np.float32), [2.0, 3.0])
    assert det.shape == (3, 0) and r.size == 0 and resp.size == 0
    assert DO.find_spheres(np.full((12, 13, 14), value, dtype=np.float32), [2.0, 3.0])[0].shape == (3, 0)


def _device_keep(keys, shape, radii, anisotropy, overlap):
    import torch
    from platymatch_b200 import device as D
    cap = len(keys) + 5
    k = torch.full((cap,), np.iinfo(np.int64).max, dtype=torch.int64, device="cuda")
    k[:len(keys)] = _dev(np.asarray(keys, dtype=np.int64))
    count = torch.tensor([len(keys)], dtype=torch.int64, device="cuda")
    st = D.detect_suppress(k, count, shape, _dev(np.asarray(radii, dtype=np.float64)), max(radii), anisotropy, overlap)
    return st[:len(keys)].cpu().numpy()


@pytest.mark.parametrize("seed", range(4))
@pytest.mark.parametrize("overlap", [0.0, 0.1, 0.5, 1.0])
def test_suppression_equals_sequential_greedy(seed, overlap):
    rng = np.random.default_rng(seed)
    shape, radii, a = (20, 60, 70), [1.5, 2.5, 4.0], 1.0 + seed * 0.5
    K = len(radii)
    keys = rng.choice(K * int(np.prod(shape)), size=3000, replace=False)      # priority = this order
    st = _device_keep(keys, shape, radii, a, overlap)
    k, z, y, x = np.unravel_index(keys, (K,) + shape)
    keep = DO.suppress_spheres(np.stack([z * a, y, x], axis=1).astype(np.float64), np.asarray(radii)[k], overlap)
    assert set(np.unique(st)) <= {1, 2}
    assert np.array_equal(st == 1, keep), int(np.count_nonzero((st == 1) != keep))


def test_suppression_long_chain_alternates():
    # spheres of radius 2 every 3 voxels along x, priority left to right: each overlaps the next by ~10 % of its volume,
    # never the one after, so the greedy keeps every other one (a dependency chain as long as the row)
    n = 2500
    shape = (1, 1, 3 * n)
    keys = 3 * np.arange(n)
    st = _device_keep(keys, shape, [2.0], 1.0, 0.05)
    assert np.array_equal(st == 1, np.arange(n) % 2 == 0)
    st = _device_keep(keys[::-1], shape, [2.0], 1.0, 0.05)
    assert np.array_equal(st == 1, np.arange(n) % 2 == 0)


def _lattice(shape, spacing, margin, rng, jitter=1.0):
    g = [np.arange(margin, s - margin, spacing) for s in shape]
    c = np.stack(np.meshgrid(*g, indexing="ij"), axis=-1).reshape(-1, 3).astype(np.float64)
    return c + rng.uniform(-jitter, jitter, c.shape)


def test_find_spheres_equals_oracle_and_finds_nuclei():
    from platymatch_b200.detect_nuclei import find_spheres
    from platymatch_b200.synthetic import make_nuclei_image
    rng = np.random.default_rng(21)
    shape = (160, 160, 160)
    centres = _lattice(shape, 14.0, 8, rng)
    img = make_nuclei_image(shape, centres, rng.uniform(4.0, 6.0, len(centres)), contrast=100, noise=4.0, seed=3)
    radii = [3.0, 4.0, 5.0, 6.0]
    det, r, resp = find_spheres(img, radii)
    rdet, rr, rresp = DO.find_spheres(img, radii)
    assert np.array_equal(det, rdet) and np.array_equal(r, rr) and np.array_equal(resp, rresp)
    d = np.linalg.norm(det.T[:, None, :] - centres[None], axis=2).min(axis=0)
    assert np.mean(d <= 1.0) >= 0.98, np.mean(d <= 1.0)


def test_find_spheres_anisotropic_equals_oracle():
    from platymatch_b200.detect_nuclei import find_spheres
    from platymatch_b200.synthetic import make_nuclei_image
    rng = np.random.default_rng(5)
    img = make_nuclei_image((40, 96, 96), rng.uniform(3, [37, 93, 93], (60, 3)), 4.0, noise=3.0, seed=6)
    for a, ov in ((2.0, 0.5), (1.5, 0.0), (3.0, 1.0)):
        got = find_spheres(img.astype(np.uint16), [2.0, 3.0, 4.5], anisotropy=a, overlap=ov, threshold_factor=0.1)
        ref = DO.find_spheres(img.astype(np.uint16), [2.0, 3.0, 4.5], anisotropy=a, overlap=ov, threshold_factor=0.1)
        for g, e in zip(got, ref):
            assert np.array_equal(g, e)


def test_find_spheres_side_stream():
    import torch
    from platymatch_b200.detect_nuclei import find_spheres
    from platymatch_b200.synthetic import make_nuclei_image
    rng = np.random.default_rng(8)
    img = make_nuclei_image((48, 64, 64), rng.uniform(4, [44, 60, 60], (40, 3)), 3.5, noise=2.0, seed=9)
    ref = find_spheres(img, [2.0, 3.0, 4.0])
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        got = find_spheres(img, [2.0, 3.0, 4.0])
    for g, e in zip(got, ref):
        assert np.array_equal(g, e)
    assert np.array_equal(ref[0], DO.find_spheres(img, [2.0, 3.0, 4.0])[0])


def test_image_to_registration():
    """Two rendered volumes related by a known rigid motion (the label-volume row's setup) -> find_spheres ->
    estimate_transform_unsupervised."""
    import platymatch_b200 as pm
    from platymatch_b200.detect_nuclei import find_spheres
    from platymatch_b200.synthetic import make_nuclei_image
    rng = np.random.default_rng(8)
    n, shape = 400, (160, 160, 160)
    centre = np.array(shape) / 2.0
    d = rng.normal(size=(n, 3))
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    fixed_c = centre + d * np.array([55.0, 48.0, 42.0]) + rng.normal(0, 1.5, size=(n, 3))
    ang = np.deg2rad(12.0)
    R = np.array([[1, 0, 0], [0, np.cos(ang), -np.sin(ang)], [0, np.sin(ang), np.cos(ang)]])
    shift = np.array([3.0, -5.0, 4.0])
    moving_c = (fixed_c - centre - shift) @ R + centre
    fixed_img = make_nuclei_image(shape, fixed_c, 2.5, noise=2.0, seed=1)
    moving_img = make_nuclei_image(shape, moving_c, 2.5, noise=2.0, seed=2)
    fd = find_spheres(fixed_img, [1.5, 2.0, 2.5, 3.0])[0]
    md = find_spheres(moving_img, [1.5, 2.0, 2.5, 3.0])[0]
    assert 0.8 * n < fd.shape[1] < 1.2 * n and 0.8 * n < md.shape[1] < 1.2 * n
    res = pm.estimate_transform_unsupervised(md, fd, ransac_trials=4000, ransac_error=5.0, seed=2)
    A = res["transform"]
    assert np.abs(A[:3, :3] - R).max() < 0.03, A
    moved = A[:3, :3] @ moving_c.T + A[:3, 3:4]
    assert np.median(np.linalg.norm(moved - fixed_c.T, axis=0)) < 1.5


def test_pass_above_2_31_voxels():
    import torch
    from platymatch_b200 import device as D
    from platymatch_b200.detect_nuclei.ss_log import log_weights
    shape = (8, 16384, 16401)                                       # 2.15e9 voxels
    assert np.prod(shape) > 2 ** 31
    g = torch.Generator(device="cuda").manual_seed(0)
    x = torch.rand(shape, generator=g, device="cuda")
    w = log_weights(2.9, 2)
    lw = w.size - 1
    for axis in (2, 0):
        out = D.detect_pass(x, axis, _dev(w))
        for (z, y) in ((7, 16383), (7, 16000), (3, 9000)):
            if axis == 2:
                line = x[z, y].double().cpu().numpy()
                got = out[z, y].cpu().numpy()
            else:
                line = x[:, y, 16400].double().cpu().numpy()
                got = out[:, y, 16400].cpu().numpy()
            n = line.size
            p = np.pad(line, lw, mode="symmetric")
            acc = p[lw:lw + n] * w[0]
            for j in range(lw, 0, -1):
                acc = acc + (p[lw - j:lw - j + n] + p[lw + j:lw + j + n]) * w[j]
            assert np.array_equal(got, acc.astype(np.float32)), (axis, z, y)
        del out
        torch.cuda.empty_cache()
