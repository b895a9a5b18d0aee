"""Synthetic embryo-like nuclei clouds (SURVEY.md §8d; BASELINE.json `configs`).

Host-side numpy only: this is the workload generator used by tests and bench.py, not part of
the registration path.  Clouds are modelled on the reference's test assets
(`platymatch/_tests/assets/02-insitu.csv`: 331 nuclei on a thick near-spherical shell, radius
~122 px, nearest-neighbour spacing ~19 px, zyx pixel coordinates).
"""
import numpy as np

__all__ = ["make_fixed_cloud", "random_affine", "make_pair", "make_keypoints", "make_specimens", "make_label_volume",
           "make_nuclei_image"]


def make_fixed_cloud(n, rng, filled=False):
    """(3, n) float64 zyx cloud: shell of radius 122*sqrt(n/331) +- 8 px, axes (1.10, 1.00, 0.92).
    filled=True: the late-stage-embryo variant of SURVEY §8(d) — nuclei uniform in the VOLUME of the same
    ellipsoid shape at the assets' nearest-neighbour spacing (~19 px for a Poisson cloud: 4.0e4 px^3 per nucleus).  Its shape-context
    histograms populate ~2.6x more bins than a shell's (every ring sees every polar angle)."""
    s = np.sqrt(n / 331.0)
    d = rng.standard_normal((3, n))
    d /= np.linalg.norm(d, axis=0, keepdims=True)
    if filled:
        big_r = (3.0 * n * 4.0e4 / (4.0 * np.pi)) ** (1.0 / 3.0)
        r = big_r * rng.random(n) ** (1.0 / 3.0)
        pts = d * r * np.array([[1.10], [1.00], [0.92]])
        return pts + (1.5 * big_r + 50.0)
    r = 122.0 * s + rng.normal(0.0, 8.0, size=n)
    pts = d * r * np.array([[1.10], [1.00], [0.92]])
    return pts + np.array([[350.0], [270.0], [280.0]]) * s


def random_affine(rng, anisotropy=None):
    """4x4: (QR-orthogonal x diag U(0.9,1.1)) linear part, translation U(-100,100)^3.
    anisotropy=a: one scale U(0.9,1.1) for all axes x per-axis U(1-a, 1+a) instead (a near-similarity)."""
    q, r = np.linalg.qr(rng.standard_normal((3, 3)))
    q = q * np.sign(np.diag(r))  # unique QR
    a = np.eye(4)
    if anisotropy is None:
        scale = rng.uniform(0.9, 1.1, size=3)
    else:
        scale = rng.uniform(0.9, 1.1) * rng.uniform(1.0 - anisotropy, 1.0 + anisotropy, size=3)
    a[:3, :3] = q @ np.diag(scale)
    a[:3, 3] = rng.uniform(-100.0, 100.0, size=3)
    return a


def make_pair(n_fixed, seed=None, jitter=2.0, dropout=0.10, filled=False):
    """One registration problem.

    Returns dict(moving (3,N1), fixed (3,N2), A_gt (4,4) with fixed ~= A_gt @ moving,
    gt_fixed_index (N1,) = index into fixed of each moving nucleus' true partner).
    """
    rng = np.random.default_rng(n_fixed if seed is None else seed)
    fixed = make_fixed_cloud(n_fixed, rng, filled)
    a_gt = random_affine(rng)
    a_inv = np.linalg.inv(a_gt)
    moving_all = a_inv[:3, :3] @ fixed + a_inv[:3, 3:4]
    moving_all = moving_all + rng.normal(0.0, jitter, size=moving_all.shape)
    keep = rng.permutation(n_fixed)[: n_fixed - int(round(dropout * n_fixed))]
    keep = rng.permutation(keep)
    return {"moving": np.ascontiguousarray(moving_all[:, keep]), "fixed": fixed, "A_gt": a_gt,
            "gt_fixed_index": keep.astype(np.int64)}


def make_keypoints(pair, n_keypoints=10, seed=0, jitter=1.0):
    """Keypoint-supervised config: n ground-truth pairs among surviving nuclei (+ click jitter)."""
    rng = np.random.default_rng(seed)
    sel = rng.choice(pair["moving"].shape[1], n_keypoints, replace=False)
    mk = pair["moving"][:, sel] + rng.normal(0.0, jitter, size=(3, n_keypoints))
    fk = pair["fixed"][:, pair["gt_fixed_index"][sel]] + rng.normal(0.0, jitter, size=(3, n_keypoints))
    return mk, fk


def make_specimens(n_specimens=12, n_nuclei=8000, jitter=2.0, dropout=0.10, seed=0, vary=0.05, anisotropy=0.02):
    """Batched all-pairs config: specimens are jittered, thinned views of one atlas with ~n_nuclei nuclei each
    (n_nuclei * (1 - U(0, vary)); vary=0: exactly equal counts), each in its own pose: rotation x overall scale
    U(0.9,1.1) x per-axis U(1-anisotropy, 1+anisotropy).  Specimens of one stage differ by pose and size, not by shape:
    the method (the reference's as well) aligns the clouds' first PCA axes, and a pair whose relative transform
    distorts the shape enough to swap that axis (the fully anisotropic `random_affine(rng)` does, for the 10 %
    elongation of this shell, in about half of all pairs) cannot be registered by it at all."""
    rng = np.random.default_rng(seed)
    atlas = make_fixed_cloud(int(round(n_nuclei / (1.0 - dropout))), rng)
    out = []
    for s in range(n_specimens):
        r = np.random.default_rng(1000 + s)
        a = random_affine(r, anisotropy)
        pts = a[:3, :3] @ atlas + a[:3, 3:4] + r.normal(0.0, jitter, size=atlas.shape)
        n_s = n_nuclei if not vary else int(round(n_nuclei * (1.0 - vary * r.random())))
        keep = r.permutation(atlas.shape[1])[:n_s]
        out.append({"points": np.ascontiguousarray(pts[:, keep]), "A": a, "atlas_index": keep})
    return out


def make_label_volume(shape=(64, 96, 128), n_nuclei=60, radius=(3.0, 6.0), seed=0, dtype=np.int32, sparse_ids=False,
                      centers=None):
    """Instance-segmentation volume: `n_nuclei` non-overlapping-ish balls with ids 1..n (or sparse, shuffled ids),
    0 = background.  Later balls overwrite earlier ones, some ids may end up partially or fully covered.
    centers: optional (n, 3) zyx ball centres (default: uniform in the volume)."""
    rng = np.random.default_rng(seed)
    nz, ny, nx = shape
    if centers is not None:
        n_nuclei = len(centers)
    vol = np.zeros(shape, dtype=np.int64)
    ids = np.arange(1, n_nuclei + 1)
    if sparse_ids:
        ids = np.sort(rng.choice(np.arange(1, 20 * n_nuclei), n_nuclei, replace=False))
        ids = rng.permutation(ids)
    zz, yy, xx = np.meshgrid(np.arange(nz), np.arange(ny), np.arange(nx), indexing="ij", sparse=True)
    for k in range(n_nuclei):
        c = rng.random(3) * np.array(shape) if centers is None else np.asarray(centers[k], dtype=np.float64)
        r = rng.uniform(*radius)
        z0, z1 = int(max(c[0] - r, 0)), int(min(c[0] + r + 1, nz))
        y0, y1 = int(max(c[1] - r, 0)), int(min(c[1] + r + 1, ny))
        x0, x1 = int(max(c[2] - r, 0)), int(min(c[2] + r + 1, nx))
        sub = ((zz[z0:z1] - c[0]) ** 2 + (yy[:, y0:y1] - c[1]) ** 2 + (xx[:, :, x0:x1] - c[2]) ** 2) <= r * r
        vol[z0:z1, y0:y1, x0:x1][sub] = ids[k]
    return vol.astype(dtype)


def make_nuclei_image(shape, centers, radius, contrast=100.0, background=10.0, noise=2.0, seed=0):
    """float32 intensity volume of nuclei-stained nuclei: background + contrast x a Gaussian blob of sigma = radius / 2
    at each (z, y, x) centre (radius: scalar or one per centre, voxels), plus Gaussian noise of std `noise`."""
    rng = np.random.default_rng(seed)
    centers = np.asarray(centers, dtype=np.float64).reshape(-1, 3)
    rad = np.broadcast_to(np.asarray(radius, dtype=np.float64), (len(centers),))
    vol = np.full(shape, float(background), dtype=np.float64)
    for c, r in zip(centers, rad):
        s = r / 2.0
        lo = [max(int(np.floor(c[h] - 4 * s)), 0) for h in range(3)]
        hi = [min(int(np.ceil(c[h] + 4 * s)) + 1, shape[h]) for h in range(3)]
        if any(a >= b for a, b in zip(lo, hi)):
            continue
        g = [np.exp(-0.5 * ((np.arange(lo[h], hi[h]) - c[h]) / s) ** 2) for h in range(3)]
        vol[lo[0]:hi[0], lo[1]:hi[1], lo[2]:hi[2]] += contrast * g[0][:, None, None] * g[1][None, :, None] * g[2]
    if noise:
        vol += rng.normal(0.0, noise, size=shape)
    return vol.astype(np.float32)
