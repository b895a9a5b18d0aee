"""CPU oracle of nuclei detection (SURVEY §2 row 10; the project's own contract, DESIGN §8 row 6), written with scipy
and numpy: scipy.ndimage.gaussian_laplace itself, a (value, index) scale-space neighbourhood minimum, skimage's
threshold_otsu restated, and the sequential greedy sphere suppression.  Only tests and tools import it; the product
(platymatch_b200.detect_nuclei) never does."""
import math

import numpy as np


def otsu_histogram(img32):
    """np.histogram(img32, 256, range=(min, max)) restated per value, as pm_detect_hist_kernel bins: float32 arithmetic
    against float32 np.linspace edges.  Returns (counts int64, edges float32)."""
    a = np.asarray(img32, dtype=np.float32).ravel()
    first, last = a.min(), a.max()
    denom = np.float32(last - first)
    step = np.float32(denom / np.float32(256))
    edges = (np.arange(257, dtype=np.float32) * step + first).astype(np.float32)
    edges[256] = last
    b = (((a - first) / denom) * np.float32(256)).astype(np.int64)
    b[b == 256] -= 1
    b[a < edges[b]] -= 1
    b[(a >= edges[b + 1]) & (b != 255)] += 1
    return np.bincount(b, minlength=256).astype(np.int64), edges


def otsu(img32):
    """skimage.filters.threshold_otsu(img32, nbins=256) restated: np.histogram over (min, max), float32 bin centres,
    float64 between-class variance from cumulative sums, first maximum; a constant image returns its value."""
    a = np.asarray(img32, dtype=np.float32)
    lo, hi = a.min(), a.max()
    if lo == hi:
        return float(lo)
    counts, edges = np.histogram(a, 256, range=(lo, hi))
    centres = (edges[:-1] + edges[1:]) / 2
    counts = counts.astype(np.float64)
    weight1 = np.cumsum(counts)
    weight2 = np.cumsum(counts[::-1])[::-1]
    mean1 = np.cumsum(counts * centres) / weight1
    mean2 = (np.cumsum((counts * centres)[::-1]) / weight2[::-1])[::-1]
    variance12 = weight1[:-1] * weight2[1:] * (mean1[:-1] - mean2[1:]) ** 2
    return float(centres[np.argmax(variance12)])


def scale_space_log(img32, radii, anisotropy=1.0):
    """[K] list of L_k = float32(sigma_k^2) * gaussian_laplace(img32, (sigma_k / a, sigma_k, sigma_k))."""
    import scipy.ndimage as nd
    out = []
    for r in radii:
        s = float(r) / np.sqrt(3.0)
        out.append(np.float32(s ** 2) * nd.gaussian_laplace(img32, (s / anisotropy, s, s)))
    return out


def scale_space_minima(L, threshold):
    """Candidates (keys = linear indices in (k, z, y, x) order, values = L) of the stack L [K][nz][ny][nx]: the pair
    (L, index) strictly smallest in the 3x3x3x3 neighbourhood, and -float64(L) > threshold.  Ascending keys."""
    L = np.asarray(L, dtype=np.float32)
    P = np.pad(L, 1, mode="constant", constant_values=np.inf)
    keys = np.flatnonzero(-L.astype(np.float64).ravel() > threshold)
    idx = np.unravel_index(keys, L.shape)
    v = L[idx]
    ok = np.ones(keys.size, dtype=bool)
    for off in np.ndindex(3, 3, 3, 3):
        d = tuple(o - 1 for o in off)
        if d == (0, 0, 0, 0):
            continue
        u = P[tuple(i + 1 + e for i, e in zip(idx, d))]
        ok &= (v <= u) if d > (0, 0, 0, 0) else (v < u)
    return keys[ok], v[ok]


def sphere_intersection(c1, r1, c2, r2):
    """Intersection volume of two spheres, float64 (the same expression, in the same order, as the product's)."""
    dz, dy, dx = c1[0] - c2[0], c1[1] - c2[1], c1[2] - c2[2]
    d = math.sqrt(dz * dz + dy * dy + dx * dx)
    rs = min(r1, r2)
    if d >= r1 + r2:
        return 0.0
    if d <= abs(r1 - r2):
        return 4.0 / 3.0 * math.pi * rs * rs * rs
    if r1 < r2:                                  # the larger radius first: symmetric in its arguments
        r1, r2 = r2, r1
    h = r1 + r2 - d
    return math.pi * h * h * (d * d + 2.0 * d * r2 - 3.0 * r2 * r2 + 2.0 * d * r1 + 6.0 * r1 * r2 - 3.0 * r1 * r1) / (
        12.0 * d)


def suppress_spheres(centres, radii, overlap):
    """Sequential greedy over spheres already in priority order: keep one unless its intersection with an already
    kept sphere is greater than overlap x the smaller sphere's volume.  Returns the boolean keep mask."""
    n = len(radii)
    keep = np.zeros(n, dtype=bool)
    cell = 2.0 * float(np.max(radii)) if n else 1.0
    grid = {}
    for i in range(n):
        c, r = [float(t) for t in centres[i]], float(radii[i])
        key = tuple(int(math.floor(t / cell)) for t in c)
        rs_ok = True
        for off in np.ndindex(3, 3, 3):
            for j in grid.get(tuple(k + o - 1 for k, o in zip(key, off)), ()):
                rj = float(radii[j])
                rs = min(r, rj)
                if sphere_intersection(c, r, [float(t) for t in centres[j]], rj) > overlap * (
                        4.0 / 3.0 * math.pi * rs * rs * rs):
                    rs_ok = False
                    break
            if not rs_ok:
                break
        if rs_ok:
            keep[i] = True
            grid.setdefault(key, []).append(i)
    return keep


def find_spheres(image, radii, anisotropy=1.0, threshold_factor=0.2, overlap=0.5, return_stages=False):
    """The detection contract with scipy and numpy: scale-space LoG, (value, index) minima, threshold_factor x Otsu,
    greedy suppression in (L, index) order.  -> (detections (3, N) float64 zyx, radii (N,), responses (N,) float32)."""
    img32 = np.asarray(image).astype(np.float32)
    radii = np.asarray(radii, dtype=np.float64)
    t = threshold_factor * otsu(img32)
    L = scale_space_log(img32, radii, anisotropy)
    keys, vals = scale_space_minima(np.stack(L), t)
    order = np.lexsort((keys, vals))
    keys, vals = keys[order], vals[order]
    k, z, y, x = np.unravel_index(keys, (len(radii),) + img32.shape)
    centres = np.stack([z * float(anisotropy), y.astype(np.float64), x.astype(np.float64)], axis=1)
    keep = suppress_spheres(centres, radii[k], overlap)
    det = np.stack([z, y, x])[:, keep].astype(np.float64)
    res = (det, radii[k][keep], vals[keep])
    if return_stages:
        return res, {"threshold": t, "L": L, "keys": keys, "values": vals, "keep": keep}
    return res
