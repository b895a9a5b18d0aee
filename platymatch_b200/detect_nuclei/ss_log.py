"""Raw nuclei-stained volume -> detections: the reference's `DetectNuclei` stage (platymatch/detect_nuclei/ss_log.py,
`find_spheres` :83-87, called by `DetectNuclei._click_run` :133-149), SURVEY §2 row 10.

The reference's exact parameters are not available to this project, so `find_spheres` implements this project's own
contract (DESIGN §8 row 6, restated with scipy in tests/detect_oracle.py).  Agreement with the reference's output and
signatures is unverified.

  1. L_k = float32(sigma_k^2) * gaussian_laplace(img32, (sigma_k / a, sigma_k, sigma_k)), sigma_k = r_k / sqrt(3),
     mode 'reflect', truncate 4 (8 separable passes on the GPU, bit-identical to scipy's 9)
  2. candidates: (L, linear index in (k, z, y, x) order) strictly smallest in the 3x3x3x3 scale-space neighbourhood
     (one voxel per tie group; unlike skimage's plateau marking, a plateau larger than the neighbourhood gives none)
  3. keep -float64(L) > threshold_factor * otsu(img32)  (skimage's threshold_otsu, 256 bins)
  4. greedy suppression in (L, index) order: a sphere (z a, y, x; r_k) is dropped when its intersection volume with an
     already kept one is greater than overlap x the smaller sphere's volume
"""
import math

import numpy as np

from .. import device as D

__all__ = ["find_spheres", "sphere_intersection", "gaussian_kernel1d", "log_weights"]

MAX_LW = 384            # longest half-kernel pm_detect_pass takes


def gaussian_kernel1d(sigma, order, radius):
    """scipy.ndimage's `_gaussian_kernel1d` (float64), restated with numpy: the weights gaussian_filter1d correlates
    with for `sigma`, derivative `order` and half-width `radius` = int(4 sigma + 0.5)."""
    exponent_range = np.arange(order + 1)
    sigma2 = sigma * sigma
    x = np.arange(-radius, radius + 1)
    phi_x = np.exp(-0.5 / sigma2 * x ** 2)
    phi_x = phi_x / phi_x.sum()
    if order == 0:
        return phi_x
    q = np.zeros(order + 1)
    q[0] = 1
    Dm = np.diag(exponent_range[1:], 1)
    P = np.diag(np.ones(order) / -sigma2, -1)
    Q_deriv = Dm + P
    for _ in range(order):
        q = Q_deriv.dot(q)
    q = (x[:, None] ** exponent_range).dot(q)
    return q * phi_x


def log_weights(sigma, order):
    """Half-kernel w[0..lw] (centre first) of gaussian_filter1d(sigma, order, truncate=4): what pm_detect_pass takes."""
    sigma = float(sigma)
    lw = int(4.0 * sigma + 0.5)
    if lw > MAX_LW:
        raise ValueError("sigma %g needs a kernel half-width of %d > %d" % (sigma, lw, MAX_LW))
    w = gaussian_kernel1d(sigma, order, lw)[::-1]
    assert np.array_equal(w, w[::-1]), "Gaussian weights must be symmetric"
    return np.ascontiguousarray(w[lw:])


def sphere_intersection(c1, r1, c2, r2):
    """Intersection volume of two spheres (centres in physical units), float64: 0 when disjoint, the smaller sphere's
    volume when one contains the other, else the lens volume.  The device evaluates the same expression in the same
    order (pm_detect.cu, pm_dt_conflict)."""
    r1, r2 = float(r1), float(r2)
    dz, dy, dx = float(c1[0]) - float(c2[0]), float(c1[1]) - float(c2[1]), float(c1[2]) - float(c2[2])
    d = math.sqrt(dz * dz + dy * dy + dx * dx)
    rs = r1 if r1 < r2 else r2
    if d >= r1 + r2:
        return 0.0
    if d <= abs(r1 - r2):
        return 4.0 / 3.0 * math.pi * rs * rs * rs
    if r1 < r2:                                  # the larger radius first: symmetric in its arguments
        r1, r2 = r2, r1
    h = r1 + r2 - d
    return math.pi * h * h * (d * d + 2.0 * d * r2 - 3.0 * r2 * r2 + 2.0 * d * r1 + 6.0 * r1 * r2 - 3.0 * r1 * r1) / (
        12.0 * d)


def _check(image, radii, anisotropy, threshold_factor, overlap):
    a = np.asarray(image)
    if a.dtype == np.bool_ or np.iscomplexobj(a) or not (np.issubdtype(a.dtype, np.integer) or
                                                        np.issubdtype(a.dtype, np.floating)):
        raise ValueError("image must have a real integer or float dtype, got %s" % a.dtype)
    if a.ndim != 3 or a.size == 0:
        raise ValueError("expected a non-empty 3-D volume, got shape %s" % (a.shape,))
    r = np.asarray(radii, dtype=np.float64).reshape(-1)
    if r.size == 0 or not np.all(np.isfinite(r)) or np.any(r <= 0) or np.any(np.diff(r) <= 0):
        raise ValueError("radii must be non-empty, finite, > 0 and strictly ascending, got %r" % (radii,))
    anisotropy = float(anisotropy)
    if not (anisotropy > 0 and math.isfinite(anisotropy)):
        raise ValueError("anisotropy must be > 0, got %r" % (anisotropy,))
    overlap = float(overlap)
    if not (0.0 <= overlap <= 1.0):
        raise ValueError("overlap must be in [0, 1], got %r" % (overlap,))
    threshold_factor = float(threshold_factor)
    if not math.isfinite(threshold_factor):
        raise ValueError("threshold_factor must be finite, got %r" % (threshold_factor,))
    weights = []
    for rk in r:
        s = rk / math.sqrt(3.0)
        weights.append([log_weights(s / anisotropy, 0), log_weights(s / anisotropy, 2), log_weights(s, 0),
                        log_weights(s, 2)])
    return a, r, anisotropy, threshold_factor, overlap, weights


def _scale_space(img, r, weights, bufs, slots, thr, keys, values, count):
    """Enqueue every scale's LoG and minima; three L slots rotate (minima of k needs L_{k-1}, L_k, L_{k+1})."""
    gz, t1, t2, acc = bufs
    K = len(r)
    for k in range(K):
        wz0, wz2, w0, w2 = weights[k]
        sigma = r[k] / math.sqrt(3.0)
        L = slots[k % 3]
        D.detect_pass(img, 0, wz0, out=gz)                         # Gz, shared by the y and x terms
        D.detect_pass(img, 0, wz2, out=t1)                         # D2z -> Gy -> Gx
        D.detect_pass(t1, 1, w0, out=t2)
        D.detect_pass(t2, 2, w0, out=acc)
        D.detect_pass(gz, 1, w2, out=t1)                           # Gz -> D2y -> Gx
        D.detect_pass(t1, 2, w0, out=t2)
        D.detect_pass(gz, 1, w0, out=t1)                           # Gz -> Gy -> D2x, + the sum and the scale
        D.detect_pass(t1, 2, w2, out=L, t0=acc, t1=t2, scale=float(np.float32(sigma ** 2)))
        if k >= 1:
            D.detect_minima(slots[(k - 2) % 3] if k >= 2 else None, slots[(k - 1) % 3], L, k - 1, thr, keys, values,
                            count)
    D.detect_minima(slots[(K - 2) % 3] if K >= 2 else None, slots[(K - 1) % 3], None, K - 1, thr, keys, values, count)


def find_spheres(image, radii, anisotropy=1.0, threshold_factor=0.2, overlap=0.5):
    """Nuclei of an intensity volume as scale-space LoG minima, on the GPU.

    image             (nz, ny, nx) volume of a real dtype (converted with astype(np.float32))
    radii             ascending nucleus radii r_k > 0 in xy voxels, one scale each
    anisotropy        z spacing over xy spacing
    threshold_factor  candidates need -L > threshold_factor * otsu(image)
    overlap           a sphere is suppressed when more than this fraction of the smaller sphere lies in a kept one
    Returns (detections (3, N) float64 integer voxel indices z, y, x; radii (N,) float64; responses (N,) float32 = L),
    strongest response first.  Synchronises with the host once (twice when the candidate buffer overflowed).
    """
    a, r, anisotropy, threshold_factor, overlap, weights = _check(image, radii, anisotropy, threshold_factor, overlap)
    torch = D._torch()
    shape = a.shape
    K, V = len(r), int(np.prod(shape))
    host = torch.from_numpy(np.ascontiguousarray(a.astype(np.float32))).pin_memory()
    img = host.to("cuda", non_blocking=True)
    flat = np.concatenate([w for ws in weights for w in ws] + [r])
    wdev = torch.from_numpy(flat).pin_memory().to("cuda", non_blocking=True)
    views, o = [], 0
    for ws in weights:
        views.append([])
        for w in ws:
            views[-1].append(wdev[o:o + w.size])
            o += w.size
    rdev = wdev[o:]
    bufs = [torch.empty_like(img) for _ in range(4)]
    slots = [torch.empty_like(img) for _ in range(min(K, 3))]
    thr = D.detect_otsu(img, threshold_factor)
    bound = ((K + 1) // 2) * ((shape[0] + 1) // 2) * ((shape[1] + 1) // 2) * ((shape[2] + 1) // 2)
    cap = min(bound, max(1 << 16, K * V // 1024))
    while True:
        keys = torch.full((cap,), np.iinfo(np.int64).max, dtype=torch.int64, device="cuda")
        values = torch.full((cap,), float("inf"), dtype=torch.float32, device="cuda")
        count = torch.zeros(1, dtype=torch.int64, device="cuda")
        _scale_space(img, r, views, bufs, slots, thr, keys, values, count)
        keys, o1 = torch.sort(keys)                               # priority: (L, linear index) ascending
        values, o2 = torch.sort(values[o1], stable=True)
        keys = keys[o2]
        state = D.detect_suppress(keys, count, shape, rdev, float(r[-1]), anisotropy, overlap)
        out = [torch.empty(t.shape, dtype=t.dtype, pin_memory=True) for t in (count, keys, values, state)]
        for h, t in zip(out, (count, keys, values, state)):
            h.copy_(t, non_blocking=True)
        torch.cuda.current_stream().synchronize()
        n_found = int(out[0][0])
        if n_found <= cap:
            break
        cap = bound                                                # retry once with the hard bound
    n = n_found
    keep = out[3].numpy()[:n] == 1
    sel = out[1].numpy()[:n][keep]
    k, z, y, x = np.unravel_index(sel, (K,) + shape)
    det = np.stack([z, y, x]).astype(np.float64)
    return det, r[k], out[2].numpy()[:n][keep].copy()
