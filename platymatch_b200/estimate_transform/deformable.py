"""Deformable refinement of a registration: a smoothing thin-plate spline fitted to matched nuclei.  DESIGN §8 row 8.

Two specimens of one stage differ by more than an affine map.  After `estimate_transform_*` (affine + ICP) what is left
is a smooth local deformation; these functions fit it on the nucleus correspondences the affine registration gives and
move points or volumes through it (`utils/images.py::transform_image_deformable`).  The reference has no deformable
step: the contract is this project's own, written down with scipy.

A spline maps source points to target points (3 x N zyx clouds, as elsewhere):
    f(x) = sum_k c_k * (-||x - y_k||) + c_K + sum_h c_{K+1+h} * (x_h - shift_h) / scale_h
with centres y_k (the source points), coefficients c [(K + 4) x 3] and per-axis shift / scale.  It is exactly
scipy.interpolate.RBFInterpolator(y, d, kernel='linear', degree=1, smoothing): in 3-D the biharmonic spline, with
scipy's monomial order and scipy's shift = (min + max) / 2, scale = (max - min) / 2 (0 -> 1), computed here in numpy.
The system [-R + lambda I, P; P^T, 0] c = [d; 0] is written by pm_spline_system and solved on the device in float64.
"""
import numpy as np

from .. import device as D
from ..evaluate_metrics import assign_by_distance
from .apply_transform import apply_affine_transform

__all__ = ["Spline", "fit_spline", "apply_spline", "match_nuclei", "estimate_deformation", "DEFAULT_SMOOTHING",
           "MAX_CENTRES"]

# chosen from {0, 1, 10, 100, 1000} by the median error on held-out nuclei of make_deformed_pair (DESIGN §8 row 8)
DEFAULT_SMOOTHING = 100.0
# the float64 system of K = 16384 centres is 2.1 GB (and the LU factorisation holds a copy)
MAX_CENTRES = 16384


class Spline:
    """A fitted spline, its arrays on the device: centres [K, 3], coeffs [K + 4, 3], shift_scale [6] = (shift, scale),
    all float64 CUDA tensors.  Call it (or `apply_spline`) on a 3 x N cloud."""

    def __init__(self, centres, coeffs, shift_scale, smoothing):
        self.centres, self.coeffs, self.shift_scale, self.smoothing = centres, coeffs, shift_scale, float(smoothing)

    @property
    def k(self):
        return self.centres.shape[0]

    def to_numpy(self):
        """dict(centres (3, K), coeffs (K + 4, 3), shift (3,), scale (3,), smoothing) on the host."""
        ss = self.shift_scale.cpu().numpy()
        return {"centres": np.ascontiguousarray(self.centres.cpu().numpy().T), "coeffs": self.coeffs.cpu().numpy(),
                "shift": ss[:3].copy(), "scale": ss[3:].copy(), "smoothing": self.smoothing}

    def __call__(self, points):
        return apply_spline(self, points)


def _cloud(a, name):
    a = np.asarray(a, dtype=np.float64)
    if a.ndim != 2 or a.shape[0] not in (3, 4):
        raise ValueError("%s: expected a 3 x N (or 4 x N) cloud, got shape %s" % (name, a.shape))
    a = np.ascontiguousarray(a[:3])
    if not np.all(np.isfinite(a)):
        raise ValueError("%s: points must be finite (NaN or inf found)" % name)
    return a


def shift_scale(points):
    """scipy's polynomial domain for K x 3 points: shift = (min + max) / 2, scale = (max - min) / 2, 0 -> 1."""
    mins, maxs = points.min(axis=0), points.max(axis=0)
    shift = (maxs + mins) / 2
    scale = (maxs - mins) / 2
    scale[scale == 0.0] = 1.0
    return shift, scale


def fit_spline(source, target, smoothing=DEFAULT_SMOOTHING):
    """The smoothing thin-plate spline f with f(source_k) ~= target_k (3 x K clouds in correspondence order), fitted on
    the GPU.  Equal to RBFInterpolator(source.T, target.T, kernel='linear', degree=1, smoothing=smoothing).

    Refused on the host, before any device work: clouds that are not 3 x K of one K, NaN or inf, K < 4 or K > 16384,
    a negative or non-finite smoothing, source points that all lie in one plane (the polynomial block has rank < 4;
    scipy refuses them too) and, when smoothing is 0, two equal source points.  The system is solved with LU
    (torch.linalg.solve_ex) in float64; fit_spline synchronises once, and raises when the factorisation reports a
    singular matrix or the coefficients are not finite.
    """
    y, d = _cloud(source, "source").T, _cloud(target, "target").T
    k = y.shape[0]
    if d.shape[0] != k:
        raise ValueError("source and target differ in size: %d and %d points" % (k, d.shape[0]))
    if k < 4:
        raise ValueError("a spline needs at least 4 points, got %d" % k)
    if k > MAX_CENTRES:
        raise ValueError("at most %d points are supported (the float64 system of K points takes 8 (K + 4)^2 bytes), "
                         "got %d" % (MAX_CENTRES, k))
    lam = float(smoothing)
    if not (np.isfinite(lam) and lam >= 0.0):
        raise ValueError("smoothing must be finite and >= 0, got %r" % (smoothing,))
    shift, scale = shift_scale(y)
    poly = np.hstack([np.ones((k, 1)), (y - shift) / scale])
    rank = np.linalg.matrix_rank(poly)
    if rank < 4:
        raise ValueError("singular matrix: the source points lie in a plane or on a line (polynomial rank %d of 4)" % rank)
    if lam == 0.0 and np.unique(y, axis=0).shape[0] < k:
        raise ValueError("singular matrix: two source points are equal, which needs smoothing > 0")
    torch = D._torch()
    dev = torch.device("cuda", torch.cuda.current_device())
    # centres, shift / scale and targets in one pinned upload, so that the only synchronisation is the status read
    staged = torch.empty(6 * k + 6, dtype=torch.float64, pin_memory=True)
    staged.numpy()[...] = np.concatenate([y.reshape(-1), shift, scale, d.reshape(-1)])
    buf = staged.to(dev, non_blocking=True)
    centres = buf[:3 * k].view(k, 3)
    ss = buf[3 * k:3 * k + 6]
    lhs = D.spline_system(centres, ss, lam)
    rhs = torch.zeros((k + 4, 3), dtype=torch.float64, device=dev)
    rhs[:k] = buf[3 * k + 6:].view(k, 3)
    coeffs, info = torch.linalg.solve_ex(lhs, rhs)
    del lhs
    status = torch.stack([info.to(torch.float64), torch.isfinite(coeffs).all().to(torch.float64)]).cpu().numpy()
    if status[0] != 0 or status[1] != 1:
        raise ValueError("singular matrix: the spline system could not be solved (LU info %d)" % int(status[0]))
    return Spline(centres.clone(), coeffs.contiguous(), ss.clone(), lam)


def apply_spline(spline, points):
    """f(points) for a 3 x N (or 4 x N) cloud -> 3 x N float64 on the host (pm_spline_eval)."""
    p = _cloud(points, "points")
    if p.shape[1] == 0:
        return np.zeros((3, 0))
    out = D.spline_eval(spline.centres, spline.coeffs, spline.shift_scale, D.to_device_points(p))
    return np.ascontiguousarray(out.cpu().numpy().T)


def match_nuclei(moving, fixed, transform, max_distance=16.0):
    """Nucleus correspondences under an affine registration: the optimal one-to-one assignment between
    `transform` @ moving and fixed by Euclidean distance (pm_cdist + the exact assignment kernel, as
    `assign_by_distance`), keeping the pairs whose distance is <= max_distance (default 16, the widget's RANSAC inlier
    distance, in the same units).  Returns (moving_idx, fixed_idx, distance), ascending in moving_idx."""
    m, f = _cloud(moving, "moving"), _cloud(fixed, "fixed")
    T = np.asarray(transform, dtype=np.float64)
    if T.shape != (4, 4) or not np.all(np.isfinite(T)):
        raise ValueError("transform must be a finite 4 x 4 matrix")
    if not max_distance >= 0:
        raise ValueError("max_distance must be >= 0, got %r" % (max_distance,))
    moved = apply_affine_transform(m, T)
    rows, cols = assign_by_distance(moved, f)
    dist = np.linalg.norm(moved[:, rows] - f[:, cols], axis=0)
    keep = dist <= max_distance
    return rows[keep], cols[keep], dist[keep]


def estimate_deformation(moving, fixed, transform, *, max_distance=16.0, smoothing=DEFAULT_SMOOTHING):
    """Refine an affine registration (transform: moving zyx -> fixed zyx, as `estimate_transform_*` returns it) with
    a smoothing thin-plate spline fitted to the nuclei `match_nuclei` pairs.

    Returns a dict:
      forward       Spline moving -> fixed (moves points: apply_spline(forward, moving))
      inverse       Spline fixed -> moving, fitted on the same pairs: the pull map that resampling needs
                    (`transform_image_deformable`).  The two are separate fits and are NOT exact inverses of each
                    other; with smoothing > 0 neither interpolates the pairs exactly.
      moving_index, fixed_index, distance   the pairs and their distance under `transform`
      median_residual_affine   median pair distance under `transform`
      median_residual_spline   median ||forward(moving_i) - fixed_i|| over the pairs
    The polynomial part of each spline is affine, so the splines map the raw clouds: `transform` only selects pairs.
    """
    m, f = _cloud(moving, "moving"), _cloud(fixed, "fixed")
    mi, fi, dist = match_nuclei(m, f, transform, max_distance)
    src, dst = m[:, mi], f[:, fi]
    forward = fit_spline(src, dst, smoothing)
    inverse = fit_spline(dst, src, smoothing)
    moved = apply_spline(forward, src)
    return {"forward": forward, "inverse": inverse, "moving_index": mi, "fixed_index": fi, "distance": dist,
            "median_residual_affine": float(np.median(dist)),
            "median_residual_spline": float(np.median(np.linalg.norm(moved - dst, axis=0)))}
