"""numpy restatements of the thin-plate spline kernels (DESIGN §8 row 8), for the tests: the system matrix pm_spline_system
writes (bit for bit) and the row-5 sampler pm_resample_spline applies at a coordinate (order 0 bit for bit; order 1 in
float64 without the kernel's FMA contraction)."""
import numpy as np


def system_matrix(y, shift, scale, smoothing):
    """[-R + smoothing I, P; P^T, 0] for centres y (K, 3): R_ij = sqrt((dz*dz + dy*dy) + dx*dx), P = [1, (y - shift) / scale]."""
    k = y.shape[0]
    dz, dy, dx = (y[:, h][:, None] - y[:, h][None, :] for h in range(3))
    lhs = np.zeros((k + 4, k + 4))
    lhs[:k, :k] = -np.sqrt((dz * dz + dy * dy) + dx * dx)
    lhs[np.arange(k), np.arange(k)] += smoothing
    p = np.hstack([np.ones((k, 1)), (y - shift) / scale])
    lhs[:k, k:] = p
    lhs[k:, :k] = p.T
    return lhs


def rbf(source, target, smoothing):
    """The scipy contract: RBFInterpolator over 3 x K clouds."""
    from scipy.interpolate import RBFInterpolator
    return RBFInterpolator(np.asarray(source).T, np.asarray(target).T, kernel="linear", degree=1, smoothing=smoothing)


def grid(shape):
    """(N, 3) float64 zyx indices of every voxel of `shape`, in C order."""
    return np.stack(np.meshgrid(*(np.arange(n, dtype=np.float64) for n in shape), indexing="ij"), -1).reshape(-1, 3)


def _cast(v, dtype):
    if dtype == np.float32:
        return v.astype(np.float32)
    info = np.iinfo(dtype)
    r = np.where(v < 0, v - 0.5, v + 0.5)
    r = np.where(np.isnan(r), info.min, r)
    return np.trunc(np.clip(r, info.min, info.max)).astype(dtype)


def _inside(src, c):
    n = np.array(src.shape, dtype=np.float64)[:, None]
    with np.errstate(invalid="ignore"):
        return np.all((c >= 0) & (c <= n - 1), axis=0)


def sample_order0(src, c, cval):
    """src sampled at coordinates c (3, N) as the row-5 kernel does with order 0: src[floor(c + 0.5)], cval outside or
    for NaN."""
    inside = _inside(src, c)
    idx = np.where(inside, np.floor(np.where(inside, c, 0) + 0.5), 0).astype(np.int64)
    out = src[idx[0], idx[1], idx[2]]
    return np.where(inside, out, _cast(np.asarray([cval], dtype=np.float64), src.dtype)[0]).astype(src.dtype)


def sample_order1(src, c, cval):
    """Order 1: trilinear in float64 with neighbours past the last voxel clamped, then scipy's cast."""
    inside = _inside(src, c)
    cc = np.where(inside, c, 0.0)
    n = np.array(src.shape)[:, None]
    i0 = np.floor(cc).astype(np.int64)
    i1 = np.minimum(i0 + 1, n - 1)
    w1 = cc - i0
    w0 = 1.0 - w1
    s = src.astype(np.float64)

    def v(a, b, d):
        return s[a[0], b[1], d[2]]
    a0 = (v(i0, i0, i0) * w0[2] + v(i0, i0, i1) * w1[2]) * w0[1] + (v(i0, i1, i0) * w0[2] + v(i0, i1, i1) * w1[2]) * w1[1]
    a1 = (v(i1, i0, i0) * w0[2] + v(i1, i0, i1) * w1[2]) * w0[1] + (v(i1, i1, i0) * w0[2] + v(i1, i1, i1) * w1[2]) * w1[1]
    val = np.where(inside, a0 * w0[0] + a1 * w1[0], cval)
    return _cast(val, src.dtype)
