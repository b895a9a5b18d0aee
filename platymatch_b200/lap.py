"""GPU replacement for `scipy.optimize.linear_sum_assignment` as used at reference
_dock_widget.py:604-611 (same return convention: rows ascending, min(nr, nc) pairs)."""
import numpy as np

from . import device as D

__all__ = ["linear_sum_assignment"]


def linear_sum_assignment(cost_matrix, maximize=False, return_stats=False, max_bid_rounds=2048, algorithm=0):
    """Minimum-cost assignment of a dense (nr, nc) matrix -> (row_ind, col_ind) int64 arrays.

    The matrix is solved as float32 values with float64 duals (optimal for the float32-rounded
    matrix).  Tall matrices are solved through the transpose, as scipy does.
    algorithm: 0 auto, 1 sparse asynchronous auction, 2 dense grid-wide auction (PM_LAP_ALGO_*).
    return_stats adds the solver's statistics; `path` holds the PM_LAP_PATH_* bits of the kernels that ran
    (platymatch_b200._lib.LAP_PATH).
    """
    torch = D._torch()
    c = np.asarray(cost_matrix)
    if c.ndim != 2:
        raise ValueError("expected a matrix (2-D array), got a %d array" % c.ndim)
    if c.size == 0:
        z = np.zeros(0, dtype=np.int64)
        return (z, z, {}) if return_stats else (z, z)
    if not np.all(np.isfinite(c)):
        raise ValueError("matrix contains invalid numeric entries")
    if maximize:
        c = -c
    if c.dtype != np.float32 and c.size <= (1 << 22):
        # the kernel solves the float32 image of the matrix (exactly); say so when that image merges distinct costs
        # (integer costs above 2^24, huge dynamic range), because scipy's float64 optimum can then be a different one
        c32 = c.astype(np.float32)
        if np.unique(c32).size < np.unique(c).size and not np.array_equal(c32.astype(np.float64), c):
            import warnings
            warnings.warn("linear_sum_assignment: float32 rounding merges distinct cost values; the result is optimal "
                          "for the rounded matrix and may differ from a float64 solve near ties", RuntimeWarning,
                          stacklevel=2)
    transposed = c.shape[0] > c.shape[1]
    if transposed:
        c = c.T
    nr, nc = c.shape
    ldc = (nc + 3) // 4 * 4
    buf = np.zeros((1, nr, ldc), dtype=np.float32)
    buf[0, :, :nc] = c
    col4row, total, stats = D.lap_solve(torch.from_numpy(buf).cuda(), nr, nc, max_bid_rounds, algorithm)
    col = col4row[0].cpu().numpy().astype(np.int64)
    st = stats[0].cpu().numpy()
    if st[4] != 0:
        raise ValueError("cost matrix is infeasible")
    rows = np.arange(nr, dtype=np.int64)
    if transposed:
        order = np.argsort(col)
        rows, col = col[order], rows[order]
    if return_stats:
        return rows, col, dict(total=float(total.item()), bid_rounds=int(st[0]), rows_after_bidding=int(st[1]),
                               augmentations=int(st[2]), dijkstra_steps=int(st[3]), bids=int(st[5]),
                               refreshes=int(st[6]), retries=int(st[7]), parked=int(st[8]),
                               refresh_cycles=int(st[9]), auction_cycles=int(st[10]), bulk_bids=int(st[11]),
                               sap_dense_relax=int(st[12]), path=int(st[13]))
    return rows, col
