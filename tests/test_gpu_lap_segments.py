"""Augmenting paths over the candidate lists (pm_lap_sap_sparse_kernel) keep, per segment of 256 columns, the
smallest tentative distance of its unscanned columns.  A Dijkstra step must still finalise the globally lowest
column among equal distances, so these matrices are built around exact ties that straddle segment boundaries.
Each has one optimal assignment, which must be the oracle's."""
import numpy as np
import pytest

from platymatch_b200._lib import LAP_PATH, LAP_STAT

pytestmark = pytest.mark.gpu

SEG = 256


@pytest.fixture(scope="module")
def torch():
    import torch
    torch.cuda.set_device(0)
    return torch


def _tied_slack_matrix(nr, nc, seed):
    """Background costs 3..6 (integers: exact distance ties everywhere), every row with one zero column of its own,
    and pairs of rows that compete for a zero column next to a segment boundary.  One row of the pair has a second
    choice of cost 1 on the other side of the boundary (its partner's is 2), tied with a taken column of cost 1 on
    this side, so exactly one assignment is optimal (cost 1 per pair) and the row that loses the shared column
    reaches it by augmenting paths through distances tied across the boundary."""
    rng = np.random.default_rng(seed)
    cost = rng.integers(3, 7, size=(nr, nc)).astype(np.float64)
    near = [b + o for b in range(SEG, nc, SEG) for o in range(-6, 6) if 0 <= b + o < nc]
    far = np.setdiff1d(np.arange(nc), near)
    rows = rng.permutation(nr)
    r = 0
    for b in range(SEG, nc - 6, SEG):
        for o in range(0, 6, 2):
            a, z = rows[r], rows[r + 1]
            shared, second_a, second_z = b - 1 - o, b + o, b + 1 + o
            cost[a, shared] = cost[z, shared] = 0.0
            cost[a, second_a], cost[z, second_z] = 1.0, 2.0        # optimum: z takes the shared column, a goes across
            decoy, w = b - 2 - o, rows[r + 2]                       # the tie at distance 1 on the lower side: a column
            cost[a, decoy] = cost[z, decoy] = 1.0                   # whose own row w has no other choice below 3
            cost[w, decoy] = 0.0
            r += 3
    for i, j in zip(rows[r:], rng.choice(far, size=nr - r, replace=False)):
        cost[i, j] = 0.0
    return cost, r // 3


@pytest.mark.parametrize("nr,nc,rounds", [(600, 1100, 1), (600, 1100, 2048), (2000, 2600, 1)])
def test_distance_ties_across_segment_boundaries(O, torch, nr, nc, rounds):
    from platymatch_b200.lap import linear_sum_assignment
    cost, pairs = _tied_slack_matrix(nr, nc, seed=nr + nc + rounds)
    r, c, st = linear_sum_assignment(cost, return_stats=True, max_bid_rounds=rounds)
    ro, co = O.linear_sum_assignment(cost)
    assert st["path"] & LAP_PATH["SAP_SPARSE"], st
    assert cost[ro, co].sum() == pairs                          # the planted optimum: cost 1 per competing pair
    assert st["total"] == pytest.approx(pairs, abs=1e-9), st
    assert np.array_equal(c, co), int((c != co).sum())
    assert set(st) >= {k.lower() for k in LAP_STAT}, st
