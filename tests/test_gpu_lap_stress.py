"""Assignment kernel (K4) under the conditions round 1 left untested (VERDICT r1 weak #5/#9, ADVICE r1):

  * problems WITHOUT slack columns (nr == nc), where an epsilon = 0 auction degenerates into sequential price wars:
    solved with eps-scaling phases + the exact finish; cost and assignment must equal the oracle's / scipy's;
  * the asynchronous auction's ticket ring / patience spin / bid caps under reduced residency and hostile knobs
    (PM_LAP_BULK_PATIENCE=0, one bulk CTA, far too many bulk CTAs, tiny bid budgets);
  * several solves in flight on different streams from different host threads (different problem sizes: the
    shared-memory attribute race of ADVICE r1), identical cost to the sequential run.
"""
import threading

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def torch():
    import torch
    torch.cuda.set_device(0)
    return torch


def _chi2_matrix(O, n, dropout, seed, variant=1):
    """A real shape-context cost matrix (float64 oracle values) of a synthetic pair: the structure the kernel is built for."""
    from platymatch_b200.synthetic import make_pair
    p = make_pair(n, seed=seed, dropout=dropout)
    m, f = p["moving"], p["fixed"]
    mc, fc = O.get_centroid(m, False), O.get_centroid(f, False)
    md, fd = O.get_mean_distance(m, False), O.get_mean_distance(f, False)
    um = O.normalise_counts(O.shape_context_counts(m.T, mc, md, O.pca_first_axis(m.T), 1)[0])
    uf = O.normalise_counts(O.shape_context_counts(f.T, fc, fd, O.pca_first_axis(f.T), variant)[0])
    return O.unary_distance_matrix(um, uf)


def _solve_and_check(O, cost, **kw):
    from platymatch_b200.lap import linear_sum_assignment
    c32 = np.asarray(cost, dtype=np.float32).astype(np.float64)
    r, c, st = linear_sum_assignment(cost, return_stats=True, **kw)
    ro, co = O.linear_sum_assignment(c32)
    assert len(np.unique(c)) == len(c) == min(cost.shape)
    assert c32[r, c].sum() == pytest.approx(c32[ro, co].sum(), rel=1e-12, abs=1e-12), st
    return c, co, st


@pytest.mark.parametrize("n,variant", [(64, 1), (300, 1), (1000, 1), (1000, 2), (3000, 1), (3000, 3)])
def test_square_chi2_matrices_exact(O, torch, n, variant):
    """nr == nc on shape-context matrices (true and false hypotheses): exact optimum, identical assignment."""
    cost = _chi2_matrix(O, n, 0.0, seed=n + variant, variant=variant)
    assert cost.shape[0] == cost.shape[1]
    c, co, st = _solve_and_check(O, cost)
    assert np.array_equal(c, co), int((c != co).sum())
    if n >= 1000:                       # eps-scaling keeps the work near the slack-column case: no 100-bids-per-row price wars
        assert st["bids"] < 150 * n, st


@pytest.mark.parametrize("kind", ["random", "integer_ties", "constant", "diagonal", "negative", "few_good_columns"])
def test_square_structured_matrices(O, torch, kind):
    rng = np.random.default_rng(len(kind))
    n = 400
    if kind == "random":
        cost = rng.random((n, n))
    elif kind == "integer_ties":
        cost = rng.integers(0, 4, size=(n, n)).astype(float)
    elif kind == "constant":
        cost = np.full((n, n), 2.5)
    elif kind == "diagonal":
        cost = np.ones((n, n)); cost[np.arange(n), rng.permutation(n)] = 0.0
    elif kind == "negative":
        cost = rng.normal(size=(n, n))
    else:
        cost = rng.random((n, n)) + 5.0
        cost[:, :20] -= 5.0
    c, co, st = _solve_and_check(O, cost)
    if kind in ("random", "negative", "diagonal"):
        assert np.array_equal(c, co)


@pytest.mark.parametrize("slack", [1, 3, 17, 120])
def test_small_slack_exact(O, torch, slack):
    """A handful of slack columns (specimens of nearly equal size, BASELINE config 5)."""
    cost = _chi2_matrix(O, 1500, slack / 1500.0, seed=40 + slack)
    assert cost.shape[1] - cost.shape[0] == slack
    c, co, st = _solve_and_check(O, cost)
    assert np.array_equal(c, co)


@pytest.mark.parametrize("env", [{"PM_LAP_BULK_PATIENCE": "0"}, {"PM_LAP_BULK_CTAS": "1"}, {"PM_LAP_BULK_CTAS": "400"},
                                 {"PM_LAP_BULK_STOP": "1"}, {"PM_LAP_STOP_LIVE": "0"}, {"PM_LAP_STOP_LIVE": "31"},
                                 {"PM_LAP_EPS_SCALING": "0"}, {"PM_LAP_EPS_SCALING": "1"}])
def test_auction_knobs_keep_exactness(O, torch, monkeypatch, env):
    """Every tuning knob keeps the exact optimum.  PM_LAP_EPS_SCALING=1 squares the 1080 x 1200 problem as well
    (120 dummy rows, far above the 2 % slack at which it is squared by default)."""
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    for n, dropout in ((1200, 0.1), (700, 0.0)):
        cost = _chi2_matrix(O, n, dropout, seed=7)
        c, co, st = _solve_and_check(O, cost)
        assert np.array_equal(c, co), (env, n)


@pytest.mark.parametrize("rounds", [1, 2, 5])
def test_tiny_bid_budgets_leave_the_rest_to_augmenting_paths(O, torch, rounds):
    for n, dropout in ((900, 0.1), (500, 0.0)):
        cost = _chi2_matrix(O, n, dropout, seed=11)
        c, co, st = _solve_and_check(O, cost, max_bid_rounds=rounds)
        assert np.array_equal(c, co)


def test_solves_in_flight_from_threads(O, torch):
    """Three host threads, three streams, problems of different sizes (square and wide) solved concurrently, three
    times each: every result equals the sequential one (the kernels' shared-memory limits are per-process state,
    the ticket rings compete for SMs)."""
    from platymatch_b200 import device as D
    rng = np.random.default_rng(0)
    shapes = [(900, 1000), (1300, 1300), (700, 1900)]
    costs = [_chi2_matrix(O, nc, 1.0 - nr / nc, seed=50 + k) for k, (nr, nc) in enumerate(shapes)]
    dev = []
    for cst in costs:
        nr, nc = cst.shape
        buf = np.zeros((1, nr, (nc + 3) // 4 * 4), dtype=np.float32)
        buf[0, :, :nc] = cst
        dev.append(torch.from_numpy(buf).cuda())
    seq = [D.lap_solve(d, c.shape[0], c.shape[1]) for d, c in zip(dev, costs)]
    torch.cuda.synchronize()
    results, errors = {}, []

    def worker(k):
        try:
            with torch.cuda.stream(torch.cuda.Stream()):
                out = []
                for rep in range(3):
                    col, tot, _ = D.lap_solve(dev[k], costs[k].shape[0], costs[k].shape[1])
                    out.append((col.clone(), tot.clone()))
                torch.cuda.current_stream().synchronize()
                results[k] = out
        except Exception as e:
            errors.append(e)

    ts = [threading.Thread(target=worker, args=(k,)) for k in range(3)]
    [t.start() for t in ts]
    [t.join() for t in ts]
    assert not errors, errors
    for k in range(3):
        for col, tot in results[k]:
            assert tot.item() == pytest.approx(seq[k][1].item(), rel=1e-12)
            assert torch.equal(col, seq[k][0])
