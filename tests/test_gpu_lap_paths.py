"""The assignment kernel (K4) against the oracle on every combination of kernels its dispatcher selects.

pm_lap_solve picks its kernels from the column count, the slack nc - nr, max_bid_rounds, algorithm and the device's
opt-in shared memory.  Each case below is named for one combination and asserts the solver's own report of it
(stats `path`, PM_LAP_PATH_* bits), so a case that drifts onto another path (a threshold change, a device with less
shared memory) fails instead of silently testing something else.  The codes are those of a B200 (227 KB opt-in
shared memory per block):

  P1  eps = 0 sparse auction + sparse augmenting paths                  nc <= 10016, slack > 2 %
  P2  squared (dummy rows, eps phases, tight filter) + sparse paths     nc <= 10016, slack <= 2 %
  P3  sparse auction + dense augmenting paths, 16 columns per thread    10017 <= nc <= 16384
  P4  squared + dense augmenting paths (dummy rows read the zero row)   nc >= 10017, slack <= 2 %
  P5  sparse auction, ring in global memory + dense paths, 24 columns   16385 <= nc <= 23040
  P6  dense cooperative auction + dense paths, 24 columns, no squaring  23041 <= nc <= 24576
  P7  max_bid_rounds = 0 or algorithm = 2: dense paths, 8 columns (prices in registers) / 16 columns
  (P8, the refusal above 24576 columns, is host-side: tests/test_abi.py)

Matrices are real shape-context chi^2 matrices built on the GPU (describe_pair + chi2_cost); row subsets and column
slices of one matrix give exact slack values.  The oracle (C shortest augmenting paths, scipy's algorithm) solves the
float64 image of the exact float32 matrix the kernel got.  Asserted per matrix: status 0, every row on a distinct
column, the total equal to the oracle's to 1e-12, and the identical assignment, except where the rows that differ
form an exact tie (their costs sum to the same float64 value both ways).  The oracle solves run in a thread pool
(ctypes releases the GIL); they are what this file spends its time on.
"""
import math
import os
import threading
import time
from concurrent.futures import ThreadPoolExecutor
from contextlib import nullcontext

import numpy as np
import pytest

from platymatch_b200._lib import LAP_PATH

pytestmark = pytest.mark.gpu

STAT_STATUS, STAT_PATH = 4, 13
_B = LAP_PATH
P1 = _B["SPARSE_AUCTION"] | _B["RING_SMEM"] | _B["SAP_SPARSE"]
P2 = _B["SQUARED"] | P1
P3 = _B["SPARSE_AUCTION"] | _B["RING_SMEM"] | _B["SAP_DENSE16"]
P4 = _B["SQUARED"] | P3
P4_RING_GLOBAL = _B["SQUARED"] | _B["SPARSE_AUCTION"] | _B["SAP_DENSE24"]
P5 = _B["SPARSE_AUCTION"] | _B["SAP_DENSE24"]
P6 = _B["DENSE_AUCTION"] | _B["SAP_DENSE24"]
P7_PATHS_8, P7_PATHS_16 = _B["SAP_DENSE8"], _B["SAP_DENSE16"]
P7_DENSE_8, P7_DENSE_16 = _B["DENSE_AUCTION"] | _B["SAP_DENSE8"], _B["DENSE_AUCTION"] | _B["SAP_DENSE16"]


@pytest.fixture(scope="module")
def torch():
    import torch
    torch.cuda.set_device(0)
    return torch


@pytest.fixture(scope="module")
def oracle_pool(O):
    """Oracle solves in parallel, at most two of >= 20000 columns at once (a float64 copy is 3-5 GB)."""
    big = threading.Semaphore(2)

    def solve(c32):
        with big if c32.shape[1] >= 20000 else nullcontext():
            t0 = time.perf_counter()
            _, co = O.linear_sum_assignment(c32.astype(np.float64))
            return co, time.perf_counter() - t0

    with ThreadPoolExecutor(max(2, min(16, len(os.sched_getaffinity(0))))) as pool:
        yield lambda c32: pool.submit(solve, c32)


def _costs(torch, p, variants=(1, 2, 3, 4)):
    """[len(variants), n_moving, ldc] float32 chi^2 matrices (moving variant 1 against fixed variant b), on the GPU."""
    from platymatch_b200 import device as D, pipeline as PL
    dm, df = PL.describe_pair(p["moving"], p["fixed"], 1, 4)
    cost = torch.zeros((len(variants), dm.n, (df.n + 3) // 4 * 4), dtype=torch.float32, device="cuda")
    for q, b in enumerate(variants):
        D.chi2_cost(dm.operand(1), df.operand(b), out=cost[q])
    return cost


def _true_and_false(torch, cost, gt):
    """Hypothesis indices ordered by the cost of the ground-truth matching: [0] the true one, [1] the closest false."""
    n1 = cost.shape[1]
    diag = cost[:, torch.arange(n1, device="cuda"), torch.from_numpy(gt).cuda()].double().sum(1)
    return [int(q) for q in torch.argsort(diag).tolist()]


def _slice(torch, m, nr, nc):
    """Rows [0, nr) x columns [0, nc) of a [n, ldc] matrix as a fresh zero-padded [1, nr, ldc'] problem."""
    out = torch.zeros((1, nr, (nc + 3) // 4 * 4), dtype=torch.float32, device="cuda")
    out[0, :, :nc] = m[:nr, :nc]
    return out


def _solve(cost, nr, nc, max_bid_rounds=2048, algorithm=0):
    """-> per matrix of the batch: (col4row int64, total, status, path), on the host."""
    from platymatch_b200 import device as D
    col, tot, st = D.lap_solve(cost, nr, nc, max_bid_rounds, algorithm)
    col, tot, st = col.cpu().numpy().astype(np.int64), tot.cpu().numpy(), st.cpu().numpy()
    return [(col[q], float(tot[q]), int(st[q, STAT_STATUS]), int(st[q, STAT_PATH])) for q in range(col.shape[0])]


def _check(label, c32, got, oracle, path):
    """got = (col4row, total, status, path) of the kernel; oracle = future of (col4row, seconds) on the same float32
    matrix c32."""
    col, total, status, got_path = got
    co, secs = oracle.result()
    nr, nc = c32.shape
    rows = np.arange(nr)
    diff = np.flatnonzero(col != co)
    print("%-34s path %3d  %5d x %5d  slack %4d  oracle %6.1f s  total %.9f  rows differing %d"
          % (label, got_path, nr, nc, nc - nr, secs, total, diff.size))
    assert status == 0, (label, status)
    assert got_path == path, (label, got_path, path)
    assert col.min() >= 0 and col.max() < nc and np.unique(col).size == nr, label
    opt = c32[rows, co].astype(np.float64).sum()
    assert total == pytest.approx(opt, rel=1e-12), (label, total, opt)
    assert c32[rows, col].astype(np.float64).sum() == pytest.approx(opt, rel=1e-12), label
    if diff.size:       # only an exact tie may differ: the differing rows cost the same both ways
        mine = math.fsum(c32[diff, col[diff]].astype(np.float64))
        theirs = math.fsum(c32[diff, co[diff]].astype(np.float64))
        assert mine == theirs, (label, diff[:16], mine, theirs)


@pytest.mark.parametrize("pair", ["slack1_3-4", "slack2_0-6", "slack43_0-1", "equal_0-1"])
def test_p2_config5_pairs_batched_and_single(O, torch, oracle_pool, pair):
    """P2 at the size of the all-pairs configuration (specimens of ~7.8k nuclei): all four hypothesis matrices of a
    pair, solved as one batch of 4 and one by one; batch and single results are bit-identical."""
    from platymatch_b200.synthetic import make_specimens
    tag, ij = pair.split("_", 1)
    s, t = (int(x) for x in ij.split("-"))
    spec = make_specimens(max(s, t) + 1, 8000, seed=0, vary=0 if tag == "equal" else 0.05)
    a, b = spec[s]["points"], spec[t]["points"]
    mov, fix = (a, b) if a.shape[1] <= b.shape[1] else (b, a)
    nr, nc = mov.shape[1], fix.shape[1]
    assert nc - nr == {"slack1": 1, "slack2": 2, "slack43": 43, "equal": 0}[tag]
    cost = _costs(torch, {"moving": mov, "fixed": fix})
    batch = _solve(cost, nr, nc)
    single = [_solve(cost[q:q + 1], nr, nc)[0] for q in range(4)]
    c32 = [cost[q, :, :nc].cpu().numpy() for q in range(4)]
    futs = [oracle_pool(c) for c in c32]
    for q in range(4):
        assert np.array_equal(batch[q][0], single[q][0]), (pair, q)
        assert batch[q][1:] == single[q][1:], (pair, q, batch[q][1:], single[q][1:])
        _check("P2 %s hyp %d" % (pair, q), c32[q], batch[q], futs[q], P2)


def test_square_slack_boundary_at_8000_columns(O, torch, oracle_pool, monkeypatch):
    """Slack 160 = 2 % of 8000 columns is squared (P2), slack 161 is not (P1); forcing eps-scaling on the 161-slack
    problem (PM_LAP_EPS_SCALING=1) returns the identical assignment."""
    from platymatch_b200.synthetic import make_pair
    p = make_pair(8000, dropout=0.0)
    cost = _costs(torch, p)
    m = cost[_true_and_false(torch, cost, p["gt_fixed_index"])[0]]
    probs = {nr: _slice(torch, m, nr, 8000) for nr in (7840, 7839)}
    got = {nr: _solve(probs[nr], nr, 8000)[0] for nr in probs}
    monkeypatch.setenv("PM_LAP_EPS_SCALING", "1")
    forced = _solve(probs[7839], 7839, 8000)[0]
    monkeypatch.delenv("PM_LAP_EPS_SCALING")
    c32 = {nr: probs[nr][0, :, :8000].cpu().numpy() for nr in probs}
    futs = {nr: oracle_pool(c32[nr]) for nr in probs}
    _check("P2 7840 rows (slack 160)", c32[7840], got[7840], futs[7840], P2)
    _check("P1 7839 rows (slack 161)", c32[7839], got[7839], futs[7839], P1)
    _check("P2 7839 rows, eps-scaling forced", c32[7839], forced, futs[7839], P2)
    assert np.array_equal(forced[0], got[7839][0])


def test_p3_sparse_auction_dense_paths_12k(O, torch, oracle_pool):
    """P3: 10800 x 12000, true and one false hypothesis; 9000 rows x 10016 / 10020 columns of the true one lie on
    either side of the largest column count whose sparse augmenting paths fit in shared memory (P1 | P3)."""
    from platymatch_b200.synthetic import make_pair
    p = make_pair(12000)
    cost = _costs(torch, p)
    true_q, false_q = _true_and_false(torch, cost, p["gt_fixed_index"])[:2]
    nr = cost.shape[1]
    cases = [("P3 10800 x 12000 true", cost[true_q:true_q + 1], nr, 12000, P3),
             ("P3 10800 x 12000 false", cost[false_q:false_q + 1], nr, 12000, P3),
             ("P1 9000 x 10016", _slice(torch, cost[true_q], 9000, 10016), 9000, 10016, P1),
             ("P3 9000 x 10020", _slice(torch, cost[true_q], 9000, 10020), 9000, 10020, P3)]
    _run(torch, oracle_pool, cases)


def test_p4_squared_dense_paths(O, torch, oracle_pool):
    """P4 (never run before this test): 12000 x 12000 and its 11880-row slice (slack 1 %), true and one false
    hypothesis; the 19800-row slice of a 20000-nucleus pair, whose squared problem keeps its ring in global memory."""
    from platymatch_b200.synthetic import make_pair
    p = make_pair(12000, dropout=0.0)
    cost = _costs(torch, p)
    true_q, false_q = _true_and_false(torch, cost, p["gt_fixed_index"])[:2]
    cases = []
    for tag, q in (("true", true_q), ("false", false_q)):
        cases.append(("P4 12000 x 12000 " + tag, cost[q:q + 1], 12000, 12000, P4))
        cases.append(("P4 11880 x 12000 " + tag, _slice(torch, cost[q], 11880, 12000), 11880, 12000, P4))
    p = make_pair(20000, seed=2, dropout=0.0)
    cost = _costs(torch, p)
    true_q = _true_and_false(torch, cost, p["gt_fixed_index"])[0]
    cases.append(("P4 19800 x 20000 true", _slice(torch, cost[true_q], 19800, 20000), 19800, 20000, P4_RING_GLOBAL))
    _run(torch, oracle_pool, cases)


def test_p5_ring_in_global_memory_false_hypothesis(O, torch, oracle_pool):
    """P5: 18000 x 20000, a false hypothesis (price wars and list refreshes; the true one is the config-4 test's)."""
    from platymatch_b200.synthetic import make_pair
    p = make_pair(20000, seed=2)
    cost = _costs(torch, p)
    false_q = _true_and_false(torch, cost, p["gt_fixed_index"])[1]
    _run(torch, oracle_pool, [("P5 18000 x 20000 false", cost[false_q:false_q + 1], 18000, 20000, P5)])


def test_p6_dense_cooperative_auction(O, torch, oracle_pool):
    """P6: the prices no longer fit in shared memory: dense grid-wide auction, no squaring.  24576 columns is the
    largest problem the solver accepts.  Seed 1 makes the 24000 pair registrable; the 24576 pair has no true
    hypothesis, and its solve (the one with the cheapest ground-truth matching) is this file's longest oracle run."""
    from platymatch_b200.synthetic import make_pair
    cases = []
    for n in (24000, 24576):
        p = make_pair(n, seed=1)
        cost = _costs(torch, p)
        true_q = _true_and_false(torch, cost, p["gt_fixed_index"])[0]
        nr = cost.shape[1]
        cases.append(("P6 %d x %d" % (nr, n), cost[true_q:true_q + 1].clone(), nr, n, P6))
        del cost
    _run(torch, oracle_pool, cases)


def test_p7_augmenting_paths_only_and_dense_auction(O, torch, oracle_pool):
    """P7 through the public numpy API: max_bid_rounds = 0 (augmenting paths only) and algorithm = 2 (dense auction)
    at 7400 x 8192 (8 columns per thread, prices in registers) and 7400 x 8193 (16 columns per thread)."""
    from platymatch_b200.lap import linear_sum_assignment
    from platymatch_b200.synthetic import make_pair
    p = make_pair(9000)
    cost = _costs(torch, p)
    m = cost[_true_and_false(torch, cost, p["gt_fixed_index"])[0]]
    for nc, paths_only, dense in ((8192, P7_PATHS_8, P7_DENSE_8), (8193, P7_PATHS_16, P7_DENSE_16)):
        c32 = m[:7400, :nc].cpu().numpy()
        fut = oracle_pool(c32)
        for label, kw, path in (("paths only", dict(max_bid_rounds=0), paths_only),
                                ("dense auction", dict(algorithm=2), dense)):
            r, c, st = linear_sum_assignment(c32, return_stats=True, **kw)
            assert np.array_equal(r, np.arange(7400))          # (a status other than 0 raises)
            _check("P7 7400 x %d %s" % (nc, label), c32, (c, st["total"], 0, st["path"]), fut, path)


def _run(torch, oracle_pool, cases):
    """cases: (label, cost [1, nr, ldc] on the GPU, nr, nc, expected path).  All GPU solves first, then the oracle
    solves of the case list in parallel."""
    got, futs, c32 = [], [], []
    for label, cost, nr, nc, path in cases:
        got.append(_solve(cost, nr, nc)[0])
        c32.append(cost[0, :, :nc].cpu().numpy())
        futs.append(oracle_pool(c32[-1]))
    for (label, _, _, _, path), c, g, f in zip(cases, c32, got, futs):
        _check(label, c, g, f, path)
