"""The chi^2 cost kernel's per-warp bin lists (16 rows x 128 columns): every entry against the oracle (1e-5 relative)
and against a float64 restatement of the kernel's own formulation on its float32 operands (1e-6 relative), on inputs
that reach what the headline workload does not: warps of one CTA with disjoint supports (some with no bin in common
with the columns), sizes that are not multiples of 16 or 128, integer counts, row sub-ranges, and the swapped
registration (rows are fixed nuclei)."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _f32_operand(h):
    """The kernel's operand values: float32 histograms, as pm_chi2_operand_f32 takes them."""
    return np.asarray(h, dtype=np.float32)


def _restated(a32, b32):
    """0.5 sum_k (a - b)^2 / (a + b) over the bins where a != b, in float64 on the float32 operands."""
    a, b = a32.astype(np.float64), b32.astype(np.float64)
    out = np.empty((a.shape[0], b.shape[0]))
    for i0 in range(0, a.shape[0], 32):
        x, y = a[i0:i0 + 32, None, :], b[None, :, :]
        s = x + y
        t = np.where(x != y, (x - y) ** 2 / np.where(s > 0, s, 1.0), 0.0)
        out[i0:i0 + 32] = 0.5 * t.sum(-1)
    return out


def _check(got, a32, b32, O):
    ref64 = _restated(a32, b32)
    oracle = O.unary_distance_matrix(a32.astype(np.float64), b32.astype(np.float64))
    for ref, tol in ((ref64, 1e-6), (oracle, 1e-5)):
        nz = ref > 0
        assert np.all(got[~nz] == 0.0)
        rel = float((np.abs(got[nz] - ref[nz]) / ref[nz]).max())
        assert rel < tol, (rel, tol)


def _hist(rng, n, bins_of_row):
    c = np.zeros((n, 360))
    for i in range(n):
        bins = np.asarray(bins_of_row(i))
        c[i, bins] = rng.integers(0, 4, size=len(bins))
        c[i, bins[rng.integers(len(bins))]] += 1                      # no empty histogram
    return c / c.sum(1, keepdims=True)


def _supports(rng, n1, n2):
    """Row blocks of 16 on four different supports: warps 0 and 4 of a CTA share nothing with any column, warps 1, 5
    share one bin, the others overlap the columns in odd and even numbers of bins."""
    sets = [np.arange(300, 340), np.arange(0, 41), np.arange(40, 81), np.arange(100, 221)]
    a = _hist(rng, n1, lambda i: sets[(i // 16) % 4])
    b = _hist(rng, n2, lambda j: np.arange(40, 201) if (j // 128) % 2 == 0 else np.arange(50, 150, 3))
    return a, b


@pytest.mark.parametrize("n1,n2", [(300, 391), (17, 1), (129, 130)])
def test_warps_with_disjoint_supports(O, n1, n2):
    import torch
    from platymatch_b200 import device as D
    rng = np.random.default_rng(n1 + 7 * n2)
    a, b = _supports(rng, n1, n2)
    a32, b32 = _f32_operand(a), _f32_operand(b)
    A, B = D.chi2_operand(torch.from_numpy(a32).cuda()), D.chi2_operand(torch.from_numpy(b32).cuda())
    got = D.chi2_cost(A, B)[:, :n2].cpu().numpy()
    _check(got, a32, b32, O)
    # the fine masks: one per 16 operand columns, OR-ing to the 128-block mask
    fine = A.fine.cpu().numpy().view(np.uint32)
    bits = np.unpackbits(fine.view(np.uint8), axis=1, bitorder="little")[:, :360].astype(bool)
    want = np.zeros_like(bits)
    for g in range((n1 + 15) // 16):
        want[g] = (a[g * 16:(g + 1) * 16] > 0).any(0)
    assert np.array_equal(bits, want)
    coarse = np.bitwise_or.reduce(fine.reshape(-1, 8, 12), axis=1)
    assert np.array_equal(coarse, A.mask.cpu().numpy().view(np.uint32))


def test_integer_counts(O):
    """Operands from integer counts (normalised by the row total in one float32 rounding) on disjoint warp supports."""
    import torch
    from platymatch_b200 import device as D
    rng = np.random.default_rng(5)
    n1, n2 = 300, 391
    a, b = _supports(rng, n1, n2)
    ca = rng.integers(0, 3, size=(n1, 360)) * (a > 0)
    ca[np.arange(n1), a.argmax(1)] += 1
    cb = rng.integers(0, 3, size=(n2, 360)) * (b > 0)
    cb[np.arange(n2), b.argmax(1)] += 1
    A = D.chi2_operand(torch.from_numpy(ca.astype(np.int32)).cuda())
    B = D.chi2_operand(torch.from_numpy(cb.astype(np.int32)).cuda())
    got = D.chi2_cost(A, B)[:, :n2].cpu().numpy()
    a32 = (ca.astype(np.float32) / ca.sum(1, keepdims=True).astype(np.float32)).astype(np.float32)
    b32 = (cb.astype(np.float32) / cb.sum(1, keepdims=True).astype(np.float32)).astype(np.float32)
    _check(got, a32, b32, O)


def test_row_ranges(O):
    import torch
    from platymatch_b200 import device as D
    rng = np.random.default_rng(3)
    n1, n2 = 300, 391
    a, b = _supports(rng, n1, n2)
    a32, b32 = _f32_operand(a), _f32_operand(b)
    A, B = D.chi2_operand(torch.from_numpy(a32).cuda()), D.chi2_operand(torch.from_numpy(b32).cuda())
    full = D.chi2_cost(A, B)[:, :n2].cpu().numpy()
    for r0, r1 in ((0, 128), (128, 300), (256, 300)):
        part = D.chi2_cost(A, B, row_begin=r0, row_end=r1)[:, :n2].cpu().numpy()
        assert part.shape[0] == r1 - r0
        assert np.array_equal(part, full[r0:r1])
        _check(part, a32[r0:r1], b32, O)


def test_described_pair(O):
    """Shape-context descriptors of a synthetic pair (real supports, 1800 x 2000)."""
    from platymatch_b200 import device as D, pipeline as P
    from platymatch_b200.synthetic import make_pair
    p = make_pair(2000, seed=21)
    dm, df = P.describe_pair(p["moving"], p["fixed"], 1, 4)
    got = D.chi2_cost(dm.operand(1), df.operand(3))[:, :df.n].cpu().numpy()
    ca, cb = dm.counts[0].cpu().numpy(), df.counts[2].cpu().numpy()
    a32 = (ca.astype(np.float32) / ca.sum(1, keepdims=True).astype(np.float32)).astype(np.float32)
    b32 = (cb.astype(np.float32) / cb.sum(1, keepdims=True).astype(np.float32)).astype(np.float32)
    _check(got, a32, b32, O)


def test_swapped_registration_cost(O):
    """More moving than fixed nuclei: rows are fixed nuclei, the matrices the assignment sees are the oracle's
    transposed problem."""
    from platymatch_b200 import pipeline as P
    from platymatch_b200.synthetic import make_pair
    p = make_pair(600, seed=11)
    moving, fixed = p["fixed"], p["moving"]             # 600 moving, 540 fixed
    dm, df = P.describe_pair(moving, fixed, 1, 4)
    res = P.register_described(dm, df, ransac_trials=200, keep_cost=True)
    cost = res["cost"].cpu().numpy()
    mc, md = O.get_centroid(moving, False), O.get_mean_distance(moving, False)
    fc, fd = O.get_centroid(fixed, False), O.get_mean_distance(fixed, False)
    um, uf = O.get_unary(mc, md, moving, "moving"), O.get_unary(fc, fd, fixed, "fixed")
    for q, (a, b) in enumerate(P.HYPOTHESES_DISTINCT):
        U = O.unary_distance_matrix(uf[b - 1], um[a - 1])
        G = cost[q][:, :moving.shape[1]]
        nz = U > 0
        assert np.all(G[~nz] == 0.0)
        assert float((np.abs(G[nz] - U[nz]) / U[nz]).max()) < 1e-5
