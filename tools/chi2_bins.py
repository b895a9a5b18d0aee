"""Bins the chi^2 cost kernel evaluates in full per (row, column) pair at the headline size, from the operands'
own masks: the per-warp lists (fine masks of 16 row-ordered rows x the 128-column block masks) against one list per
128 x 128 tile of rows in natural order.  Needs a GPU (the operands are built there).

    python tools/chi2_bins.py [n_fixed] [slot]
"""
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from platymatch_b200 import pipeline as P                     # noqa: E402
from platymatch_b200.synthetic import make_pair               # noqa: E402


def bits(mask):
    m = mask.cpu().numpy().view(np.uint32)
    return np.unpackbits(m.view(np.uint8), axis=1, bitorder="little")[:, :360].astype(np.int64)


def per_pair(rows, cols, rows_per_block, n1, n2):
    """Mean over all n1 x n2 pairs of the bins populated on both the pair's row block and its 128-column block."""
    both = bits(rows) @ bits(cols).T
    wr = np.minimum(rows_per_block, n1 - rows_per_block * np.arange(both.shape[0])).clip(0)
    wc = np.minimum(128, n2 - 128 * np.arange(both.shape[1])).clip(0)
    return float((wr[:, None] * wc[None, :] * both).sum() / (n1 * n2))


def main():
    n_fixed = int(sys.argv[1]) if len(sys.argv) > 1 else 8000
    slot = int(sys.argv[2]) if len(sys.argv) > 2 else 0
    p = make_pair(n_fixed, seed=n_fixed + 97 * slot)
    dm, df = P.describe_pair(p["moving"], p["fixed"], 1, 4)
    A = dm.operand(1)
    print("%d x %d, slot %d" % (dm.n, df.n, slot))
    for b in range(1, 5):
        B = df.operand(b)
        print("hypothesis (1,%d): both-side bins per pair  128 x 128 tile lists %.1f  per-warp 16 x 128 lists (the kernel) %.1f"
              % (b, per_pair(A.mask, B.mask, 128, dm.n, df.n), per_pair(A.fine, B.mask, 16, dm.n, df.n)))


if __name__ == "__main__":
    main()
