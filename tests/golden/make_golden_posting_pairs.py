"""Samples of the reference's seven saved posting pairs (fixtures/{lhs,rhs,mask}_<n>.npy of the reference tree,
up to 3.1M words a side, 55 MB in all) and what the REAL reference's intersect / intersect_with_adjacents
return on each sample.  Writes tests/golden/posting_pairs.npz.

    python oracle/build_ref.py && python tests/golden/make_golden_posting_pairs.py <reference tree>/fixtures

A pair at most CAP words a side is kept whole.  Otherwise lhs is cut to a seeded window of CAP consecutive
words, and rhs to the words whose masked key falls inside that window's key range (one block either side):
all of those that equal or neighbour (one block after or before) an lhs key, plus a seeded sample of the
rest up to CAP.  Every sample keeps the pair's order, duplicates and real key structure.
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

from oracle.build_ref import import_reference  # noqa: E402

SUFFIXES = (128, 185, 24179, 27685, 44358, 45907, 90596)
CAP = 1024


def sample_pair(lhs, rhs, mask, rng):
    if len(lhs) > CAP:
        start = int(rng.integers(0, len(lhs) - CAP + 1))
        lhs = lhs[start:start + CAP]
    if len(rhs) <= CAP:
        return lhs, rhs
    step = (~mask + np.uint64(1)) & mask               # one block: the lowest bit of the mask
    lm, rm = lhs & mask, rhs & mask
    lo = lm[0] - step if lm[0] >= step else np.uint64(0)
    idx = np.arange(np.searchsorted(rm, lo, "left"), np.searchsorted(rm, lm[-1] + step, "right"))
    if len(idx) > CAP:
        near = np.isin(rm[idx], np.concatenate((lm - step, lm, lm + step)))
        rest = idx[~near]
        extra = rng.choice(rest, min(len(rest), max(0, CAP - int(near.sum()))), replace=False)
        idx = np.sort(np.concatenate((idx[near], extra)))
    return lhs, rhs[idx]


def main(fixtures):
    import_reference()
    from searcharray.roaringish import intersect
    from searcharray.roaringish.intersect import intersect_with_adjacents
    rng = np.random.default_rng(20261017)
    out = {}
    for n in SUFFIXES:
        lhs = np.load(os.path.join(fixtures, f"lhs_{n}.npy"))
        rhs = np.load(os.path.join(fixtures, f"rhs_{n}.npy"))
        mask = np.load(os.path.join(fixtures, f"mask_{n}.npy"))
        lhs, rhs = sample_pair(lhs, rhs, np.uint64(mask), rng)
        li, ri = intersect(lhs, rhs, mask=mask)
        adj = intersect_with_adjacents(lhs, rhs, mask=mask)
        out.update({f"{n}.lhs": lhs, f"{n}.rhs": rhs, f"{n}.mask": np.uint64(mask),
                    f"{n}.intersect.lhs_idx": li, f"{n}.intersect.rhs_idx": ri})
        out.update({f"{n}.with_adjacents.{i}": np.asarray(a, dtype=np.uint64) for i, a in enumerate(adj)})
        print(n, len(lhs), len(rhs), len(li), [len(a) for a in adj])
    path = os.path.join(HERE, "posting_pairs.npz")
    np.savez_compressed(path, **out)
    print(os.path.getsize(path))


if __name__ == "__main__":
    main(sys.argv[1])
