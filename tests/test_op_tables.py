"""CPU: the oracle's C restatement of the reference's native ops (oracle/sa_oracle.c) against the
known-answer tables of the reference's own op tests (test/test_snp_ops.py, test/test_bitcount64.py;
extracted by tests/golden/make_golden_op_tables.py), and against the reference's output on samples of its
seven saved posting pairs."""
import hashlib
import json
import os

import numpy as np
import pytest

from conftest import GOLDEN

T = json.load(open(os.path.join(GOLDEN, "op_tables.json")))
P = np.load(os.path.join(GOLDEN, "posting_pairs.npz"))
U = lambda xs: np.asarray(xs, dtype=np.uint64)


def digest(a):
    return hashlib.sha256(np.ascontiguousarray(a, dtype=np.uint64).tobytes()).hexdigest()


@pytest.mark.parametrize("sc", T["intersect"], ids=[s["name"] for s in T["intersect"]])
def test_intersect_table(sc):
    from oracle import ops
    lhs, rhs, mask = U(sc["lhs"]), U(sc["rhs"]), np.uint64(sc["mask"])
    li, ri = ops.intersect(lhs, rhs, mask=mask)
    assert np.array_equal(lhs[li.astype(np.int64)] & mask, U(sc["expected"]))
    assert np.array_equal(li, U(sc["lhs_idx"])) and np.array_equal(ri, U(sc["rhs_idx"]))
    lk, rk = ops.intersect(lhs, rhs, mask=mask, drop_duplicates=False)
    assert np.array_equal(lk, U(sc["keep_lhs_idx"])) and np.array_equal(rk, U(sc["keep_rhs_idx"]))
    got = ops.intersect_with_adjacents(lhs, rhs, mask=mask)
    for g, w in zip(got, sc["with_adjacents"]):
        assert np.array_equal(g, U(w))
    # strided inputs (reference test_intersect_strided): same answers as on a contiguous copy
    ls, rs = lhs[::2], rhs[::2]
    li2, _ = ops.intersect(ls, rs, mask=mask)
    assert np.array_equal(ls[li2.astype(np.int64)] & mask, np.intersect1d(ls & mask, rs & mask))


@pytest.mark.parametrize("sc", T["adjacent"], ids=[s["name"] for s in T["adjacent"]])
def test_adjacent_table(sc):
    from oracle import ops
    lhs, rhs, mask = U(sc["lhs"]), U(sc["rhs"]), np.uint64(sc["mask"])
    if sc["delta"] == -1:
        ri, li = ops.adjacent(rhs, lhs, mask)
    else:
        li, ri = ops.adjacent(lhs, rhs, mask)
    assert np.array_equal(li, U(sc["lhs_idx"])) and np.array_equal(ri, U(sc["rhs_idx"]))


@pytest.mark.parametrize("sc", T["merge"], ids=[s["name"] for s in T["merge"]])
def test_merge_table(sc):
    from oracle import ops
    assert np.array_equal(ops.merge(U(sc["lhs"]), U(sc["rhs"])), U(sc["merged"]))
    assert np.array_equal(ops.merge(U(sc["lhs"]), U(sc["rhs"]), drop_duplicates=True), U(sc["merged_dropdup"]))


def test_bitcount_and_unique_tables():
    from oracle import ops
    for sc in T["bitcount"]:
        assert list(ops.popcount64(U(sc["bits"]))) == sc["expected"], sc["name"]
    for sc in T["unique"]:
        assert np.array_equal(ops.unique(U(sc["arr"]), sc["shift"]), U(sc["expected"]))


@pytest.mark.parametrize("sc", T["fixtures"], ids=[str(s["suffix"]) for s in T["fixtures"]])
def test_saved_posting_pairs(sc):
    """The reference's seven real posting pairs, each kept whole up to 1,024 words a side and sampled to about
    that size above it, with the reference's output on each (tests/golden/make_golden_posting_pairs.py)."""
    from oracle import ops
    n = sc["suffix"]
    lhs, rhs, mask = P[f"{n}.lhs"], P[f"{n}.rhs"], P[f"{n}.mask"][()]
    assert mask == np.uint64(sc["mask"])
    li, ri = ops.intersect(lhs, rhs, mask=mask)
    assert np.array_equal(li, P[f"{n}.intersect.lhs_idx"]) and np.array_equal(ri, P[f"{n}.intersect.rhs_idx"])
    got = ops.intersect_with_adjacents(lhs, rhs, mask=mask)
    for i, g in enumerate(got):
        assert np.array_equal(g, P[f"{n}.with_adjacents.{i}"]), i
    if (len(lhs), len(rhs)) == (sc["n_lhs"], sc["n_rhs"]):        # a whole pair: the digests of the full output too
        assert [len(li), digest(li), digest(ri)] == sc["intersect"]
        assert [[len(x), digest(x)] for x in got] == sc["with_adjacents"]
