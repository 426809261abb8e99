"""CPU checks of tests/long_segment_reference.py: the split bookkeeping, max / min winners equal to the sequential ones, and sums that
reduce to the sequential order when every long segment is one piece."""
import numpy as np
import pytest

import long_segment_reference as lr
import segment_reference as sr
from hgn_b200 import _cabi

F32 = np.float32


def _library_constants():
    lib = _cabi.load()
    return lib.hgn_segment_split_threshold(), lib.hgn_segment_split_piece()


def _ids(rng, sizes):
    ids = np.repeat(np.arange(len(sizes)), sizes)
    return ids[rng.permutation(len(ids))]


def test_library_constants():
    T, P = _library_constants()
    assert T >= P >= 1


@pytest.mark.parametrize("T,P", [(8, 3), (16, 16), (2048, 256)])
def test_split_bookkeeping(T, P):
    rng = np.random.default_rng(T + P)
    sizes = [0, 1, T, T + 1, 2 * P, 2 * P + 1, 3 * P - 1, 5 * T + 7, 0, T + P, 3]
    perm, rowptr = sr.csr(_ids(rng, sizes), len(sizes))
    sp = lr.split(perm, rowptr, T, P)
    counts = np.diff(rowptr)
    assert list(sp["long_ids"]) == [s for s, n in enumerate(sizes) if n > T]
    for i, s in enumerate(sp["long_ids"]):
        ps = sp["pieces"][sp["piece_ptr"][i]:sp["piece_ptr"][i + 1]]
        assert (ps[:, 0] == s).all()
        assert ps[0, 1] == rowptr[s] and ps[-1, 2] == rowptr[s + 1]
        assert (ps[1:, 1] == ps[:-1, 2]).all()              # consecutive, no gap
        lens = ps[:, 2] - ps[:, 1]
        assert (lens[:-1] == P).all() and 1 <= lens[-1] <= P
    assert sp["piece_ptr"][-1] == len(sp["pieces"]) <= 2 * len(perm) // P
    # short CSR = the plan minus the long segments, order kept
    short = [s for s in range(len(sizes)) if counts[s] <= T]
    assert (np.diff(sp["rowptr_short"])[short] == counts[short]).all()
    assert (np.diff(sp["rowptr_short"])[sp["long_ids"]] == 0).all()
    want = np.concatenate([perm[rowptr[s]:rowptr[s + 1]] for s in short] or [np.zeros(0, np.int64)])
    assert np.array_equal(sp["perm_short"], want)


@pytest.mark.parametrize("largest", [True, False])
def test_piecewise_winners_equal_sequential(largest):
    rng = np.random.default_rng(7)
    T, P = 8, 3
    sizes = [0, 5, 9, 10, 20, 31]
    perm, rowptr = sr.csr(_ids(rng, sizes), len(sizes))
    E = len(perm)
    # few distinct values, so ties across pieces are common, and signed zeros
    x = rng.integers(-2, 3, size=(E, 16)).astype(F32)
    x[rng.random((E, 16)) < 0.3] = F32(-0.0)
    v, a = lr.segment_argext(x, perm, rowptr, T, P, largest)
    vs, as_ = sr.segment_argext(x, perm, rowptr, largest)
    assert np.array_equal(a, as_)
    assert np.array_equal(v.view(np.uint32), vs.view(np.uint32))


def test_one_piece_sums_are_sequential():
    rng = np.random.default_rng(3)
    sizes = [0, 1, 4, 17, 40]
    perm, rowptr = sr.csr(_ids(rng, sizes), len(sizes))
    x = rng.standard_normal((len(perm), 8)).astype(F32)
    prior = rng.standard_normal((len(sizes), 8)).astype(F32)
    got = lr.segment_sum(x, perm, rowptr, 0, 64, prior=prior)            # every non-empty segment is long, with one piece
    assert np.array_equal(got.view(np.uint32), sr.segment_sum(x, perm, rowptr, prior=prior).view(np.uint32))
    got = lr.segment_mean(x, perm, rowptr, 0, 64)
    assert np.array_equal(got.view(np.uint32), sr.segment_mean(x, perm, rowptr).view(np.uint32))


def test_many_piece_sums_follow_the_piece_order():
    rng = np.random.default_rng(4)
    perm, rowptr = sr.csr(_ids(rng, [50]), 1)
    x = rng.standard_normal((50, 4)).astype(F32)
    got = lr.segment_sum(x, perm, rowptr, 10, 16)
    p = [sr.sequential_sum(x[perm[b:b + 16]], np.arange(len(perm[b:b + 16])), np.array([0, len(perm[b:b + 16])]))[0]
         for b in range(0, 50, 16)]
    want = ((F32(0) + p[0]) + p[1]) + p[2]
    want = want + p[3]
    assert np.array_equal(got[0].view(np.uint32), want.astype(F32).view(np.uint32))
