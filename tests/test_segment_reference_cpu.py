"""CPU checks of tests/segment_reference.py, the order-exact reference the segment-kernel tests compare with bit for bit: its bf16
rounding, its summation order, its tie rule (ties, +-0, empty segments) and its agreement with the oracle's segment_reduce."""
import numpy as np
import torch

import hgn_oracle as orc
import segment_reference as sr

F32 = np.float32


def _bits(a):
    return np.ascontiguousarray(a, dtype=F32).view(np.uint32)


def test_round_bf16_matches_torch_including_ties():
    rng = np.random.default_rng(0)
    x = rng.standard_normal(100_000).astype(F32) * F32(1e3)
    # exact halfway cases: bf16 value + half a bf16 ulp, with even and odd last kept bit
    halves = (np.arange(-2000, 2000, dtype=np.int64).astype(np.uint32) << 16) | np.uint32(0x8000)
    x = np.concatenate([x, halves.view(F32)[np.isfinite(halves.view(F32))], np.array([0.0, -0.0, 3.0e38, -3.0e38], dtype=F32)])
    want = torch.from_numpy(x).to(torch.bfloat16).float().numpy()
    assert np.array_equal(_bits(sr.round_bf16(x)), _bits(want))


def test_csr_is_a_stable_grouping():
    ids = np.array([2, 0, 2, 1, 0, 2, 4])
    perm, rowptr = sr.csr(ids, 5)
    assert perm.tolist() == [1, 4, 3, 0, 2, 5, 6] and rowptr.tolist() == [0, 2, 3, 6, 6, 7]


def test_sum_is_sequential_in_element_order():
    # segment 0 = elements 0, 2, 3 (element 1 is in segment 1): ((0 + 1e8) - 1e8) + 1 = 1, where any other order gives 0
    x = np.array([[1e8], [5.0], [-1e8], [1.0]], dtype=F32)
    perm, rowptr = sr.csr(np.array([0, 1, 0, 0]), 2)
    assert sr.segment_sum(x, perm, rowptr).ravel().tolist() == [1.0, 5.0]
    # accumulate: (0 + 3 + 3) + 1e8 = 1e8 + 8 (one rounding of 1e8 + 6); adding the prior first would give 1e8
    x = np.array([[3.0], [3.0]], dtype=F32)
    perm, rowptr = sr.csr(np.array([0, 0]), 1)
    got = sr.segment_sum(x, perm, rowptr, prior=np.array([[1e8]], dtype=F32))
    assert got[0, 0] == F32(1e8) + F32(8) and F32(F32(1e8) + F32(3)) + F32(3) == F32(1e8)
    # multi-source sum: base first, then the sources -- here that is (1e8 + 3) + 3 = 1e8
    got = sr.multi_segment_sum([(x, perm, rowptr)], base=np.array([[1e8]], dtype=F32))
    assert got[0, 0] == F32(1e8)
    # the bf16 result is rounded once, at the end: 1 + 2^-8 + 2^-8 = 1 + 2^-7, where rounding each partial sum (a tie, to even)
    # would give 1
    x = np.array([[1.0], [2.0 ** -8], [2.0 ** -8]], dtype=F32)
    perm, rowptr = sr.csr(np.zeros(3, dtype=np.int64), 1)
    assert sr.segment_sum(x, perm, rowptr, out_dtype="bfloat16")[0, 0] == F32(1 + 2.0 ** -7)


def test_max_min_first_winner_and_signed_zeros():
    #                 seg 0: 2, 5, 5, 1    seg 1 (empty)    seg 2: -0, +0    seg 3: +0, -0    seg 4: 3 (first), 1, 3 (last)
    vals = [2.0, 5.0, 5.0, 1.0, -0.0, 0.0, 0.0, -0.0, 3.0, 1.0, 3.0]
    segs = [0, 0, 0, 0, 2, 2, 3, 3, 4, 4, 4]
    # interleave the elements so that the segments' element ids are not contiguous: perm order must still be ascending id
    order = np.random.default_rng(1).permutation(len(vals))
    x = np.array(vals, dtype=F32)[order][:, None]
    ids = np.array(segs)[order]
    inv = np.argsort(order)                               # inv[k] = element id of original entry k
    perm, rowptr = sr.csr(ids, 5)
    mx, amx = sr.segment_argext(x, perm, rowptr, True)
    mn, amn = sr.segment_argext(x, perm, rowptr, False)

    def first(cands):                                     # among original entries, the one with the lowest element id
        return int(min(inv[c] for c in cands))
    assert amx[:, 0].tolist() == [first([1, 2]), -1, first([4, 5]), first([6, 7]), first([8, 10])]
    assert amn[:, 0].tolist() == [int(inv[3]), -1, first([4, 5]), first([6, 7]), int(inv[9])]
    assert mx[:, 0].tolist() == [5.0, 0.0, 0.0, 0.0, 3.0] and mn[:, 0].tolist() == [1.0, 0.0, 0.0, 0.0, 1.0]
    # the value is the winner's own: its sign bit survives; an empty segment is +0.0
    for out, arg in ((mx, amx), (mn, amn)):
        for s in (2, 3):
            assert _bits(out[s, 0]) == _bits(x[arg[s, 0], 0])
        assert _bits(out[1, 0]) == 0
    # the backward routes g_max / g_min to the winner only; everything else gets +0.0
    g = np.arange(1, 6, dtype=F32)[:, None]
    grad = sr.segment_backward(ids, rowptr, g_max=g, argmax=amx)
    want = np.zeros_like(x)
    for s in (0, 2, 3, 4):
        want[amx[s, 0], 0] = g[s, 0]
    assert np.array_equal(_bits(grad), _bits(want))


def test_empty_segments_and_no_elements():
    x = np.ones((3, 4), dtype=F32)
    perm, rowptr = sr.csr(np.array([3, 3, 0]), 6)
    assert np.array_equal(sr.segment_sum(x, perm, rowptr)[[1, 2, 4, 5]], np.zeros((4, 4), F32))
    assert np.array_equal(sr.segment_mean(x, perm, rowptr)[[1, 2, 4, 5]], np.zeros((4, 4), F32))
    assert sr.segment_mean(x, perm, rowptr)[3, 0] == 1.0
    v, a = sr.segment_argext(x, perm, rowptr, True)
    assert (a[[1, 2, 4, 5]] == -1).all() and (_bits(v[[1, 2, 4, 5]]) == 0).all()
    perm, rowptr = sr.csr(np.zeros(0, dtype=np.int64), 3)
    empty = np.zeros((0, 4), dtype=F32)
    assert np.array_equal(sr.segment_sum(empty, perm, rowptr), np.zeros((3, 4), F32))
    v, a = sr.segment_argext(empty, perm, rowptr, False)
    assert (a == -1).all() and (_bits(v) == 0).all()


def test_reference_agrees_with_the_oracle_on_random_data():
    rng = np.random.default_rng(7)
    for E, S, D, ties in ((1, 1, 4, False), (300, 20, 3, True), (5000, 400, 8, False), (4000, 7, 128, True)):
        ids = rng.integers(0, max(S - 1, 1), size=E)                   # the last segment stays empty (S > 1)
        x = (rng.integers(-3, 4, size=(E, D)) if ties else rng.standard_normal((E, D))).astype(F32)
        x = sr.round_bf16(x)
        perm, rowptr = sr.csr(ids, S)
        xt = torch.from_numpy(x).requires_grad_(True)
        idt = torch.from_numpy(ids)
        # sum / mean: the same value up to fp32 rounding of a different order
        bound = (np.diff(rowptr)[:, None] + 1) * 2.0 ** -24 * sr.segment_sum(np.abs(x), perm, rowptr).astype(np.float64)
        for op, got in (("sum", sr.segment_sum(x, perm, rowptr)), ("mean", sr.segment_mean(x, perm, rowptr, reciprocal=False))):
            want = orc.segment_reduce(xt, idt, S, op).detach().numpy()
            div = 1.0 if op == "sum" else np.maximum(np.diff(rowptr), 1)[:, None]
            assert (np.abs(got.astype(np.float64) - want) <= bound / div + 1e-30).all(), op
        # max / min: the same values and the same winner (compared through the gradient the oracle routes to it)
        for largest, op in ((True, "max"), (False, "min")):
            v, a = sr.segment_argext(x, perm, rowptr, largest)
            xt.grad = None
            out = orc.segment_reduce(xt, idt, S, op)
            assert np.array_equal(v, out.detach().numpy()), op
            g = rng.standard_normal((S, D)).astype(F32)
            out.backward(torch.from_numpy(g))
            kw = {"g_max": g, "argmax": a} if largest else {"g_min": g, "argmin": a}
            assert np.array_equal(sr.segment_backward(ids, rowptr, **kw), xt.grad.numpy()), op
        # sum / mean backward: the oracle's autograd gathers g and divides by the count
        g = rng.standard_normal((S, D)).astype(F32)
        for op, kw in (("sum", {"g_sum": g}), ("mean", {"g_mean": g, "reciprocal": False})):
            xt.grad = None
            orc.segment_reduce(xt, idt, S, op).backward(torch.from_numpy(g))
            assert np.array_equal(sr.segment_backward(ids, rowptr, **kw), xt.grad.numpy()), op
