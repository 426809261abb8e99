"""The long-segment split (csrc/segment_long.cu) through the C ABI and through ``ops``.

Sums and means of long segments are compared bit for bit against tests/long_segment_reference.py (pieces of P perm positions, piece
partials combined in ascending order).  Everything else is compared bit for bit against the existing entry points on the same plan:
max / min and their winners, every combination of backward terms, and the short segments of a mixed plan.  Plans are built with
numpy here, like tests/test_segment_kernels_gpu.py, and the split with hgn_segment_split_build, checked against the CPU bookkeeping.
"""
import ctypes
import itertools

import numpy as np
import pytest
import torch

import long_segment_reference as lr
import segment_reference as sr
from hgn_b200 import _cabi, ops
from hgn_b200.plan import SegmentPlan

pytestmark = pytest.mark.gpu

F32 = np.float32
BF = _cabi.HGN_BF16
OK, INVALID, WORKSPACE = 0, -1, -4


def _lib():
    return _cabi.load()


def _TP():
    return _lib().hgn_segment_split_threshold(), _lib().hgn_segment_split_piece()


def _gpu32(a):
    a = np.asarray(a, dtype=np.int32)
    return torch.from_numpy(a if a.size else np.zeros(1, np.int32)).cuda()


class Plan:
    """numpy CSR of ``ids`` and its split, built on the GPU."""

    def __init__(self, ids, S):
        lib = _lib()
        self.ids = np.asarray(ids, dtype=np.int64)
        self.S, self.E = S, len(self.ids)
        self.perm_np, self.rowptr_np = sr.csr(self.ids, S)
        self.perm, self.rowptr, self.ids32 = _gpu32(self.perm_np), _gpu32(self.rowptr_np), _gpu32(self.ids)
        E, S = self.E, self.S
        max_long = lib.hgn_segment_split_max_long(E, S)
        self.long_ids = torch.empty(max(max_long, 1), dtype=torch.int32, device="cuda")
        self.piece_ptr = torch.empty(max_long + 1, dtype=torch.int32, device="cuda")
        self.pieces = torch.empty(max(3 * lib.hgn_segment_split_max_pieces(E), 1), dtype=torch.int32, device="cuda")
        self.perm_short = torch.empty(max(E, 1), dtype=torch.int32, device="cuda")
        self.rowptr_short = torch.empty(S + 1, dtype=torch.int32, device="cuda")
        ws_bytes = lib.hgn_segment_split_build_workspace_bytes(E, S)
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device="cuda")
        counts = (ctypes.c_int64 * 3)()
        _cabi.check(lib.hgn_segment_split_build(self.perm.data_ptr(), self.rowptr.data_ptr(), E, S, self.long_ids.data_ptr(),
                                                self.piece_ptr.data_ptr(), self.pieces.data_ptr(), self.perm_short.data_ptr(),
                                                self.rowptr_short.data_ptr(), counts, ws.data_ptr(), ws_bytes, _cabi.stream_ptr()))
        self.n_long, self.n_pieces, self.n_short = (int(c) for c in counts)
        self.c = _cabi.SegmentSplit(S, E, self.n_long, self.n_pieces, self.n_short, self.long_ids.data_ptr(), self.piece_ptr.data_ptr(),
                                    self.pieces.data_ptr(), self.perm_short.data_ptr(), self.rowptr_short.data_ptr())

    def split_ref(self):
        return lr.split(self.perm_np, self.rowptr_np, *_TP())


def _ids(rng, sizes):
    ids = np.repeat(np.arange(len(sizes)), sizes)
    return ids[rng.permutation(len(ids))]


def _rows(rng, E, seed_scale=1.0):
    x = (rng.standard_normal((E, 128)) * seed_scale).astype(F32)
    t = torch.from_numpy(x).to(torch.bfloat16).cuda()
    return t, t.float().cpu().numpy()


def _np(t):
    return t.detach().float().cpu().numpy() if t.dtype != torch.int32 else t.cpu().numpy().astype(np.int64)


def _assert_bits(got, want, what):
    g = _np(got) if isinstance(got, torch.Tensor) else np.asarray(got)
    w = np.asarray(want)
    assert g.shape == w.shape, f"{what}: shape {g.shape} != {w.shape}"
    if g.dtype.kind == "f":
        g, w = np.ascontiguousarray(g, dtype=F32).view(np.uint32), np.ascontiguousarray(w, dtype=F32).view(np.uint32)
    bad = g != w
    if bad.any():
        i = tuple(np.argwhere(bad)[0])
        raise AssertionError(f"{what}: {int(bad.sum())} of {bad.size} differ; first at {i}: {g[i]!r} != {w[i]!r}")


def _ws(*plans):
    n = max([_lib().hgn_segment_split_reduce_workspace_bytes(ctypes.byref(p.c)) for p in plans] + [1])
    return torch.empty(n, dtype=torch.uint8, device="cuda")


def _outs(S, which):
    outs = [torch.empty((S, 128), dtype=torch.bfloat16, device="cuda") if w else None for w in which]
    am = torch.empty((S, 128), dtype=torch.int32, device="cuda") if which[2] else None
    an = torch.empty((S, 128), dtype=torch.int32, device="cuda") if which[3] else None
    return outs, am, an


def _reduce_split(x, p, which, prior=None):
    outs, am, an = _outs(p.S, which)
    if prior is not None:
        outs[0].copy_(prior)
    ws = _ws(p)
    _cabi.check(_lib().hgn_segment_reduce_split(BF, x.data_ptr(), p.E, 128, p.perm.data_ptr(), p.rowptr.data_ptr(), p.S, ctypes.byref(p.c),
                                                *[_cabi.ptr(o) for o in outs], _cabi.ptr(am), _cabi.ptr(an), int(prior is not None),
                                                ws.data_ptr(), ws.numel(), _cabi.stream_ptr()), "split")
    return outs, am, an


def _reduce_old(x, p, which, prior=None):
    outs, am, an = _outs(p.S, which)
    if prior is not None:
        outs[0].copy_(prior)
    _cabi.check(_lib().hgn_segment_reduce(BF, x.data_ptr(), p.E, 128, p.perm.data_ptr(), p.rowptr.data_ptr(), p.S,
                                          *[_cabi.ptr(o) for o in outs], _cabi.ptr(am), _cabi.ptr(an), int(prior is not None),
                                          _cabi.stream_ptr()), "old")
    return outs, am, an


def _size_cases():
    T, P = _TP()
    return {
        "T": [T], "T+1": [T + 1], "kP": [16 * P, T + 1], "kP+1": [5 * P + 1], "kP-1": [9 * P - 1],
        "mixed": [0, 3, T, T + 1, 0, 17, 12 * P, 2 * T + 5, 1, 0],
    }


SIZE_CASES = ["T", "T+1", "kP", "kP+1", "kP-1", "mixed"]


@pytest.mark.parametrize("case", SIZE_CASES + ["million", "up_pooling"])
def test_split_build_matches_cpu_bookkeeping(case):
    rng = np.random.default_rng(1)
    if case == "million":
        sizes = [1_000_000]
    elif case == "up_pooling":
        sizes = None
    else:
        sizes = _size_cases()[case]
    if sizes is None:
        ids = np.concatenate([np.repeat(np.arange(16) + 1_000_000, 62_500)])        # 16 clusters after 10^6 empty segments
        p = Plan(ids[rng.permutation(len(ids))], 1_000_016)
    else:
        p = Plan(_ids(rng, sizes), len(sizes))
    ref = p.split_ref()
    assert (p.n_long, p.n_pieces, p.n_short) == (len(ref["long_ids"]), len(ref["pieces"]), len(ref["perm_short"]))
    _assert_bits(p.rowptr_short, ref["rowptr_short"], "rowptr_short")
    _assert_bits(p.perm_short[:p.n_short], ref["perm_short"], "perm_short")
    if p.n_long:
        _assert_bits(p.long_ids[:p.n_long], ref["long_ids"], "long_ids")
        _assert_bits(p.piece_ptr[:p.n_long + 1], ref["piece_ptr"], "piece_ptr")
        _assert_bits(p.pieces[:3 * p.n_pieces].view(-1, 3), ref["pieces"], "pieces")


def _long_plan(case, rng):
    if case == "million":
        return Plan(np.zeros(1_000_000, dtype=np.int64), 1)
    if case == "up_pooling":
        ids = np.repeat(np.arange(16) + 1_000_000, 62_500)
        return Plan(ids[rng.permutation(len(ids))], 1_000_016)
    sizes = _size_cases()[case]
    return Plan(_ids(rng, sizes), len(sizes))


@pytest.mark.parametrize("case", SIZE_CASES + ["million", "up_pooling"])
def test_forward_vs_reference_and_existing_entry_point(case):
    rng = np.random.default_rng(2)
    T, P = _TP()
    p = _long_plan(case, rng)
    x, x_np = _rows(rng, p.E)
    # sum without prior (the sum-only path), vs the reference
    (s, _, _, _), _, _ = _reduce_split(x, p, (1, 0, 0, 0))
    want = lr.segment_sum(x_np, p.perm_np, p.rowptr_np, T, P, out_dtype="bfloat16")
    _assert_bits(s, want, "sum")
    # short segments: bit-identical to the existing entry point
    (s_old, _, _, _), _, _ = _reduce_old(x, p, (1, 0, 0, 0))
    short = np.diff(p.rowptr_np) <= T
    _assert_bits(s[torch.from_numpy(short).cuda()], _np(s_old)[short], "short sums")
    # sum with a prior (including -0 and +0 priors), mean, max, min and the winners in one call
    prior_np = rng.standard_normal((p.S, 128)).astype(F32)
    prior_np[:, :8] = F32(-0.0)
    prior_np[:, 8:16] = F32(0.0)
    prior = torch.from_numpy(prior_np).to(torch.bfloat16).cuda()
    prior_np = prior.float().cpu().numpy()
    (s, m, mx, mn), am, an = _reduce_split(x, p, (1, 1, 1, 1), prior=prior)
    _assert_bits(s, lr.segment_sum(x_np, p.perm_np, p.rowptr_np, T, P, prior=prior_np, out_dtype="bfloat16"), "sum + prior")
    _assert_bits(m, lr.segment_mean(x_np, p.perm_np, p.rowptr_np, T, P, out_dtype="bfloat16"), "mean")
    (s_o, m_o, mx_o, mn_o), am_o, an_o = _reduce_old(x, p, (1, 1, 1, 1), prior=prior)
    for got, old, what in ((mx, mx_o, "max"), (mn, mn_o, "min"), (am, am_o, "argmax"), (an, an_o, "argmin")):
        _assert_bits(got, _np(old), what)
    sh = torch.from_numpy(short).cuda()
    _assert_bits(s[sh], _np(s_o)[short], "short sums + prior")
    _assert_bits(m[sh], _np(m_o)[short], "short means")
    # sum-only with a prior (the bf16 sum kernel on the short CSR)
    (s, _, _, _), _, _ = _reduce_split(x, p, (1, 0, 0, 0), prior=prior)
    _assert_bits(s, lr.segment_sum(x_np, p.perm_np, p.rowptr_np, T, P, prior=prior_np, out_dtype="bfloat16"), "sum-only + prior")


def test_max_min_ties_across_pieces():
    """Few distinct values and signed zeros: winners are decided by ties across pieces."""
    rng = np.random.default_rng(3)
    T, P = _TP()
    p = Plan(_ids(rng, [T + 3 * P + 5, 2 * T + 1, 7]), 3)
    v = rng.integers(-1, 2, size=(p.E, 128)).astype(F32)
    v[rng.random((p.E, 128)) < 0.4] = F32(-0.0)
    x = torch.from_numpy(v).to(torch.bfloat16).cuda()
    (_, _, mx, mn), am, an = _reduce_split(x, p, (0, 0, 1, 1))
    (_, _, mx_o, mn_o), am_o, an_o = _reduce_old(x, p, (0, 0, 1, 1))
    for got, old, what in ((mx, mx_o, "max"), (mn, mn_o, "min"), (am, am_o, "argmax"), (an, an_o, "argmin")):
        _assert_bits(got, _np(old), what)
    for largest, val, arg in ((True, mx, am), (False, mn, an)):
        rv, ra = lr.segment_argext(v, p.perm_np, p.rowptr_np, T, P, largest)
        _assert_bits(val, rv, "reference value")
        _assert_bits(arg, ra, "reference arg")


TERMS = [c for c in itertools.product([0, 1], repeat=4) if any(c)]


@pytest.mark.parametrize("case", ["mixed", "kP+1", "up_pooling"])
def test_backward_terms_bit_identical_to_existing(case):
    rng = np.random.default_rng(4)
    p = _long_plan(case, rng)
    x, _ = _rows(rng, p.E)
    _, am, an = _reduce_old(x, p, (0, 0, 1, 1))
    g = [torch.from_numpy(rng.standard_normal((p.S, 128)).astype(F32)).to(torch.bfloat16).cuda() for _ in range(4)]
    base = torch.from_numpy(rng.standard_normal((p.E, 128)).astype(F32)).to(torch.bfloat16).cuda()
    for terms in TERMS:
        gs = [gi if t else None for gi, t in zip(g, terms)]
        a_max, a_min = (am if terms[2] else None), (an if terms[3] else None)
        got = torch.full((p.E, 128), float("nan"), dtype=torch.bfloat16, device="cuda")
        old = torch.full((p.E, 128), float("nan"), dtype=torch.bfloat16, device="cuda")
        _cabi.check(_lib().hgn_segment_reduce_bwd_split(BF, p.E, 128, p.ids32.data_ptr(), p.perm.data_ptr(), p.rowptr.data_ptr(), p.S,
                                                        ctypes.byref(p.c), *[_cabi.ptr(t) for t in gs], _cabi.ptr(a_max), _cabi.ptr(a_min),
                                                        got.data_ptr(), _cabi.stream_ptr()))
        _cabi.check(_lib().hgn_segment_reduce_bwd(BF, p.E, 128, p.ids32.data_ptr(), p.perm.data_ptr(), p.rowptr.data_ptr(), p.S,
                                                  *[_cabi.ptr(t) for t in gs], _cabi.ptr(a_max), _cabi.ptr(a_min), old.data_ptr(), 0,
                                                  _cabi.stream_ptr()))
        _assert_bits(got, _np(old), f"reduce_bwd {terms}")
        for with_base in (False, True):
            res = {}
            for name in ("split", "old"):
                agg = torch.full((p.S, 128), float("nan"), dtype=torch.bfloat16, device="cuda") if (terms[0] or terms[1]) else None
                eg = (torch.full((p.E, 128), float("nan"), dtype=torch.bfloat16, device="cuda")
                      if (terms[2] or terms[3] or with_base) else None)
                b = base if with_base else None
                if name == "split":
                    rc = _lib().hgn_segment_layer_grad_split(BF, p.E, 128, p.perm.data_ptr(), p.rowptr.data_ptr(), p.S, ctypes.byref(p.c),
                                                             *[_cabi.ptr(t) for t in gs], _cabi.ptr(a_max), _cabi.ptr(a_min), _cabi.ptr(b),
                                                             _cabi.ptr(agg), _cabi.ptr(eg), _cabi.stream_ptr())
                else:
                    rc = _lib().hgn_segment_layer_grad(BF, p.E, 128, p.perm.data_ptr(), p.rowptr.data_ptr(), p.S,
                                                       *[_cabi.ptr(t) for t in gs], _cabi.ptr(a_max), _cabi.ptr(a_min), _cabi.ptr(b),
                                                       _cabi.ptr(agg), _cabi.ptr(eg), _cabi.stream_ptr())
                _cabi.check(rc, name)
                res[name] = (agg, eg)
            for i, what in ((0, "agg_grad"), (1, "edge_grad")):
                if res["old"][i] is not None:
                    _assert_bits(res["split"][i], _np(res["old"][i]), f"layer_grad {what} {terms} base={with_base}")


@pytest.mark.parametrize("sides", ["a", "b", "both"])
def test_sum_pair_with_split(sides):
    rng = np.random.default_rng(5)
    T, P = _TP()
    E = 3 * T + 2 * P + 11
    long_ids = _ids(rng, [E - 40, 40])                         # one long segment and one short one
    short_ids = rng.integers(0, 500, size=E)                   # all short
    ids_a = long_ids if sides in ("a", "both") else short_ids
    ids_b = long_ids if sides in ("b", "both") else short_ids
    pa, pb = Plan(ids_a, int(ids_a.max()) + 1), Plan(ids_b, int(ids_b.max()) + 1)
    x, x_np = _rows(rng, E)
    oa = torch.empty((pa.S, 128), dtype=torch.bfloat16, device="cuda")
    ob = torch.empty((pb.S, 128), dtype=torch.bfloat16, device="cuda")
    sa = ctypes.byref(pa.c) if pa.n_long else None
    sb = ctypes.byref(pb.c) if pb.n_long else None
    ws = _ws(pa, pb)
    _cabi.check(_lib().hgn_segment_sum_pair_split(BF, x.data_ptr(), E, 128, pa.perm.data_ptr(), pa.rowptr.data_ptr(), pa.S, sa, oa.data_ptr(),
                                                  pb.perm.data_ptr(), pb.rowptr.data_ptr(), pb.S, sb, ob.data_ptr(), ws.data_ptr(), ws.numel(),
                                                  _cabi.stream_ptr()))
    for p, o in ((pa, oa), (pb, ob)):
        _assert_bits(o, lr.segment_sum(x_np, p.perm_np, p.rowptr_np, T, P, out_dtype="bfloat16"), "pair side")


def test_refusals():
    rng = np.random.default_rng(6)
    T, P = _TP()
    p = Plan(_ids(rng, [T + 1, 3]), 2)
    x, _ = _rows(rng, p.E)
    out = torch.empty((p.S, 128), dtype=torch.bfloat16, device="cuda")
    ws = _ws(p)
    lib = _lib()

    def call(dtype=BF, D=128, S=p.S, E=p.E, ws_bytes=ws.numel()):
        return lib.hgn_segment_reduce_split(dtype, x.data_ptr(), E, D, p.perm.data_ptr(), p.rowptr.data_ptr(), S, ctypes.byref(p.c),
                                            out.data_ptr(), None, None, None, None, None, 0, ws.data_ptr(), ws_bytes, _cabi.stream_ptr())
    assert call() == OK
    assert call(dtype=_cabi.HGN_F32) == INVALID
    assert call(D=64) == INVALID
    assert call(S=p.S + 1) == INVALID and b"split built for" in lib.hgn_last_error()
    assert call(E=p.E - 1) == INVALID
    assert call(ws_bytes=ws.numel() - 1) == WORKSPACE
    g = torch.zeros((p.S, 128), dtype=torch.bfloat16, device="cuda")
    grad = torch.empty((p.E, 128), dtype=torch.bfloat16, device="cuda")
    assert lib.hgn_segment_reduce_bwd_split(_cabi.HGN_F32, p.E, 128, p.ids32.data_ptr(), p.perm.data_ptr(), p.rowptr.data_ptr(), p.S,
                                            ctypes.byref(p.c), g.data_ptr(), None, None, None, None, None, grad.data_ptr(),
                                            _cabi.stream_ptr()) == INVALID
    assert lib.hgn_segment_layer_grad_split(BF, p.E, 128, p.perm.data_ptr(), p.rowptr.data_ptr(), p.S + 2, ctypes.byref(p.c), g.data_ptr(),
                                            None, None, None, None, None, None, out.data_ptr(), None, _cabi.stream_ptr()) == INVALID
    assert lib.hgn_segment_sum_pair_split(BF, x.data_ptr(), p.E, 128, p.perm.data_ptr(), p.rowptr.data_ptr(), p.S, ctypes.byref(p.c),
                                          out.data_ptr(), p.perm.data_ptr(), p.rowptr.data_ptr(), p.S, None, out.data_ptr(), ws.data_ptr(), 0,
                                          _cabi.stream_ptr()) == WORKSPACE
    assert lib.hgn_segment_reduce_split(BF, x.data_ptr(), p.E, 128, p.perm.data_ptr(), p.rowptr.data_ptr(), p.S, None, out.data_ptr(),
                                        None, None, None, None, None, 0, ws.data_ptr(), ws.numel(), _cabi.stream_ptr()) == INVALID


def test_bitwise_repeatable():
    rng = np.random.default_rng(8)
    p = _long_plan("up_pooling", rng)
    x, _ = _rows(rng, p.E)
    a = _reduce_split(x, p, (1, 1, 1, 1))
    b = _reduce_split(x, p, (1, 1, 1, 1))
    for u, v in zip(list(a[0]) + [a[1], a[2]], list(b[0]) + [b[1], b[2]]):
        assert torch.equal(u.view(torch.int16) if u.dtype == torch.bfloat16 else u, v.view(torch.int16) if v.dtype == torch.bfloat16 else v)


# ---- through ops ---------------------------------------------------------------------------------------------------------------
def test_plan_without_long_segment_has_no_split_and_unchanged_launches():
    rng = np.random.default_rng(9)
    T, _ = _TP()
    ids = torch.from_numpy(_ids(rng, [T, 5, 0, T - 1] * 3)).cuda()
    plan = SegmentPlan(ids, 12)
    assert plan.split is None
    x = torch.randn((ids.numel(), 128), device="cuda").to(torch.bfloat16)
    out = torch.empty((12, 128), dtype=torch.bfloat16, device="cuda")
    n0 = ops.launch_count
    ops._segment_sum(x, plan, out)
    ops._segment_reduce(x, plan, [out, None, None, None], None, None)
    ops._segment_sum_pair(x, plan, out, plan, torch.empty_like(out))
    assert ops.launch_count - n0 == 3


def test_ops_bindings_route_through_the_split():
    rng = np.random.default_rng(10)
    T, P = _TP()
    sizes = [3, 4 * T + 3, 0, 2 * P + T, 11]
    ids_np = _ids(rng, sizes)
    ids = torch.from_numpy(ids_np).cuda()
    plan = SegmentPlan(ids, len(sizes))
    assert plan.split is not None and plan.split.n_long == 2
    perm_np, rowptr_np = sr.csr(ids_np, len(sizes))
    x = torch.randn((ids.numel(), 128), device="cuda").to(torch.bfloat16).requires_grad_(True)
    x_np = x.detach().float().cpu().numpy()
    want = lr.segment_sum(x_np, perm_np, rowptr_np, T, P, out_dtype="bfloat16")
    out = torch.empty((len(sizes), 128), dtype=torch.bfloat16, device="cuda")
    n0 = ops.launch_count
    ops._segment_sum(x.detach(), plan, out)
    assert ops.launch_count - n0 == 3
    _assert_bits(out, want, "ops._segment_sum")
    # the autograd aggregate: forward vs reference / sequential winners, backward vs the existing entry point
    s, m, mx, mn = ops.segment_aggregate(x, plan, ["sum", "mean", "max", "min"])
    _assert_bits(s, want, "segment_aggregate sum")
    _assert_bits(m, lr.segment_mean(x_np, perm_np, rowptr_np, T, P, out_dtype="bfloat16"), "segment_aggregate mean")
    _assert_bits(mx, sr._out(sr.segment_argext(x_np, perm_np, rowptr_np, True)[0], "bfloat16"), "segment_aggregate max")
    gs = [torch.randn_like(t) for t in (s, m, mx, mn)]
    torch.autograd.backward([s, m, mx, mn], gs)
    p = Plan(ids_np, len(sizes))
    _, am, an = _reduce_old(x.detach(), p, (0, 0, 1, 1))
    old = torch.empty((p.E, 128), dtype=torch.bfloat16, device="cuda")
    _cabi.check(_lib().hgn_segment_reduce_bwd(BF, p.E, 128, p.ids32.data_ptr(), p.perm.data_ptr(), p.rowptr.data_ptr(), p.S,
                                              *[g.data_ptr() for g in gs], am.data_ptr(), an.data_ptr(), old.data_ptr(), 0, _cabi.stream_ptr()))
    _assert_bits(x.grad, _np(old), "segment_aggregate backward")


def test_ops_layer_grad_and_sum_pair_route_through_the_split():
    """``ops._segment_layer_grad`` (the fused non-'sum' layer's backward) and ``ops._segment_sum_pair`` (the edge update's backward)
    on a plan with long segments: the split entry points' results, and the launches their ``_count`` adds."""
    rng = np.random.default_rng(11)
    T, P = _TP()
    sizes = [5, 3 * T + 7, 0, T + 2 * P, 9]
    ids_np = _ids(rng, sizes)
    E, S = len(ids_np), len(sizes)
    plan = SegmentPlan(torch.from_numpy(ids_np).cuda(), S)
    short_np = rng.integers(0, 300, size=E)
    plan_short = SegmentPlan(torch.from_numpy(short_np).cuda(), 300)
    assert plan.split is not None and plan_short.split is None
    p, ps = Plan(ids_np, S), Plan(short_np, 300)
    x, x_np = _rows(rng, E)
    _, am, an = _reduce_old(x, p, (0, 0, 1, 1))
    g = {op: torch.randn((S, 128), device="cuda").to(torch.bfloat16) for op in ("sum", "mean", "max", "min")}
    base = torch.randn((E, 128), device="cuda").to(torch.bfloat16)
    agg, eg = torch.empty((S, 128), dtype=torch.bfloat16, device="cuda"), torch.empty((E, 128), dtype=torch.bfloat16, device="cuda")
    n0 = ops.launch_count
    ops._segment_layer_grad(plan, E, g, am, an, base, agg, eg)
    assert ops.launch_count - n0 == 2
    agg_o, eg_o = torch.empty_like(agg), torch.empty_like(eg)
    _cabi.check(_lib().hgn_segment_layer_grad(BF, E, 128, p.perm.data_ptr(), p.rowptr.data_ptr(), S, *[g[op].data_ptr() for op in g],
                                              am.data_ptr(), an.data_ptr(), base.data_ptr(), agg_o.data_ptr(), eg_o.data_ptr(),
                                              _cabi.stream_ptr()))
    _assert_bits(agg, _np(agg_o), "ops layer_grad agg_grad")
    _assert_bits(eg, _np(eg_o), "ops layer_grad edge_grad")
    oa, ob = torch.empty((S, 128), dtype=torch.bfloat16, device="cuda"), torch.empty((300, 128), dtype=torch.bfloat16, device="cuda")
    n0 = ops.launch_count
    ops._segment_sum_pair(x, plan, oa, plan_short, ob)
    assert ops.launch_count - n0 == 1 + 2
    _assert_bits(oa, lr.segment_sum(x_np, p.perm_np, p.rowptr_np, T, P, out_dtype="bfloat16"), "ops pair, split side")
    _assert_bits(ob, sr.segment_sum(x_np, ps.perm_np, ps.rowptr_np, out_dtype="bfloat16"), "ops pair, short side")
