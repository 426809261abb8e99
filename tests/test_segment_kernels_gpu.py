"""The C ABI of csrc/segment.cu against the order-exact reference of tests/segment_reference.py.

The segment kernels add, compare and copy in an order the header documents, and the library is built without fast-math, so most of
their results are compared bit for bit: sum (with and without accumulation), max / min and their winners, every backward with one
gradient term, the paired and the multi-source sums, the row gathers / scatters.  'mean' is compared bit for bit against the kernels'
formula (the vector kernels multiply by the fp32 reciprocal of the count, the scalar kernels divide) and within one unit in the last
place of the output dtype against sum / count.  The backward with all four gradient terms set is compared bit for bit against one of
two roundings: the vector kernels' g_sum + g_mean * (1 / count) may be contracted into one fused multiply-add by the compiler.

The arguments are chosen with the launch-site predicates of segment_reduce_impl / segment_reduce_bwd_impl so that every kernel runs:
bf16 rows of width 128 with only 'sum' -> segment_sum_bf16_128_kernel, other D % 4 == 0 -> the vector kernel, odd D -> the scalar
kernel; backward: bf16 / 128 with perm and without accumulation -> segment_bwd_bf16_128_kernel, else D % 4 == 0 -> the vector kernel,
else the scalar one.  Segment sizes 0 .. 33 cross the 2-row, 8-row and 16-row unroll boundaries of the three kernels.

Plans are built here with numpy (a stable argsort), so these tests do not depend on hgn_csr_build, which is checked on its own.
Non-finite inputs (NaN, +-inf) are out of scope: the kernels make no promise about them beyond what IEEE comparisons give.
"""
import ctypes

import numpy as np
import pytest
import torch

import segment_reference as sr
from hgn_b200 import _cabi, ops

pytestmark = pytest.mark.gpu

F32 = np.float32
DTYPES = {"fp32": torch.float32, "bf16": torch.bfloat16}
OUT = {"fp32": "float32", "bf16": "bfloat16"}
HGN_ERR_INVALID_ARGUMENT = -1
NAN = float("nan")


class Plan:
    """CSR grouping of ``ids`` (numpy) for the kernels (int32 on the GPU) and for the reference (int64 numpy)."""

    def __init__(self, ids, S):
        self.ids = np.asarray(ids, dtype=np.int64)
        self.S, self.E = S, len(self.ids)
        self.perm_np, self.rowptr_np = sr.csr(self.ids, S)
        gpu = lambda a: torch.from_numpy(np.asarray(a, dtype=np.int32)).cuda()
        self.perm = gpu(self.perm_np if self.E else [0])
        self.rowptr = gpu(self.rowptr_np)
        self.ids32 = gpu(self.ids if self.E else [0])


def _np(t):
    return t.detach().float().cpu().numpy()


def _rows(rng, E, D, dtype, positive=False):
    x = rng.standard_normal((E, D)).astype(F32)
    if positive:
        x = np.abs(x) + F32(1e-2)
    t = torch.from_numpy(x).to(DTYPES[dtype]).cuda()
    return t, _np(t)


def _assert_bits(got, want, what):
    g = _np(got) if isinstance(got, torch.Tensor) else np.asarray(got, dtype=F32)
    w = np.ascontiguousarray(want, dtype=F32)
    assert g.shape == w.shape, f"{what}: shape {g.shape} != {w.shape}"
    bad = g.view(np.uint32) != w.view(np.uint32)
    if bad.any():
        i = tuple(np.argwhere(bad)[0])
        raise AssertionError(f"{what}: {int(bad.sum())} of {bad.size} elements differ in their bits; first at {i}: {g[i]!r} != {w[i]!r}")


def _ulps(got, want, dtype):
    """max |got - want| in units of the last place of ``want`` in the output dtype."""
    g, w = _np(got).astype(np.float64), np.asarray(want, dtype=np.float64)
    _, e = np.frexp(w)
    ulp = np.ldexp(1.0, e - (24 if dtype == "fp32" else 8))
    return float((np.abs(g - w) / ulp).max()) if w.size else 0.0


def _degree_ids(rng, degrees):
    """Element -> segment ids for the given segment sizes, elements in random order (a segment's element ids are not contiguous)."""
    ids = np.repeat(np.arange(len(degrees)), degrees)
    rng.shuffle(ids)
    return ids


def _fan_in_plan(rng, copies=3):
    """Every segment size 0 .. 33, ``copies`` times each, segments in random order."""
    degrees = np.tile(np.arange(34), copies)
    rng.shuffle(degrees)
    return Plan(_degree_ids(rng, degrees), len(degrees))


# ------------------------------------------------------------------------------------------------------------------------------------
# forward
# ------------------------------------------------------------------------------------------------------------------------------------
def _reduce(x, plan, ops_, dtype, prior=None, args=True, D=None):
    """hgn_segment_reduce with the requested outputs NaN-filled (every element must be written), args -7-filled."""
    S, D = plan.S, x.shape[1] if x is not None else D
    tdt = DTYPES[dtype]
    outs = {op: (torch.full((S, D), NAN, dtype=tdt, device="cuda") if op in ops_ else None) for op in ("sum", "mean", "max", "min")}
    if prior is not None:
        outs["sum"] = prior.clone()
    am = {op: (torch.full((S, D), -7, dtype=torch.int32, device="cuda") if op in ops_ and args else None) for op in ("max", "min")}
    rc = _cabi.load().hgn_segment_reduce(_cabi.dtype_code(tdt), _cabi.ptr(x) if plan.E else None, plan.E, D, plan.perm.data_ptr(),
                                          plan.rowptr.data_ptr(), S, *[_cabi.ptr(outs[k]) for k in ("sum", "mean", "max", "min")],
                                          _cabi.ptr(am["max"]), _cabi.ptr(am["min"]), int(prior is not None), _cabi.stream_ptr())
    _cabi.check(rc, "hgn_segment_reduce")
    return outs, am


def _check_forward(x_np, plan, dtype, ops_, outs, am, prior_np=None, tag=""):
    D = x_np.shape[1]
    od = OUT[dtype]
    if "sum" in ops_:
        _assert_bits(outs["sum"], sr.segment_sum(x_np, plan.perm_np, plan.rowptr_np, prior_np, od), f"{tag} sum")
    if "mean" in ops_:
        _assert_bits(outs["mean"], sr.segment_mean(x_np, plan.perm_np, plan.rowptr_np, D % 4 == 0, od), f"{tag} mean")
        ulps = _ulps(outs["mean"], sr.segment_mean(x_np, plan.perm_np, plan.rowptr_np, False, od), dtype)
        assert ulps <= 1.0, f"{tag} mean: {ulps} ulp from sum / count"
    for op, largest in (("max", True), ("min", False)):
        if op in ops_:
            v, a = sr.segment_argext(x_np, plan.perm_np, plan.rowptr_np, largest)
            _assert_bits(outs[op], v, f"{tag} {op}")
            if am[op] is not None:
                assert np.array_equal(am[op].cpu().numpy(), a), f"{tag} arg{op}"


ALL = ("sum", "mean", "max", "min")
# (dtype, D, requested reductions): the kernel each one reaches
_FORWARD_CASES = [("bf16", 128, ("sum",))]                                                           # segment_sum_bf16_128_kernel
_FORWARD_CASES += [(dt, D, o) for dt in DTYPES for D in (4, 128, 132, 260) for o in (ALL, ("sum",), ("mean",), ("max",), ("min",))
                   if not (dt == "bf16" and D == 128 and o == ("sum",))]                            # segment_reduce_vec_kernel
_FORWARD_CASES += [(dt, D, ALL) for dt in DTYPES for D in (1, 3, 130)]                                # segment_reduce_scalar_kernel
# accumulate_sum only matters where 'sum' is requested
_FORWARD_CASES = [c + (acc,) for c in _FORWARD_CASES for acc in ((False, True) if "sum" in c[2] else (False,))]


@pytest.mark.parametrize("dtype,D,ops_,accumulate", _FORWARD_CASES)
def test_segment_reduce_bit_exact(dtype, D, ops_, accumulate):
    """Every segment size 0 .. 33 on each forward kernel; sum with and without accumulate_sum (prior added after the segment sum)."""
    rng = np.random.default_rng(D * 7 + len(ops_) + 100 * accumulate)
    plan = _fan_in_plan(rng)
    x, x_np = _rows(rng, plan.E, D, dtype)
    prior, prior_np = _rows(rng, plan.S, D, dtype) if accumulate and "sum" in ops_ else (None, None)
    outs, am = _reduce(x, plan, ops_, dtype, prior)
    _check_forward(x_np, plan, dtype, ops_, outs, am, prior_np, f"{dtype} D={D} {ops_}")


def _tied_rows(rng, plan, D, dtype):
    """Rows with purpose-built ties: columns c % 4 == 0 draw from {-1, -0, +0} (max is a tie of signed zeros), c % 4 == 1 from
    {1, -0, +0} (min is), the others from {-2, -1, -0, +0, 1, 2}; in every segment of three or more elements the second element
    copies the first and the last but one copies the last, so ties sit at the first and at the last position."""
    E = plan.E
    x = rng.choice(np.array([-2.0, -1.0, -0.0, 0.0, 1.0, 2.0], dtype=F32), size=(E, D))
    c = np.arange(D)
    x[:, c % 4 == 0] = rng.choice(np.array([-1.0, -0.0, 0.0], dtype=F32), size=(E, int((c % 4 == 0).sum())))
    x[:, c % 4 == 1] = rng.choice(np.array([1.0, -0.0, 0.0], dtype=F32), size=(E, int((c % 4 == 1).sum())))
    cnt = np.diff(plan.rowptr_np)
    for s in np.flatnonzero(cnt >= 3):
        b, e = plan.rowptr_np[s], plan.rowptr_np[s + 1]
        x[plan.perm_np[b + 1]] = x[plan.perm_np[b]]
        x[plan.perm_np[e - 2]] = x[plan.perm_np[e - 1]]
    return torch.from_numpy(x).to(DTYPES[dtype]).cuda(), x


def _tie_kinds(x_np, plan, largest):
    """How many (segment, column) extremes are ties won at the first position, ties that include the last position, and ties of
    -0 against +0."""
    v, a = sr.segment_argext(x_np, plan.perm_np, plan.rowptr_np, largest)
    first = last = zeros = 0
    for s in np.flatnonzero(np.diff(plan.rowptr_np) >= 2):
        seg = x_np[plan.perm_np[plan.rowptr_np[s]: plan.rowptr_np[s + 1]]]
        eq = seg == v[s]
        tie = eq.sum(0) >= 2
        first += int((tie & eq[0]).sum())
        last += int((tie & eq[-1]).sum())
        zeros += int((tie & (v[s] == 0) & (np.signbit(seg) & eq).any(0) & (~np.signbit(seg) & eq).any(0)).sum())
    return first, last, zeros


@pytest.mark.parametrize("D", [128, 4, 3])
@pytest.mark.parametrize("dtype", list(DTYPES))
def test_max_min_ties_first_element_wins(dtype, D):
    """Ties at the first position, at the last position and of -0 against +0: the first element in perm order wins, its own value
    (sign of zero included) is the output, and the backward routes g_max / g_min to that element only."""
    rng = np.random.default_rng(D + (dtype == "bf16"))
    plan = _fan_in_plan(rng)
    x, x_np = _tied_rows(rng, plan, D, dtype)
    for largest in (True, False):
        first, last, zeros = _tie_kinds(x_np, plan, largest)
        assert min(first, last, zeros) > 0, (largest, first, last, zeros)
    outs, am = _reduce(x, plan, ("max", "min"), dtype)
    _check_forward(x_np, plan, dtype, ("max", "min"), outs, am, tag=f"ties {dtype} D={D}")
    g, g_np = _rows(rng, plan.S, D, dtype)
    for op in ("max", "min"):
        grad = _backward(plan, dtype, D, {op: g}, {op: am[op]}, use_perm=True)
        want = sr.segment_backward(plan.ids, plan.rowptr_np, **{f"g_{op}": g_np, f"arg{op}": am[op].cpu().numpy()},
                                   out_dtype=OUT[dtype])
        _assert_bits(grad, want, f"ties {dtype} D={D} grad via arg{op}")


@pytest.mark.parametrize("dtype", list(DTYPES))
def test_segment_reduce_edges(dtype):
    """No elements (every segment empty: 0 and arg -1), no segments (nothing written), max / min without their arg outputs, one
    segment holding every element."""
    rng = np.random.default_rng(5)
    for D, ops_ in ((128, ("sum",)), (128, ALL), (4, ALL), (3, ALL)):
        plan = Plan(np.zeros(0, dtype=np.int64), 9)
        outs, am = _reduce(None, plan, ops_, dtype, D=D)
        for op in ops_:
            _assert_bits(outs[op], np.zeros((9, D), F32), f"E=0 D={D} {op}")
        for a in am.values():
            assert a is None or (a == -1).all()
        outs, _ = _reduce(None, plan, ops_, dtype, prior=torch.ones(9, D, dtype=DTYPES[dtype], device="cuda"), D=D)
        _assert_bits(outs["sum"], np.ones((9, D), F32), f"E=0 D={D} accumulate")
        # S = 0: returns without touching anything
        x, _ = _rows(rng, 5, D, dtype)
        sentinel = torch.full((4, D), 3.0, dtype=DTYPES[dtype], device="cuda")
        rowptr = torch.zeros(1, dtype=torch.int32, device="cuda")
        perm = torch.arange(5, dtype=torch.int32, device="cuda")
        _cabi.check(_cabi.load().hgn_segment_reduce(_cabi.dtype_code(DTYPES[dtype]), x.data_ptr(), 5, D, perm.data_ptr(), rowptr.data_ptr(), 0,
                                                    sentinel.data_ptr(), None, None, None, None, None, 0, _cabi.stream_ptr()))
        assert (sentinel == 3.0).all()
        # max / min with argmax / argmin NULL; S = 1
        for plan in (_fan_in_plan(rng, 1), Plan(np.zeros(77, dtype=np.int64), 1)):
            x, x_np = _rows(rng, plan.E, D, dtype)
            outs, am = _reduce(x, plan, ops_, dtype, args=False)
            _check_forward(x_np, plan, dtype, ops_, outs, am, tag=f"no args / S={plan.S} D={D}")


@pytest.mark.parametrize("dtype", list(DTYPES))
def test_segment_reduce_long_segments(dtype):
    """Hyper-node pooling: a handful of segments of ~1e5 elements each (plus an empty one), on every forward kernel and the backward."""
    rng = np.random.default_rng(17)
    plan = Plan(_degree_ids(rng, [100_000, 0, 99_999, 100_001, 3]), 5)
    for D, ops_ in ((128, ("sum",)), (128, ALL), (3, ALL)):
        x, x_np = _rows(rng, plan.E, D, dtype)
        prior, prior_np = _rows(rng, plan.S, D, dtype)
        outs, am = _reduce(x, plan, ops_, dtype, prior if ops_ == ("sum",) else None)
        _check_forward(x_np, plan, dtype, ops_, outs, am, prior_np if ops_ == ("sum",) else None, f"long D={D} {ops_}")
    g, g_np = _rows(rng, plan.S, 128, dtype)
    _assert_bits(_backward(plan, dtype, 128, {"mean": g}, {}, use_perm=True),
                 sr.segment_backward(plan.ids, plan.rowptr_np, g_mean=g_np, out_dtype=OUT[dtype]), "long backward g_mean")


def test_segment_kernels_at_grid_scale():
    """About 2 M elements over 2^19 + 1 segments: the forward kernels' and the per-segment backward's grids."""
    rng = np.random.default_rng(19)
    S = 2 ** 19 + 1
    plan = Plan(rng.integers(0, S, size=2_000_000), S)
    x, x_np = _rows(rng, plan.E, 128, "bf16")
    outs, am = _reduce(x, plan, ("sum",), "bf16")
    _check_forward(x_np, plan, "bf16", ("sum",), outs, am, tag="2M bf16 sum")
    g, g_np = _rows(rng, S, 128, "bf16")
    _assert_bits(_backward(plan, "bf16", 128, {"sum": g}, {}, use_perm=True),
                 sr.segment_backward(plan.ids, plan.rowptr_np, g_sum=g_np, out_dtype="bfloat16"), "2M bf16 backward")
    del x, x_np, g, g_np
    x, x_np = _rows(rng, plan.E, 4, "fp32")
    outs, am = _reduce(x, plan, ALL, "fp32")
    _check_forward(x_np, plan, "fp32", ALL, outs, am, tag="2M fp32 D=4")


# ------------------------------------------------------------------------------------------------------------------------------------
# backward
# ------------------------------------------------------------------------------------------------------------------------------------
def _backward(plan, dtype, D, grads, args, use_perm, prior=None):
    """hgn_segment_reduce_bwd; the output is NaN-filled unless ``prior`` (accumulate = 1) is given."""
    tdt = DTYPES[dtype]
    grad = prior.clone() if prior is not None else torch.full((plan.E, D), NAN, dtype=tdt, device="cuda")
    _cabi.check(_cabi.load().hgn_segment_reduce_bwd(
        _cabi.dtype_code(tdt), plan.E, D, plan.ids32.data_ptr(), plan.perm.data_ptr() if use_perm else None, plan.rowptr.data_ptr(),
        plan.S, *[_cabi.ptr(grads.get(k)) for k in ("sum", "mean", "max", "min")], _cabi.ptr(args.get("max")), _cabi.ptr(args.get("min")),
        grad.data_ptr(), int(prior is not None), _cabi.stream_ptr()), "hgn_segment_reduce_bwd")
    return grad


# (dtype, D, pass perm, accumulate): bf16 / 128 / perm / no accumulate -> segment_bwd_bf16_128_kernel; perm NULL or accumulate, or
# another dtype / width with D % 4 == 0 -> segment_reduce_bwd_vec_kernel; odd D -> segment_reduce_bwd_scalar_kernel
_BACKWARD_CASES = [("bf16", 128, True, False), ("bf16", 128, False, False), ("bf16", 128, True, True), ("bf16", 260, True, False),
                   ("fp32", 128, True, False), ("fp32", 128, False, True), ("fp32", 4, True, False),
                   ("bf16", 3, True, False), ("bf16", 130, True, True), ("fp32", 1, True, False), ("fp32", 3, False, True)]


@pytest.mark.parametrize("dtype,D,use_perm,accumulate", _BACKWARD_CASES)
def test_segment_backward(dtype, D, use_perm, accumulate):
    """Each gradient term alone, bit for bit (one term: no contraction can change the result); all four together bit for bit, with or
    without the contraction of g_mean * (1 / count) into the addition; every segment size 0 .. 33."""
    rng = np.random.default_rng(D + 2 * use_perm + 4 * accumulate + 8 * (dtype == "bf16"))
    plan = _fan_in_plan(rng)
    x, x_np = _rows(rng, plan.E, D, dtype)
    _, am = _reduce(x, plan, ("max", "min"), dtype)
    args = {"max": am["max"], "min": am["min"]}
    args_np = {"argmax": am["max"].cpu().numpy(), "argmin": am["min"].cpu().numpy()}
    prior, prior_np = _rows(rng, plan.E, D, dtype) if accumulate else (None, None)
    od, recip = OUT[dtype], D % 4 == 0
    for term in ("sum", "mean", "max", "min"):
        g, g_np = _rows(rng, plan.S, D, dtype)
        got = _backward(plan, dtype, D, {term: g}, args, use_perm, prior)
        want = sr.segment_backward(plan.ids, plan.rowptr_np, **{f"g_{term}": g_np}, **args_np, prior=prior_np, reciprocal=recip, out_dtype=od)
        _assert_bits(got, want, f"{dtype} D={D} perm={use_perm} acc={accumulate} g_{term}")
    gs = {k: _rows(rng, plan.S, D, dtype) for k in ("sum", "mean", "max", "min")}
    got = _backward(plan, dtype, D, {k: v[0] for k, v in gs.items()}, args, use_perm, prior)
    want = {contract: sr.segment_backward(plan.ids, plan.rowptr_np, **{f"g_{k}": v[1] for k, v in gs.items()}, **args_np, prior=prior_np,
                                          reciprocal=recip, contract_mean=contract, out_dtype=od)
            for contract in ((False, True) if recip else (False,))}
    bits = _np(got).view(np.uint32)
    match = [c for c, w in want.items() if np.array_equal(bits, w.view(np.uint32))]
    print(f"\nbackward {dtype} D={D} perm={use_perm} accumulate={accumulate}, all four terms: bit-exact "
          f"{'with' if match == [True] else 'without' if match else 'NEITHER with nor without'} the contraction of g_mean * (1 / count)"
          f" ({_ulps(got, want[False], dtype):.0f} ulp from the uncontracted form)")
    assert match


# ------------------------------------------------------------------------------------------------------------------------------------
# paired and multi-source sums
# ------------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("dtype,D,Sa,Sb", [("bf16", 128, 300, 37), ("bf16", 128, 1, 1), ("bf16", 128, 0, 50), ("bf16", 128, 50, 0),
                                           ("bf16", 128, 102, 2000), ("fp32", 128, 300, 37), ("bf16", 132, 300, 37), ("bf16", 3, 40, 41)])
def test_segment_sum_pair_vs_reference(dtype, D, Sa, Sb):
    """hgn_segment_sum_pair against the reference itself: the interleaved bf16 / 128 kernel, and the fall-back to two
    hgn_segment_reduce calls (one side without segments, fp32, D != 128)."""
    rng = np.random.default_rng(Sa * 3 + Sb + D)
    ids_a = _fan_in_plan(rng).ids if Sa == 102 else rng.integers(0, max(Sa - 1, 1), size=1700)    # else the last segment of A stays empty
    E = len(ids_a)
    pa = Plan(ids_a if Sa else np.zeros(0, np.int64), Sa)
    pb = Plan(rng.integers(0, Sb, size=E) if Sb else np.zeros(0, np.int64), Sb)
    x, x_np = _rows(rng, E, D, dtype)
    out_a = torch.full((Sa, D), NAN, dtype=DTYPES[dtype], device="cuda")
    out_b = torch.full((Sb, D), NAN, dtype=DTYPES[dtype], device="cuda")
    _cabi.check(_cabi.load().hgn_segment_sum_pair(_cabi.dtype_code(DTYPES[dtype]), x.data_ptr(), E, D, pa.perm.data_ptr(), pa.rowptr.data_ptr(),
                                                  Sa, out_a.data_ptr(), pb.perm.data_ptr(), pb.rowptr.data_ptr(), Sb, out_b.data_ptr(),
                                                  _cabi.stream_ptr()), "hgn_segment_sum_pair")
    for p, out, tag in ((pa, out_a, "a"), (pb, out_b, "b")):
        _assert_bits(out, sr.segment_sum(x_np[:p.E], p.perm_np, p.rowptr_np, out_dtype=OUT[dtype]), f"pair side {tag}")


def _sources(rng, n, S, D, dtype, sizes):
    """``n`` sources of different element counts into S segments: ([(x, plan)], reference triples)."""
    srcs, ref = [], []
    for k in range(n):
        plan = _fan_in_plan(rng, 1) if k == 0 and S == 34 else Plan(rng.integers(0, S, size=sizes[k]), S)
        x, x_np = _rows(rng, plan.E, D, dtype)
        srcs.append((x, plan))
        ref.append((x_np, plan.perm_np, plan.rowptr_np))
    return srcs, ref


def _multi_sum(srcs, S, D, dtype, base, out):
    ms = ops.SegmentSources()
    ms.n_sources = len(srcs)
    for k, (x, plan) in enumerate(srcs):
        ms.data[k], ms.perm[k], ms.rowptr[k] = x.data_ptr(), plan.perm.data_ptr(), plan.rowptr.data_ptr()
    return _cabi.load().hgn_multi_segment_sum(_cabi.dtype_code(DTYPES[dtype]), ctypes.byref(ms), S, D, _cabi.ptr(base), out.data_ptr(),
                                              _cabi.stream_ptr())


@pytest.mark.parametrize("base_mode", ["none", "separate", "alias"])
@pytest.mark.parametrize("n_sources", [0, 1, 2, 3, 4])
@pytest.mark.parametrize("dtype", list(DTYPES))
def test_multi_segment_sum(dtype, n_sources, base_mode):
    """base first, then sources 0 .. k-1 each in perm order, rounded once; base NULL, a separate tensor, or the output itself."""
    rng = np.random.default_rng(n_sources * 3 + ["none", "separate", "alias"].index(base_mode) + 20 * (dtype == "bf16"))
    S, D = 34, (128 if n_sources != 3 else 260)
    srcs, ref = _sources(rng, n_sources, S, D, dtype, [700, 33, 1500, 1])
    base, base_np = _rows(rng, S, D, dtype) if base_mode != "none" else (None, None)
    out = base if base_mode == "alias" else torch.full((S, D), NAN, dtype=DTYPES[dtype], device="cuda")
    _cabi.check(_multi_sum(srcs, S, D, dtype, base, out), "hgn_multi_segment_sum")
    _assert_bits(out, sr.multi_segment_sum(ref, base_np, (S, D), OUT[dtype]), f"{n_sources} sources, base {base_mode}")


@pytest.mark.parametrize("dtype", list(DTYPES))
def test_multi_segment_sum_chained_like_the_fused_mlp_backward(dtype):
    """ops._FusedMLP.backward with more than four gathered chunks of one source: the first call writes grad_src (base = the dense
    chunk's gradient already in grad_src, i.e. out aliases base), the next call adds the remaining chunks with base = out = grad_src;
    the partial result is rounded to the dtype between the calls."""
    rng = np.random.default_rng(31 + (dtype == "bf16"))
    S, D = 3000, 128
    srcs, ref = _sources(rng, 6, S, D, dtype, [9000, 9000, 2000, 2000, 500, 12000])
    grad_src, dense_np = _rows(rng, S, D, dtype)
    base = grad_src
    for i in range(0, 6, 4):
        _cabi.check(_multi_sum(srcs[i:i + 4], S, D, dtype, base, grad_src), "hgn_multi_segment_sum")
        base = grad_src
    want = sr.multi_segment_sum(ref[:4], dense_np, out_dtype=OUT[dtype])
    want = sr.multi_segment_sum(ref[4:], want, out_dtype=OUT[dtype])
    _assert_bits(grad_src, want, "chained multi-source sum")


# ------------------------------------------------------------------------------------------------------------------------------------
# rows gather / scatter, column sums, refusals, plan
# ------------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("D", [4, 128, 260])
@pytest.mark.parametrize("dtype", list(DTYPES))
def test_rows_gather_scatter(dtype, D):
    """gather dst[i] = src[idx[i]]; scatter dst[idx[i]] = src[i] or, with accumulate, dst[idx[i]] + src[i] rounded once; rows not
    named by idx stay untouched."""
    rng = np.random.default_rng(D + (dtype == "bf16"))
    lib, code, st = _cabi.load(), _cabi.dtype_code(DTYPES[dtype]), _cabi.stream_ptr()
    for n_rows, n in ((50, 0), (50, 1), (5000, 1777), (200_000, 100_000)):
        src, src_np = _rows(rng, n_rows, D, dtype)
        idx_np = rng.permutation(n_rows)[:n]
        idx = torch.from_numpy(idx_np.astype(np.int32)).cuda()
        dst = torch.full((max(n, 1), D), NAN, dtype=DTYPES[dtype], device="cuda")
        _cabi.check(lib.hgn_rows_gather(code, src.data_ptr(), idx.data_ptr(), n, D, dst.data_ptr(), st), "hgn_rows_gather")
        if n:
            _assert_bits(dst, src_np[idx_np], f"gather n={n}")
        rows, rows_np = _rows(rng, n, D, dtype)
        for accumulate in (0, 1):
            table, table_np = _rows(rng, n_rows, D, dtype)
            _cabi.check(lib.hgn_rows_scatter(code, _cabi.ptr(rows) if n else None, idx.data_ptr(), n, D, table.data_ptr(), accumulate, st),
                        "hgn_rows_scatter")
            want = table_np.copy()
            want[idx_np] = rows_np + table_np[idx_np] if accumulate else rows_np
            _assert_bits(table, sr.round_bf16(want) if dtype == "bf16" else want, f"scatter n={n} accumulate={accumulate}")


@pytest.mark.parametrize("rows", [1, 2047, 2049, 3 * 2048 + 5, 1_000_000])
@pytest.mark.parametrize("dtype", list(DTYPES))
def test_colsum_vs_fp64(dtype, rows):
    """hgn_colsum against fp64 within chain length x 2^-24 x sum |x| per column, chain length = rows per row lane + row lanes + row
    blocks (2048 rows per block, 256 / (D / 4) row lanes per block); every width it accepts."""
    lib, code = _cabi.load(), _cabi.dtype_code(DTYPES[dtype])
    torch.manual_seed(rows + (dtype == "bf16"))
    worst = 0.0
    for D in (4, 8, 16, 32, 64, 128, 256):
        x = torch.randn(rows, D, device="cuda").to(DTYPES[dtype])
        out = torch.full((D,), NAN, device="cuda")
        ws = torch.empty(lib.hgn_colsum_workspace_bytes(rows, D), dtype=torch.uint8, device="cuda")
        _cabi.check(lib.hgn_colsum(code, x.data_ptr(), rows, D, out.data_ptr(), ws.data_ptr(), ws.numel(), _cabi.stream_ptr()), "hgn_colsum")
        lanes, blocks = 256 // (D // 4), -(-rows // 2048)
        chain = -(-min(rows, 2048) // lanes) + lanes + blocks
        xd = x.double()
        bound = chain * 2.0 ** -24 * xd.abs().sum(0)
        err = (out.double() - xd.sum(0)).abs()
        assert bool((err <= bound).all()), f"D={D}: error {float(err.max()):.3e} beyond its bound"
        worst = max(worst, float((err / bound).max()))
        del x, xd
    print(f"\ncolsum {dtype} rows={rows}: worst error / bound {worst:.3f}")


def test_argument_refusals():
    lib, st = _cabi.load(), _cabi.stream_ptr()
    bf = _cabi.HGN_BF16
    buf = torch.zeros(4096, dtype=torch.float32, device="cuda")
    plan = Plan(np.array([0, 1, 1]), 2)
    ws = torch.empty(lib.hgn_colsum_workspace_bytes(10, 1024), dtype=torch.uint8, device="cuda")
    for D in (12, 260, 512, 1024):
        assert lib.hgn_colsum(_cabi.HGN_F32, buf.data_ptr(), 2, D, buf.data_ptr(), ws.data_ptr(), ws.numel(), st) == HGN_ERR_INVALID_ARGUMENT, D
    for which in ("max", "min"):
        g = [None, None, buf.data_ptr() if which == "max" else None, buf.data_ptr() if which == "min" else None]
        assert lib.hgn_segment_reduce_bwd(bf, 3, 4, plan.ids32.data_ptr(), plan.perm.data_ptr(), plan.rowptr.data_ptr(), 2, *g, None, None,
                                          buf.data_ptr(), 0, st) == HGN_ERR_INVALID_ARGUMENT, which
    ms = ops.SegmentSources()
    ms.n_sources = 5
    assert lib.hgn_multi_segment_sum(bf, ctypes.byref(ms), 2, 4, None, buf.data_ptr(), st) == HGN_ERR_INVALID_ARGUMENT
    idx = torch.zeros(3, dtype=torch.int32, device="cuda")
    for D in (1, 3, 130):
        assert lib.hgn_rows_gather(bf, buf.data_ptr(), idx.data_ptr(), 3, D, buf.data_ptr(), st) == HGN_ERR_INVALID_ARGUMENT, D
        assert lib.hgn_rows_scatter(bf, buf.data_ptr(), idx.data_ptr(), 3, D, buf.data_ptr(), 1, st) == HGN_ERR_INVALID_ARGUMENT, D
    torch.cuda.synchronize()
    assert (buf == 0).all()


@pytest.mark.parametrize("S", [2, 3, 2 ** 16, 2 ** 16 + 1, 2 ** 20 + 3])
def test_csr_plan_at_sort_width_boundaries(S):
    """hgn_csr_build where the radix sort's key width (bits for ids < S) steps, with the largest id present, and with every element in
    one segment: perm bit-exact with a stable sort, rowptr with the counts' prefix sum."""
    from hgn_b200.plan import segment_plan
    rng = np.random.default_rng(S)
    E = min(3 * S, 1_000_000)
    cases = [rng.integers(0, S, size=E), np.full(E, S - 1), np.zeros(E, dtype=np.int64)]
    cases[0][rng.integers(0, E)] = S - 1
    for ids_np in cases:
        ids = torch.from_numpy(ids_np.astype(np.int64))
        plan = segment_plan(ids.cuda(), S)
        assert torch.equal(plan.perm.cpu()[:E], torch.sort(ids, stable=True).indices.to(torch.int32))
        rowptr = torch.cat([torch.zeros(1, dtype=torch.int64), torch.bincount(ids, minlength=S).cumsum(0)]).to(torch.int32)
        assert torch.equal(plan.rowptr.cpu(), rowptr)
