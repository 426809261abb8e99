"""Autograd glue between torch tensors and the C ABI (``include/hgn_b200.h``).

Two primitives cover every block schedule of the reference's ``src/migration``:

* ``segment_aggregate``  -- ``GraphNet.aggregation`` / ``util.unsorted_segment_operation``
  (graphnet.py:50-70, util.py:92-134): one kernel pass per edge set yields sum / mean / max / min.
* ``fused_mlp``          -- gather + MLP + LayerNorm + residual: ``_update_edge_features`` and the
  ``_update_*node*`` functions (graphnet.py:22-48, 94-124; heterographnet.py:17-33).

torch is used for memory, streams and the autograd graph only; all arithmetic on the path is in
``libhgn_b200.so``.  Nothing here falls back to torch ops: a missing library or a CPU tensor raises.
"""
from __future__ import annotations

import ctypes
from typing import List, Optional, Sequence, Tuple

import torch

from . import _cabi
from ._cabi import AGG_MAX, AGG_MEAN, AGG_MIN, AGG_SUM, Chunks
from .plan import SegmentPlan

D_LATENT = 128
OP_BITS = {"sum": AGG_SUM, "mean": AGG_MEAN, "max": AGG_MAX, "min": AGG_MIN}
PNA_MASK = AGG_SUM | AGG_MEAN | AGG_MAX | AGG_MIN

# launch counter (bench.py reports "gpu_launches": kernels of ours launched in the timed region)
launch_count = 0


def _count(n: int = 1) -> None:
    global launch_count
    launch_count += n


class SegmentSources(ctypes.Structure):
    _fields_ = [("n_sources", ctypes.c_int32), ("data", ctypes.c_void_p * 4), ("perm", ctypes.c_void_p * 4),
                ("rowptr", ctypes.c_void_p * 4)]


# ------------------------------------------------------------------------------------------------
# segment aggregation
# ------------------------------------------------------------------------------------------------
class _SegmentAggregate(torch.autograd.Function):
    @staticmethod
    def forward(ctx, data: torch.Tensor, plan: SegmentPlan, mask: int):
        lib = _cabi.load()
        _cabi.require_cuda(data)
        x = data.contiguous()
        E = x.shape[0]
        D = 1
        for n in x.shape[1:]:
            D *= int(n)
        assert E == plan.num_elements, "segment plan was built for a different number of elements"
        S = plan.num_segments
        out_shape = (S,) + tuple(x.shape[1:])
        need_arg = bool(mask & (AGG_MAX | AGG_MIN)) and data.requires_grad
        outs = {}
        for name, bit in OP_BITS.items():
            outs[name] = torch.empty(out_shape, dtype=x.dtype, device=x.device) if mask & bit else None
        argmax = torch.empty(out_shape, dtype=torch.int32, device=x.device) if (need_arg and mask & AGG_MAX) else None
        argmin = torch.empty(out_shape, dtype=torch.int32, device=x.device) if (need_arg and mask & AGG_MIN) else None
        split = _split_of(plan, S, E) if x.dtype == torch.bfloat16 and D == D_LATENT else None
        with torch.cuda.device(x.device):
            if split is None:
                _cabi.check(lib.hgn_segment_reduce(
                    _cabi.dtype_code(x.dtype), x.data_ptr(), E, D, plan.perm.data_ptr(), plan.rowptr.data_ptr(), S,
                    _cabi.ptr(outs["sum"]), _cabi.ptr(outs["mean"]), _cabi.ptr(outs["max"]), _cabi.ptr(outs["min"]),
                    _cabi.ptr(argmax), _cabi.ptr(argmin), 0, _cabi.stream_ptr()), "hgn_segment_reduce")
                _count()
            else:
                _reduce_split(x, plan, split, [outs[name] for name in OP_BITS], argmax, argmin)
        ctx.plan, ctx.mask, ctx.D, ctx.E = plan, mask, D, E
        ctx.in_shape = tuple(x.shape)
        ctx.save_for_backward(*[t for t in (argmax, argmin) if t is not None])
        ctx.has_argmax, ctx.has_argmin = argmax is not None, argmin is not None
        return tuple(outs[name] for name in OP_BITS if mask & OP_BITS[name])

    @staticmethod
    def backward(ctx, *grads):
        lib = _cabi.load()
        saved = list(ctx.saved_tensors)
        argmax = saved.pop(0) if ctx.has_argmax else None
        argmin = saved.pop(0) if ctx.has_argmin else None
        plan = ctx.plan
        g = {}
        it = iter(grads)
        for name, bit in OP_BITS.items():
            gi = next(it) if ctx.mask & bit else None
            g[name] = gi.contiguous() if gi is not None else None
        ref = next(t for t in g.values() if t is not None)
        grad = torch.empty(ctx.in_shape, dtype=ref.dtype, device=ref.device)
        split = _split_of(plan, plan.num_segments, ctx.E) if ref.dtype == torch.bfloat16 and ctx.D == D_LATENT else None
        with torch.cuda.device(ref.device):
            if split is None:
                _cabi.check(lib.hgn_segment_reduce_bwd(
                    _cabi.dtype_code(ref.dtype), ctx.E, ctx.D, plan.ids32.data_ptr(), plan.perm.data_ptr(), plan.rowptr.data_ptr(),
                    plan.num_segments, _cabi.ptr(g["sum"]), _cabi.ptr(g["mean"]), _cabi.ptr(g["max"]), _cabi.ptr(g["min"]),
                    _cabi.ptr(argmax), _cabi.ptr(argmin), grad.data_ptr(), 0, _cabi.stream_ptr()), "hgn_segment_reduce_bwd")
                _count()
            else:
                _cabi.check(lib.hgn_segment_reduce_bwd_split(
                    _BF, ctx.E, D_LATENT, plan.ids32.data_ptr(), plan.perm.data_ptr(), plan.rowptr.data_ptr(), plan.num_segments,
                    ctypes.byref(split.c), _cabi.ptr(g["sum"]), _cabi.ptr(g["mean"]), _cabi.ptr(g["max"]), _cabi.ptr(g["min"]),
                    _cabi.ptr(argmax), _cabi.ptr(argmin), grad.data_ptr(), _cabi.stream_ptr()), "hgn_segment_reduce_bwd_split")
                _count(2)       # hgn_segment_reduce_bwd_split: segment_bwd_bf16_128_kernel on the short CSR, segment_long_bwd_kernel
        return grad, None, None


def segment_aggregate(data: torch.Tensor, plan: SegmentPlan, ops: Sequence[str]) -> List[torch.Tensor]:
    """Reductions of ``data[E, ...]`` over the plan's segments, in the order of ``ops``."""
    mask = 0
    for op in ops:
        mask |= OP_BITS[op]
    res = _SegmentAggregate.apply(data, plan, mask)
    by_name = dict(zip([n for n in OP_BITS if mask & OP_BITS[n]], res))
    return [by_name[op] for op in ops]


# ------------------------------------------------------------------------------------------------
# fused gather + MLP + LayerNorm + residual
# ------------------------------------------------------------------------------------------------
class ChunkSpec:
    """One 128-wide slice of the MLP input: rows of ``sources[source]`` either gathered through a plan's
    ``ids32`` (sender / receiver latents) or taken densely from ``row_offset``."""
    __slots__ = ("source", "plan", "row_offset")

    def __init__(self, source: int, plan: Optional[SegmentPlan] = None, row_offset: int = 0):
        self.source, self.plan, self.row_offset = source, plan, row_offset


class MLPCall:
    """Static description of one fused call (not a tensor: passed through autograd untouched)."""
    __slots__ = ("rows", "chunks", "resid_source", "resid_offset", "packed_cache")

    def __init__(self, rows, chunks, resid_source, resid_offset, packed_cache):
        self.rows, self.chunks, self.resid_source, self.resid_offset, self.packed_cache = rows, chunks, resid_source, resid_offset, packed_cache


_PACK_EPOCH = [0]


def invalidate_packed_weights() -> None:
    """Drop every staged (packed bf16 / fp32) weight copy.  The staged copies follow ``Parameter._version`` (optimizer steps,
    ``load_state_dict``, in-place ops); writes through ``p.data`` (``p.data.copy_()``, EMA swaps, manual loading) do not bump it --
    call this after such a write."""
    _PACK_EPOCH[0] += 1


def _pack_weights(cache: dict, dtype: torch.dtype, n_chunks: int, params: Sequence[torch.Tensor]) -> torch.Tensor:
    """Layout/precision conversion of the eight parameter tensors, redone only when a parameter changed
    (optimizer steps bump ``_version``)."""
    def pack():
        lib = _cabi.load()
        code = _cabi.dtype_code(dtype)
        blob = torch.empty(lib.hgn_mlp_packed_bytes(code, n_chunks), dtype=torch.uint8, device=params[0].device)
        ps = _master_weights(params)
        _cabi.check(lib.hgn_mlp_pack(code, n_chunks, *[p.data_ptr() for p in ps], blob.data_ptr(), _cabi.stream_ptr()), "hgn_mlp_pack")
        return blob
    return _cached_blob(cache, (dtype, n_chunks), params, pack)


def _master_weights(params: Sequence[torch.Tensor]) -> List[torch.Tensor]:
    ps = [p.detach().contiguous() for p in params]
    if any(p.dtype != torch.float32 for p in ps):
        raise _cabi.HgnError("MLP parameters must be float32 (master weights)")
    return ps


def _cached_blob(cache: dict, key, params: Sequence[torch.Tensor], pack) -> torch.Tensor:
    """``pack()`` (one pack kernel), redone only when a parameter changed (optimizer steps bump ``_version``)."""
    versions = (_PACK_EPOCH[0],) + tuple((p.data_ptr(), p._version) for p in params)
    hit = cache.get(key)
    # While a CUDA graph is being captured the pack kernel always becomes part of the graph: a replay must re-read the master
    # weights the (captured) optimizer step has changed, and the host-side version check does not run at replay time.
    capturing = torch.cuda.is_current_stream_capturing()
    if hit is not None and hit[0] == versions and not capturing:
        return hit[1]
    blob = pack()
    _count()
    if not capturing:
        cache[key] = (versions, blob)
    return blob


def _fill_chunks(call: MLPCall, sources: Sequence[torch.Tensor]) -> Chunks:
    ch = Chunks()
    ch.n_chunks = len(call.chunks)
    for c, spec in enumerate(call.chunks):
        ch.src[c] = sources[spec.source].data_ptr()
        ch.idx[c] = spec.plan.ids32.data_ptr() if spec.plan is not None else None
        ch.row_offset[c] = spec.row_offset
    return ch


class _FusedMLP(torch.autograd.Function):
    @staticmethod
    def forward(ctx, call: MLPCall, W0, b0, W1, b1, W2, b2, gamma, beta, *sources):
        lib = _cabi.load()
        _cabi.require_cuda(*sources)
        srcs = [s.contiguous() for s in sources]
        dtype = srcs[0].dtype
        n_chunks = len(call.chunks)
        if W0.shape != (D_LATENT, D_LATENT * n_chunks) or W1.shape != (D_LATENT, D_LATENT) or W2.shape != (D_LATENT, D_LATENT):
            raise _cabi.HgnError(
                f"fused MLP kernels are specialised for latent 128: got W0 {tuple(W0.shape)} for {n_chunks} chunks, "
                f"W1 {tuple(W1.shape)}, W2 {tuple(W2.shape)}")
        for s in srcs:
            if s.dtype != dtype or s.shape[-1] != D_LATENT:
                raise _cabi.HgnError("fused MLP sources must share one dtype and be 128 wide")
        params = (W0, b0, W1, b1, W2, b2, gamma, beta)
        with torch.cuda.device(srcs[0].device):
            packed = _pack_weights(call.packed_cache, dtype, n_chunks, params)
            ch = _fill_chunks(call, srcs)
            out = torch.empty((call.rows, D_LATENT), dtype=dtype, device=srcs[0].device)
            _cabi.check(lib.hgn_mlp_forward(_cabi.dtype_code(dtype), call.rows, ctypes.byref(ch), packed.data_ptr(),
                                            srcs[call.resid_source].data_ptr(), call.resid_offset, out.data_ptr(),
                                            _cabi.stream_ptr()), "hgn_mlp_forward")
        _count()
        ctx.call = call
        ctx.packed = packed
        ctx.n_sources = len(srcs)
        ctx.save_for_backward(*srcs)
        ctx.param_shapes = [tuple(p.shape) for p in params]
        return out

    @staticmethod
    def backward(ctx, grad_out):
        lib = _cabi.load()
        call: MLPCall = ctx.call
        srcs = list(ctx.saved_tensors)
        dtype = srcs[0].dtype
        dev = srcs[0].device
        code = _cabi.dtype_code(dtype)
        rows = call.rows
        n_chunks = len(call.chunks)
        grad_out = grad_out.contiguous()
        if grad_out.dtype != dtype:
            grad_out = grad_out.to(dtype)
        needs = ctx.needs_input_grad[9:]

        # where does each chunk's data gradient go?
        grad_src: List[Optional[torch.Tensor]] = [None] * len(srcs)
        chunk_bufs: List[Optional[torch.Tensor]] = [None] * n_chunks
        dense_owner = {}          # source -> chunk that writes straight into grad_src
        for c, spec in enumerate(call.chunks):
            if needs[spec.source] and spec.plan is None and spec.source not in dense_owner:
                dense_owner[spec.source] = c
        resid_chunk = -1
        for s, src in enumerate(srcs):
            if not needs[s]:
                continue
            c = dense_owner.get(s)
            if c is not None:
                spec = call.chunks[c]
                full = spec.row_offset == 0 and rows == src.shape[0]
                grad_src[s] = torch.empty_like(src) if full else torch.zeros_like(src)
                chunk_bufs[c] = grad_src[s][spec.row_offset: spec.row_offset + rows]
                if s == call.resid_source and spec.row_offset == call.resid_offset:
                    resid_chunk = c
        for c, spec in enumerate(call.chunks):
            if needs[spec.source] and chunk_bufs[c] is None:
                chunk_bufs[c] = torch.empty((rows, D_LATENT), dtype=dtype, device=dev)

        gparams = [torch.empty(shape, dtype=torch.float32, device=dev) for shape in ctx.param_shapes]
        with torch.cuda.device(dev):
            ch = _fill_chunks(call, srcs)
            ws_bytes = lib.hgn_mlp_backward_workspace_bytes(code, rows, n_chunks)
            ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
            gptrs = (ctypes.c_void_p * n_chunks)(*[b.data_ptr() if b is not None else None for b in chunk_bufs])
            _cabi.check(lib.hgn_mlp_backward(code, rows, ctypes.byref(ch), ctx.packed.data_ptr(), grad_out.data_ptr(), resid_chunk,
                                             gptrs, *[g.data_ptr() for g in gparams], ws.data_ptr(), ws_bytes, _cabi.stream_ptr()),
                        "hgn_mlp_backward")
            _count()
            # scatter the gathered chunks back to their source rows (deterministic, one rounding)
            for s, src in enumerate(srcs):
                if not needs[s]:
                    continue
                gathered = [c for c, spec in enumerate(call.chunks) if spec.source == s and spec.plan is not None]
                extra_dense = [c for c, spec in enumerate(call.chunks)
                               if spec.source == s and spec.plan is None and dense_owner.get(s) != c]
                if gathered:
                    if grad_src[s] is None:
                        base = None
                        grad_src[s] = torch.empty_like(src)
                    else:
                        base = grad_src[s]
                    for i in range(0, len(gathered), 4):
                        part = gathered[i:i + 4]
                        ms = SegmentSources()
                        ms.n_sources = len(part)
                        for k, c in enumerate(part):
                            plan = call.chunks[c].plan
                            ms.data[k] = chunk_bufs[c].data_ptr()
                            ms.perm[k] = plan.perm.data_ptr()
                            ms.rowptr[k] = plan.rowptr.data_ptr()
                        _cabi.check(lib.hgn_multi_segment_sum(code, ctypes.byref(ms), src.shape[0], D_LATENT,
                                                              _cabi.ptr(base), grad_src[s].data_ptr(), _cabi.stream_ptr()),
                                    "hgn_multi_segment_sum")
                        _count()
                        base = grad_src[s]
                elif grad_src[s] is None:
                    grad_src[s] = torch.zeros_like(src)
                for c in extra_dense:   # same source used densely twice: not on any reference path
                    off = call.chunks[c].row_offset
                    grad_src[s][off: off + rows] += chunk_bufs[c]
            if resid_chunk < 0 and needs[call.resid_source]:
                s = call.resid_source
                if grad_src[s] is None:
                    grad_src[s] = torch.zeros_like(srcs[s])
                grad_src[s][call.resid_offset: call.resid_offset + rows] += grad_out
        return (None, *gparams, *grad_src)


def fused_mlp(params: Sequence[torch.Tensor], packed_cache: dict, sources: Sequence[torch.Tensor], chunks: Sequence[ChunkSpec],
              rows: int, resid_source: int, resid_offset: int = 0) -> torch.Tensor:
    """``out[rows,128] = resid + LayerNorm(MLP([chunk_0 | chunk_1 | ...]))``."""
    call = MLPCall(int(rows), list(chunks), int(resid_source), int(resid_offset), packed_cache)
    return _FusedMLP.apply(call, *params, *sources)


# ------------------------------------------------------------------------------------------------
# projected edge update (bf16): node-side pre-projection + fused edge kernels (csrc/edge_tc.cu)
# ------------------------------------------------------------------------------------------------
# One binding per entry point: marshal the pointers, check the return code, count the kernels the C side launches.
_BF = _cabi.HGN_BF16


def _edge_project_forward(v, packed, ps, pr) -> None:
    n = v.shape[0]
    _cabi.check(_cabi.load().hgn_edge_project_forward(_BF, n, v.data_ptr(), packed.data_ptr(), ps.data_ptr(), pr.data_ptr(),
                                                      _cabi.stream_ptr()), "hgn_edge_project_forward")
    _count(int(n > 0))          # edge_project_forward_tc: one proj_tc_kernel


def _edge_project_backward(v, packed, gs, gr, grad_v_add, grad_v, grad_w0, ws=None) -> None:
    lib, n = _cabi.load(), v.shape[0]
    if ws is None:
        ws = torch.empty(lib.hgn_edge_project_backward_workspace_bytes(_BF, n), dtype=torch.uint8, device=v.device)
    _cabi.check(lib.hgn_edge_project_backward(_BF, n, v.data_ptr(), packed.data_ptr(), gs.data_ptr(), gr.data_ptr(), _cabi.ptr(grad_v_add),
                                              grad_v.data_ptr(), grad_w0.data_ptr(), ws.data_ptr(), ws.numel(), _cabi.stream_ptr()),
                "hgn_edge_project_backward")
    _count(4)                   # edge_project_backward_tc: dgrad, pair wgrad, two reduce_w0_block_kernel


def _edge_update_forward(e, ps, pr, s_plan, r_plan, packed, out) -> None:
    E = e.shape[0]
    _cabi.check(_cabi.load().hgn_edge_update_forward(_BF, E, e.data_ptr(), ps.data_ptr(), pr.data_ptr(), s_plan.ids32.data_ptr(),
                                                     r_plan.ids32.data_ptr(), packed.data_ptr(), out.data_ptr(), _cabi.stream_ptr()),
                "hgn_edge_update_forward")
    _count(int(E > 0))          # edge_fwd_tc_launch: one edge_fwd_tc_kernel


def _edge_update_backward(e, ps, pr, s_plan, r_plan, packed, grad_out, grad_agg, grad_e, g0, gparams, ws=None) -> None:
    lib, E = _cabi.load(), e.shape[0]
    if ws is None:
        ws = torch.empty(lib.hgn_edge_update_backward_workspace_bytes(_BF, E), dtype=torch.uint8, device=e.device)
    _cabi.check(lib.hgn_edge_update_backward(
        _BF, E, e.data_ptr(), ps.data_ptr(), pr.data_ptr(), s_plan.ids32.data_ptr(), r_plan.ids32.data_ptr(), packed.data_ptr(),
        _cabi.ptr(grad_out), _cabi.ptr(grad_agg), grad_e.data_ptr(), g0.data_ptr(), *[g.data_ptr() for g in gparams], ws.data_ptr(),
        ws.numel(), _cabi.stream_ptr()), "hgn_edge_update_backward")
    _count(2)                   # projected_backward_launch: edge_bwd_tc_kernel, edge_bwd_reduce_kernel


def _node_update_forward(v, aggs, packed, q1, q2, out) -> None:
    n, k = v.shape[0], len(aggs)
    agg_ptrs = (ctypes.c_void_p * k)(*[a.data_ptr() for a in aggs])
    _cabi.check(_cabi.load().hgn_node_update_forward(_BF, n, v.data_ptr(), k, agg_ptrs, packed.data_ptr(), q1.data_ptr(), _cabi.ptr(q2),
                                                     out.data_ptr(), _cabi.stream_ptr()), "hgn_node_update_forward")
    _count((k + 1) // 2 + 1 if n > 0 else 0)    # node_update_forward_tc: one projection per table of two aggregates, node_fwd_tc


def _node_update_backward(v, aggs, q1, q2, packed, grad_out, grad_v, grad_aggs, gparams, ws=None) -> None:
    lib, n, k = _cabi.load(), v.shape[0], len(aggs)
    if ws is None:
        ws = torch.empty(lib.hgn_node_update_backward_workspace_bytes(_BF, n), dtype=torch.uint8, device=v.device)
    agg_ptrs = (ctypes.c_void_p * k)(*[a.data_ptr() for a in aggs])
    gagg_ptrs = (ctypes.c_void_p * k)(*[g.data_ptr() for g in grad_aggs])
    _cabi.check(lib.hgn_node_update_backward(_BF, n, v.data_ptr(), k, agg_ptrs, q1.data_ptr(), _cabi.ptr(q2), packed.data_ptr(),
                                             grad_out.data_ptr(), grad_v.data_ptr(), gagg_ptrs, *[g.data_ptr() for g in gparams],
                                             ws.data_ptr(), ws.numel(), _cabi.stream_ptr()), "hgn_node_update_backward")
    # node_update_backward_tc: node_bwd_tc and its reduction; per table a dgrad, a pair wgrad and one reduce_w0_block_kernel per aggregate
    _count(2 + 2 * ((k + 1) // 2) + k)


def _split_of(plan: SegmentPlan, S: int, E: int):
    """The plan's split, when the plan has one and the call covers all of its ``S`` segments and ``E`` elements; else ``None`` (the call
    then runs exactly as without a split)."""
    split = plan.split
    return split if split is not None and S == plan.num_segments and E == plan.num_elements else None


def _split_workspace(device, *splits) -> torch.Tensor:
    lib = _cabi.load()
    n = max(lib.hgn_segment_split_reduce_workspace_bytes(ctypes.byref(sp.c)) if sp is not None else 0 for sp in splits)
    return torch.empty(max(n, 1), dtype=torch.uint8, device=device)


def _reduce_split(data, plan: SegmentPlan, split, outs, argmax, argmin) -> None:
    """``hgn_segment_reduce_split`` of bf16 rows of width 128 into ``outs`` = (sum, mean, max, min; None = not requested)."""
    ws = _split_workspace(data.device, split)
    _cabi.check(_cabi.load().hgn_segment_reduce_split(
        _BF, data.data_ptr(), data.shape[0], D_LATENT, plan.perm.data_ptr(), plan.rowptr.data_ptr(), plan.num_segments, ctypes.byref(split.c),
        *[_cabi.ptr(o) for o in outs], _cabi.ptr(argmax), _cabi.ptr(argmin), 0, ws.data_ptr(), ws.numel(), _cabi.stream_ptr()),
        "hgn_segment_reduce_split")
    _count(3)                   # hgn_segment_reduce_split: one kernel on the short CSR, segment_long_partial, segment_long_combine


def _segment_sum(data, plan: SegmentPlan, out) -> None:
    """``out[s] = sum of data's rows in segment s`` for the ``out.shape[0]`` segments of ``plan`` (bf16 rows of width 128)."""
    S = out.shape[0]
    split = _split_of(plan, S, data.shape[0])
    if split is not None:
        _reduce_split(data, plan, split, [out, None, None, None], None, None)
        return
    _cabi.check(_cabi.load().hgn_segment_reduce(_BF, data.data_ptr(), data.shape[0], D_LATENT, plan.perm.data_ptr(), plan.rowptr.data_ptr(),
                                                S, out.data_ptr(), None, None, None, None, None, 0, _cabi.stream_ptr()),
                "hgn_segment_reduce")
    _count(int(S > 0))          # segment_reduce_impl: one kernel


def _segment_reduce(data, plan: SegmentPlan, outs, argmax, argmin) -> None:
    """The reductions ``outs`` = (sum, mean, max, min; None = not requested) of ``data``'s bf16 rows of width 128 over the segments of
    ``plan``, with the max / min winners when ``argmax`` / ``argmin`` are given."""
    S = plan.num_segments
    split = _split_of(plan, S, data.shape[0])
    if split is not None:
        _reduce_split(data, plan, split, outs, argmax, argmin)
        return
    _cabi.check(_cabi.load().hgn_segment_reduce(_BF, data.data_ptr(), data.shape[0], D_LATENT, plan.perm.data_ptr(), plan.rowptr.data_ptr(),
                                                S, *[_cabi.ptr(o) for o in outs], _cabi.ptr(argmax), _cabi.ptr(argmin), 0,
                                                _cabi.stream_ptr()), "hgn_segment_reduce")
    _count(int(S > 0))          # segment_reduce_impl: one kernel


def _segment_layer_grad(plan: SegmentPlan, E: int, grads: dict, argmax, argmin, base, agg_grad, edge_grad) -> None:
    """``agg_grad[r] = g_sum[r] + g_mean[r] / cnt_r`` and ``edge_grad[e] = base[e] + the max / min winners' gradients`` over the receiver
    plan (``grads``: reducer name -> gradient of that aggregate)."""
    S = plan.num_segments
    split = _split_of(plan, S, E)
    if split is not None:
        _cabi.check(_cabi.load().hgn_segment_layer_grad_split(
            _BF, E, D_LATENT, plan.perm.data_ptr(), plan.rowptr.data_ptr(), S, ctypes.byref(split.c),
            *[_cabi.ptr(grads.get(op)) for op in OP_BITS], _cabi.ptr(argmax), _cabi.ptr(argmin), _cabi.ptr(base), _cabi.ptr(agg_grad),
            _cabi.ptr(edge_grad), _cabi.stream_ptr()), "hgn_segment_layer_grad_split")
        # hgn_segment_layer_grad_split: segment_layer_grad_bf16_128_kernel on the short CSR, segment_long_bwd_kernel
        _count(2 * int(agg_grad is not None or edge_grad is not None))
        return
    _cabi.check(_cabi.load().hgn_segment_layer_grad(
        _BF, E, D_LATENT, plan.perm.data_ptr(), plan.rowptr.data_ptr(), S, *[_cabi.ptr(grads.get(op)) for op in OP_BITS],
        _cabi.ptr(argmax), _cabi.ptr(argmin), _cabi.ptr(base), _cabi.ptr(agg_grad), _cabi.ptr(edge_grad), _cabi.stream_ptr()),
        "hgn_segment_layer_grad")
    _count(int(S > 0 and (agg_grad is not None or edge_grad is not None)))     # hgn_segment_layer_grad: one kernel


def _segment_sum_pair(data, plan_a: SegmentPlan, out_a, plan_b: SegmentPlan, out_b) -> None:
    """Two ``_segment_sum``s of the same rows under two groupings."""
    S_a, S_b = out_a.shape[0], out_b.shape[0]
    E = data.shape[0]
    split_a, split_b = _split_of(plan_a, S_a, E), _split_of(plan_b, S_b, E)
    if split_a is not None or split_b is not None:
        ws = _split_workspace(data.device, split_a, split_b)
        _cabi.check(_cabi.load().hgn_segment_sum_pair_split(
            _BF, data.data_ptr(), E, D_LATENT, plan_a.perm.data_ptr(), plan_a.rowptr.data_ptr(), S_a,
            ctypes.byref(split_a.c) if split_a is not None else None, out_a.data_ptr(), plan_b.perm.data_ptr(), plan_b.rowptr.data_ptr(), S_b,
            ctypes.byref(split_b.c) if split_b is not None else None, out_b.data_ptr(), ws.data_ptr(), ws.numel(), _cabi.stream_ptr()),
            "hgn_segment_sum_pair_split")
        # hgn_segment_sum_pair_split: hgn_segment_sum_pair on the short CSRs, then segment_long_partial and _combine per split side
        _count((1 if S_a > 0 and S_b > 0 else int(S_a > 0) + int(S_b > 0)) + 2 * (split_a is not None) + 2 * (split_b is not None))
        return
    _cabi.check(_cabi.load().hgn_segment_sum_pair(_BF, data.data_ptr(), data.shape[0], D_LATENT, plan_a.perm.data_ptr(),
                                                  plan_a.rowptr.data_ptr(), S_a, out_a.data_ptr(), plan_b.perm.data_ptr(),
                                                  plan_b.rowptr.data_ptr(), S_b, out_b.data_ptr(), _cabi.stream_ptr()),
                "hgn_segment_sum_pair")
    _count(1 if S_a > 0 and S_b > 0 else int(S_a > 0) + int(S_b > 0))   # hgn_segment_sum_pair: the paired kernel, else one sum per side


def _rows_add(rows, index32, dst) -> None:
    """``dst[index32[i]] += rows[i]`` (bf16; ``index32`` has no duplicates)."""
    n = rows.shape[0]
    _cabi.check(_cabi.load().hgn_rows_scatter(_BF, rows.data_ptr(), index32.data_ptr(), n, dst.shape[1], dst.data_ptr(), 1,
                                              _cabi.stream_ptr()), "hgn_rows_scatter")
    _count(int(n > 0))          # hgn_rows_scatter: one rows_scatter_kernel


def _segment_partials(data, plan: SegmentPlan, out, minmax: bool, argmax, argmin) -> None:
    """``out[S, HGN_SEGMENT_PARTIAL_WIDTH]`` fp32 = each segment's unrounded sum (and max / min with ``minmax``) and element count, as
    the bf16 segment reductions of ``plan`` would round them (``data``: bf16 rows of width 128)."""
    S, E = plan.num_segments, data.shape[0]
    split = _split_of(plan, S, E)
    ws = _split_workspace(data.device, split)
    _cabi.check(_cabi.load().hgn_segment_partials(
        _BF, data.data_ptr(), E, D_LATENT, plan.perm.data_ptr(), plan.rowptr.data_ptr(), S, ctypes.byref(split.c) if split is not None else None,
        int(minmax), out.data_ptr(), _cabi.ptr(argmax), _cabi.ptr(argmin), ws.data_ptr(), ws.numel(), _cabi.stream_ptr()), "hgn_segment_partials")
    # segment_partial_short_kernel; with a long segment also segment_long_partial and segment_long_partial_combine
    _count(int(S > 0) + 2 * int(S > 0 and split is not None))


def _segment_backward(plan: SegmentPlan, E: int, g_sum, g_max, g_min, argmax, argmin, grad) -> None:
    """``grad[e] = g_sum[r] + the max / min winners' gradients`` over the segments of ``plan`` (bf16 rows of width 128): the backward of
    ``segment_aggregate`` without a 'mean' term."""
    S = plan.num_segments
    split = _split_of(plan, S, E)
    lib = _cabi.load()
    g = [_cabi.ptr(g_sum), None, _cabi.ptr(g_max), _cabi.ptr(g_min), _cabi.ptr(argmax), _cabi.ptr(argmin)]
    if split is not None:
        _cabi.check(lib.hgn_segment_reduce_bwd_split(_BF, E, D_LATENT, plan.ids32.data_ptr(), plan.perm.data_ptr(), plan.rowptr.data_ptr(), S,
                                                     ctypes.byref(split.c), *g, grad.data_ptr(), _cabi.stream_ptr()), "hgn_segment_reduce_bwd_split")
        _count(2)               # segment_bwd_bf16_128_kernel on the short CSR, segment_long_bwd_kernel
        return
    _cabi.check(lib.hgn_segment_reduce_bwd(_BF, E, D_LATENT, plan.ids32.data_ptr(), plan.perm.data_ptr(), plan.rowptr.data_ptr(), S, *g,
                                           grad.data_ptr(), 0, _cabi.stream_ptr()), "hgn_segment_reduce_bwd")
    _count()                    # one backward kernel


def _cluster_combine(slots, world: int, rank: int, outs, argmax, argmin, count) -> None:
    """Rank-ordered reduction of every rank's partial rows ``slots[world, C, HGN_SEGMENT_PARTIAL_WIDTH]`` into ``outs`` = (sum, mean, max,
    min; None = not wanted), bf16 ``[C, 128]``; clears this rank's winners where another rank won and writes the total counts."""
    C = slots.shape[1]
    _cabi.check(_cabi.load().hgn_cluster_combine(slots.data_ptr(), world, rank, C, *[_cabi.ptr(o) for o in outs], _cabi.ptr(argmax),
                                                 _cabi.ptr(argmin), _cabi.ptr(count), _cabi.stream_ptr()), "hgn_cluster_combine")
    _count(int(C > 0))          # one cluster_combine_kernel


def _cluster_grad_sum(slots, out) -> None:
    """``out[C, D] = sum over ranks, in rank order, of slots[r]`` (bf16 rows, fp32 accumulation, one rounding)."""
    world, C, D = slots.shape
    _cabi.check(_cabi.load().hgn_cluster_grad_sum(_BF, slots.data_ptr(), world, C, D, out.data_ptr(), _cabi.stream_ptr()), "hgn_cluster_grad_sum")
    _count(int(C * D > 0))      # one cluster_grad_sum_kernel


def _cluster_mean_grad(g_sum, g_mean, count, out) -> None:
    """``out = g_sum + g_mean / count`` per cluster row (bf16 ``[C, 128]``, one rounding)."""
    C = g_mean.shape[0]
    _cabi.check(_cabi.load().hgn_cluster_mean_grad(_cabi.ptr(g_sum), g_mean.data_ptr(), count.data_ptr(), C, out.data_ptr(), _cabi.stream_ptr()),
                "hgn_cluster_mean_grad")
    _count(int(C > 0))          # one cluster_mean_grad_kernel


class _NodeProjection(torch.autograd.Function):
    """``Ps = v W0[:, 0:128]^T``, ``Pr = v W0[:, 128:256]^T`` -- the sender / receiver blocks of the edge MLP's first
    linear (graphnet.py:28-31 concatenation order), applied once per node instead of once per edge."""

    @staticmethod
    def forward(ctx, v, W0, packed):
        n = v.shape[0]
        ps = torch.empty((n, D_LATENT), dtype=v.dtype, device=v.device)
        pr = torch.empty((n, D_LATENT), dtype=v.dtype, device=v.device)
        with torch.cuda.device(v.device):
            _edge_project_forward(v, packed, ps, pr)
        ctx.save_for_backward(v)
        ctx.packed = packed
        ctx.w0_shape = tuple(W0.shape)
        return ps, pr

    @staticmethod
    def backward(ctx, gs, gr):
        (v,) = ctx.saved_tensors
        gs = gs.contiguous() if gs is not None else torch.zeros_like(v)
        gr = gr.contiguous() if gr is not None else torch.zeros_like(v)
        grad_v = torch.empty_like(v)
        grad_w0 = torch.zeros(ctx.w0_shape, dtype=torch.float32, device=v.device)
        with torch.cuda.device(v.device):
            _edge_project_backward(v, ctx.packed, gs, gr, None, grad_v, grad_w0)
        return grad_v, grad_w0, None


class _EdgeUpdate(torch.autograd.Function):
    """``e' = e + LN(MLP(Ps[s] + Pr[r] + We e ...))`` and, when ``want_agg``, ``agg = segment_sum(e', receivers)``.
    Returning the aggregate from the same node of the autograd graph lets the backward kernel gather its gradient
    through ``receivers`` instead of materialising it as an ``[E,128]`` tensor and adding it to the next layer's."""

    @staticmethod
    def forward(ctx, ps, pr, e, W0, b0, W1, b1, W2, b2, gamma, beta, packed, s_plan, r_plan, want_agg):
        out = torch.empty_like(e)
        with torch.cuda.device(e.device):
            _edge_update_forward(e, ps, pr, s_plan, r_plan, packed, out)
            agg = None
            if want_agg:
                agg = torch.empty((r_plan.num_segments, D_LATENT), dtype=e.dtype, device=e.device)
                _segment_sum(out, r_plan, agg)
        ctx.save_for_backward(e, ps, pr)              # the hidden activations are recomputed by the backward kernel
        ctx.n_nodes = ps.shape[0]
        ctx.packed, ctx.s_plan, ctx.r_plan = packed, s_plan, r_plan
        ctx.param_shapes = [tuple(p.shape) for p in (W0, b0, W1, b1, W2, b2, gamma, beta)]
        if want_agg:
            return out, agg
        return out, None

    @staticmethod
    def backward(ctx, grad_out, grad_agg):
        e, ps, pr = ctx.saved_tensors
        dev = e.device
        n = ctx.n_nodes
        if grad_out is not None:
            grad_out = grad_out.contiguous().to(e.dtype)
        if grad_agg is not None:
            grad_agg = grad_agg.contiguous().to(e.dtype)
        grad_e = torch.empty_like(e)
        g0 = torch.empty_like(e)
        gparams = [torch.zeros(shape, dtype=torch.float32, device=dev) if i == 0 else torch.empty(shape, dtype=torch.float32, device=dev)
                   for i, shape in enumerate(ctx.param_shapes)]
        gs = torch.empty((n, D_LATENT), dtype=e.dtype, device=dev)
        gr = torch.empty((n, D_LATENT), dtype=e.dtype, device=dev)
        with torch.cuda.device(dev):
            _edge_update_backward(e, ps, pr, ctx.s_plan, ctx.r_plan, ctx.packed, grad_out, grad_agg, grad_e, g0, gparams)
            # d loss / d Ps, d Pr: sender- and receiver-keyed segment sums of G0 (deterministic CSR passes)
            _segment_sum_pair(g0, ctx.s_plan, gs, ctx.r_plan, gr)
        return (gs, gr, grad_e, *gparams, None, None, None, None)


def edge_update(params: Sequence[torch.Tensor], packed_cache: dict, v: torch.Tensor, e: torch.Tensor, s_plan: SegmentPlan,
                r_plan: SegmentPlan, want_agg: bool):
    """Projected bf16 edge update (graphnet.py:22-32).  Returns ``(e', agg)`` where ``agg`` is the receiver-keyed 'sum'
    aggregate of ``e'`` when ``want_agg`` else ``None``."""
    _cabi.require_cuda(v, e)
    if v.dtype != torch.bfloat16 or e.dtype != torch.bfloat16:
        raise _cabi.HgnError("edge_update is the bf16 tcgen05 path; fp32 features go through fused_mlp")
    W0 = params[0]
    if W0.shape != (D_LATENT, 3 * D_LATENT) or v.shape[-1] != D_LATENT or e.shape[-1] != D_LATENT:
        raise _cabi.HgnError(f"edge_update is specialised for latent 128: W0 {tuple(W0.shape)}, v {tuple(v.shape)}, e {tuple(e.shape)}")
    v, e = v.contiguous(), e.contiguous()
    with torch.cuda.device(v.device):
        packed = _pack_weights(packed_cache, torch.bfloat16, 3, params)
    ps, pr = _NodeProjection.apply(v, W0, packed)
    return _EdgeUpdate.apply(ps, pr, e, *params, packed, s_plan, r_plan, bool(want_agg))


class _NodeUpdate(torch.autograd.Function):
    """``v' = v + LN(MLP([v | agg_1 | ... | agg_n]))`` (graphnet.py:34-48, one edge set: n = 1, or 4 for 'pna') on the projected
    kernels: the aggregates' blocks of the first linear are applied once per node row into one or two tables
    (``q1 = agg_1 Wa_1^T + agg_2 Wa_2^T``, ``q2 = agg_3 Wa_3^T + agg_4 Wa_4^T``) that enter the fused kernel as table rows."""

    @staticmethod
    def forward(ctx, v, W0, b0, W1, b1, W2, b2, gamma, beta, packed, *aggs):
        k = len(aggs)
        q1 = torch.empty_like(v)
        q2 = torch.empty_like(v) if k > 2 else None
        out = torch.empty_like(v)
        with torch.cuda.device(v.device):
            _node_update_forward(v, aggs, packed, q1, q2, out)
        ctx.save_for_backward(v, *aggs, q1, *([q2] if q2 is not None else []))
        ctx.k = k
        ctx.packed = packed
        ctx.param_shapes = [tuple(p.shape) for p in (W0, b0, W1, b1, W2, b2, gamma, beta)]
        return out

    @staticmethod
    def backward(ctx, grad_out):
        saved = list(ctx.saved_tensors)
        k = ctx.k
        v, aggs, rest = saved[0], saved[1:1 + k], saved[1 + k:]
        q1 = rest[0]
        q2 = rest[1] if len(rest) > 1 else None
        dev = v.device
        grad_out = grad_out.contiguous().to(v.dtype)
        grad_v = torch.empty_like(v)
        grad_aggs = [torch.empty_like(a) for a in aggs]
        gparams = [torch.empty(shape, dtype=torch.float32, device=dev) for shape in ctx.param_shapes]
        with torch.cuda.device(dev):
            _node_update_backward(v, aggs, q1, q2, ctx.packed, grad_out, grad_v, grad_aggs, gparams)
        return (grad_v, *gparams, None, *grad_aggs)


def node_update(params: Sequence[torch.Tensor], packed_cache: dict, v: torch.Tensor, aggs) -> torch.Tensor:
    """Projected bf16 node update ``v + LN(MLP([v | agg_1 | ... | agg_n]))`` with 1 to 4 aggregates (one tensor or a sequence)."""
    if isinstance(aggs, torch.Tensor):
        aggs = [aggs]
    aggs = list(aggs)
    _cabi.require_cuda(v, *aggs)
    if v.dtype != torch.bfloat16 or any(a.dtype != torch.bfloat16 for a in aggs):
        raise _cabi.HgnError("node_update is the bf16 tcgen05 path; fp32 features go through fused_mlp")
    W0, k = params[0], len(aggs)
    if (not 1 <= k <= 4 or W0.shape != (D_LATENT, (1 + k) * D_LATENT) or any(a.shape != v.shape for a in aggs)
            or v.shape[-1] != D_LATENT or v.shape[0] == 0):
        raise _cabi.HgnError(f"node_update is specialised for latent 128 and 1..4 aggregates: W0 {tuple(W0.shape)}, v {tuple(v.shape)}, "
                             f"{k} aggregates")
    v = v.contiguous()
    aggs = [a.contiguous() for a in aggs]
    with torch.cuda.device(v.device):
        packed = _pack_weights(packed_cache, torch.bfloat16, 1 + k, params)
    return _NodeUpdate.apply(v, *params, packed, *aggs)


def _layer_workspace(n: int, E: int, device) -> torch.Tensor:
    """One workspace for the backward entry points of a layer of ``n`` nodes and ``E`` edges (they run one after another on one
    stream)."""
    lib = _cabi.load()
    nbytes = max(lib.hgn_node_update_backward_workspace_bytes(_BF, n), lib.hgn_edge_update_backward_workspace_bytes(_BF, E),
                 lib.hgn_edge_project_backward_workspace_bytes(_BF, n))
    return torch.empty(nbytes, dtype=torch.uint8, device=device)


class _GraphNetLayer(torch.autograd.Function):
    """One whole ``GraphNet`` block with ONE edge set (graphnet.py:72-84) as a single autograd node, for the reducers of its
    aggregator (``('sum',)``, ``('mean',)``, ``('max',)``, ``('min',)`` or the four of 'pna', in the order of graphnet.py:53-64):

        forward   node projection -> fused edge update -> receiver aggregate(s) -> aggregate projection + fused node update
        backward  fused node backward -> [not 'sum': incoming gradient of e' from the aggregate gradients] -> fused edge backward
                  (the 'sum' / 'mean' share of the aggregate gradient gathered inside) -> sender / receiver sums of G0 -> node-level
                  dgrad with the node update's share of d loss / d v added in its epilogue -> node-level wgrads

    Same kernels and same forward arithmetic as ``edge_update`` + ``segment_aggregate`` / the edge update's 'sum' + ``node_update``;
    what goes away is the autograd glue between them: the bf16 ``at::add`` of the two partial gradients of ``v`` (the node update's
    share is added in fp32 instead), zero fills, four autograd nodes' worth of Python per layer, and for a non-'sum' aggregator the
    dense ``[E,128]`` aggregate gradient and its ``at::add`` to the next layer's d e' (``hgn_segment_layer_grad`` writes per-node rows
    for 'sum' / 'mean' and adds the max / min winners to d e' in one pass).

    ``halo`` (not a tensor: passed through untouched, like the plans) makes this the block of one rank of a partitioned graph
    (``partition.PeerLayerHalo``).  ``v`` then holds the owned nodes, and the senders index ``[owned | ghosts]``.  The halo provides
    the sender table ``Ps`` (``[n_own + n_ghost, 128]``; this rank writes the owned rows), a forward exchange that fills the ghost
    rows after the projection, and a backward exchange that sends the ghost rows of the sender sums home and adds the rows the peers
    return into the owned ones.  Every edge of an owned receiver is local, so the aggregates and the max / min winners are complete
    without further exchanges.  Everything else is this schedule, so an owned row sees the kernels and the rounding points of the
    one-GPU layer."""

    @staticmethod
    def forward(ctx, v, e, s_plan, r_plan, packed_e, packed_n, halo, reducers, *params):
        k = len(reducers)
        ps = halo.sender_table() if halo is not None else torch.empty_like(v)
        pr, q1 = torch.empty_like(v), torch.empty_like(v)
        q2 = torch.empty_like(v) if k > 2 else None
        e_new, v_new = torch.empty_like(e), torch.empty_like(v)
        aggs = [torch.empty_like(v) for _ in reducers]
        winners = any(ctx.needs_input_grad)             # the backward needs the max / min winners
        new_arg = lambda op: torch.empty(v.shape, dtype=torch.int32, device=v.device) if winners and op in reducers else None
        argmax, argmin = new_arg("max"), new_arg("min")
        with torch.cuda.device(v.device):
            _edge_project_forward(v, packed_e, ps, pr)
            if halo is not None:
                halo.exchange_forward()
            _edge_update_forward(e, ps, pr, s_plan, r_plan, packed_e, e_new)
            if reducers == ("sum",):
                _segment_sum(e_new, r_plan, aggs[0])
            else:
                by_op = dict(zip(reducers, aggs))
                _segment_reduce(e_new, r_plan, [by_op.get(op) for op in OP_BITS], argmax, argmin)
            _node_update_forward(v, aggs, packed_n, q1, q2, v_new)
        ctx.save_for_backward(v, e, ps, pr, q1, q2, argmax, argmin, *aggs)
        ctx.plans, ctx.packed, ctx.halo, ctx.reducers = (s_plan, r_plan), (packed_e, packed_n), halo, reducers
        ctx.param_shapes = [tuple(p.shape) for p in params]
        return v_new, e_new

    @staticmethod
    def backward(ctx, grad_v_new, grad_e_new):
        v, e, ps, pr, q1, q2, argmax, argmin, *aggs = ctx.saved_tensors
        s_plan, r_plan = ctx.plans
        packed_e, packed_n = ctx.packed
        dev = v.device
        grad_v_new = grad_v_new.contiguous().to(v.dtype) if grad_v_new is not None else torch.zeros_like(v)
        grad_e_new = grad_e_new.contiguous().to(e.dtype) if grad_e_new is not None else None
        new = lambda like: torch.empty_like(like)
        grad_v_node, grad_v, gs, gr = new(v), new(v), new(ps), new(v)
        grad_aggs = [new(v) for _ in aggs]
        grad_e, g0 = new(e), new(e)
        ge = [torch.empty(shape, dtype=torch.float32, device=dev) for shape in ctx.param_shapes[:8]]
        gn = [torch.empty(shape, dtype=torch.float32, device=dev) for shape in ctx.param_shapes[8:]]
        with torch.cuda.device(dev):
            ws = _layer_workspace(v.shape[0], e.shape[0], dev)
            _node_update_backward(v, aggs, q1, q2, packed_n, grad_v_new, grad_v_node, grad_aggs, gn, ws)
            if ctx.reducers == ("sum",):
                grad_out, grad_agg = grad_e_new, grad_aggs[0]
            else:
                g = dict(zip(ctx.reducers, grad_aggs))
                grad_agg = new(v) if "sum" in g or "mean" in g else None
                edge_grad = new(e) if "max" in g or "min" in g else None
                _segment_layer_grad(r_plan, e.shape[0], g, argmax, argmin, grad_e_new if edge_grad is not None else None, grad_agg,
                                    edge_grad)
                grad_out = edge_grad if edge_grad is not None else grad_e_new
            _edge_update_backward(e, ps, pr, s_plan, r_plan, packed_e, grad_out, grad_agg, grad_e, g0, ge, ws)
            _segment_sum_pair(g0, s_plan, gs, r_plan, gr)
            if ctx.halo is not None:
                ctx.halo.exchange_backward(gs)
            # the edge backward wrote only the We block of d W0 (columns 256:384); the node-level kernel fills columns 0:256
            _edge_project_backward(v, packed_e, gs, gr, grad_v_node, grad_v, ge[0], ws)
        return (grad_v, grad_e, None, None, None, None, None, None, *ge, *gn)


def graphnet_layer(edge_params: Sequence[torch.Tensor], edge_cache: dict, node_params: Sequence[torch.Tensor], node_cache: dict,
                   v: torch.Tensor, e: torch.Tensor, s_plan: SegmentPlan, r_plan: SegmentPlan, aggregator: str, halo=None):
    """``(v', e')`` of one GraphNet block (one edge set, bf16 latents of width 128) with ``aggregator`` 'sum', 'mean', 'max', 'min' or
    'pna': see ``_GraphNetLayer``."""
    _cabi.require_cuda(v, e)
    if aggregator != "pna" and aggregator not in OP_BITS:
        raise _cabi.HgnError(f"graphnet_layer: unknown aggregator {aggregator!r}")
    reducers = tuple(OP_BITS) if aggregator == "pna" else (aggregator,)
    if v.dtype != torch.bfloat16 or e.dtype != torch.bfloat16 or v.shape[-1] != D_LATENT or e.shape[-1] != D_LATENT:
        raise _cabi.HgnError("graphnet_layer is the bf16 tcgen05 path for latent 128")
    if edge_params[0].shape != (D_LATENT, 3 * D_LATENT) or node_params[0].shape != (D_LATENT, (1 + len(reducers)) * D_LATENT):
        raise _cabi.HgnError(f"graphnet_layer ({aggregator}): first linears {tuple(edge_params[0].shape)} / {tuple(node_params[0].shape)}")
    v, e = v.contiguous(), e.contiguous()
    with torch.cuda.device(v.device):
        packed_e = _pack_weights(edge_cache, torch.bfloat16, 3, edge_params)
        packed_n = _pack_weights(node_cache, torch.bfloat16, 1 + len(reducers), node_params)
    return _GraphNetLayer.apply(v, e, s_plan, r_plan, packed_e, packed_n, halo, reducers, *edge_params, *node_params)


def graphnet_sum_layer(edge_params: Sequence[torch.Tensor], edge_cache: dict, node_params: Sequence[torch.Tensor], node_cache: dict,
                       v: torch.Tensor, e: torch.Tensor, s_plan: SegmentPlan, r_plan: SegmentPlan, halo=None):
    """``graphnet_layer`` with the 'sum' aggregator."""
    return graphnet_layer(edge_params, edge_cache, node_params, node_cache, v, e, s_plan, r_plan, "sum", halo)


def colsum(x: torch.Tensor) -> torch.Tensor:
    """fp32 column sums of ``x[rows, D]`` (deterministic)."""
    lib = _cabi.load()
    _cabi.require_cuda(x)
    x = x.contiguous()
    rows, D = x.shape
    out = torch.empty(D, dtype=torch.float32, device=x.device)
    ws_bytes = lib.hgn_colsum_workspace_bytes(rows, D)
    ws = torch.empty(max(ws_bytes, 4), dtype=torch.uint8, device=x.device)
    with torch.cuda.device(x.device):
        _cabi.check(lib.hgn_colsum(_cabi.dtype_code(x.dtype), x.data_ptr(), rows, D, out.data_ptr(), ws.data_ptr(), ws_bytes,
                                   _cabi.stream_ptr()), "hgn_colsum")
    _count(2)
    return out


# ------------------------------------------------------------------------------------------------
# encoder / decoder MLPs (bf16 tcgen05, csrc/io_mlp_tc.cu): raw fp32 features -> bf16 latents, bf16 latents -> fp32 outputs
# ------------------------------------------------------------------------------------------------
IO_ENCODER, IO_DECODER = 0, 1
IO_MAX_OUT = 16
_IO_SLAB_ROWS = 1 << 21          # rows per backward pass (io_bwd_layout)


def _io_backward_launches(rows: int) -> int:
    """Kernels of one hgn_encoder_backward / hgn_decoder_backward: per pass the data-gradient kernel (rows > 0), the weight-gradient
    GEMMs and the two colsum5 kernels; then one reduction."""
    passes = max(1, -(-rows // _IO_SLAB_ROWS))
    return passes * (3 + int(rows > 0)) + 1


def io_mlp_pack(cache: dict, kind: int, width: int, params: Sequence[torch.Tensor]) -> torch.Tensor:
    """Packed bf16 blob of an encoder (``width`` = K, eight tensors) or decoder (``width`` = n_out, six tensors) MLP."""
    def pack():
        lib = _cabi.load()
        blob = torch.empty(lib.hgn_io_mlp_packed_bytes(), dtype=torch.uint8, device=params[0].device)
        ps = _master_weights(params)
        gamma_beta = [p.data_ptr() for p in ps[6:8]] if kind == IO_ENCODER else [None, None]
        _cabi.check(lib.hgn_io_mlp_pack(kind, width, *[p.data_ptr() for p in ps[:6]], *gamma_beta, blob.data_ptr(), _cabi.stream_ptr()),
                    "hgn_io_mlp_pack")
        return blob
    return _cached_blob(cache, ("io", kind, width), params, pack)


class _EncoderMLP(torch.autograd.Function):
    """``LN(W2 relu(W1 relu(W0 x + b0) + b1) + b2)`` of raw fp32 features ``x[R, K]`` -> bf16 ``[R, 128]``."""

    @staticmethod
    def forward(ctx, x, packed, W0, b0, W1, b1, W2, b2, gamma, beta):
        rows, k = x.shape
        out = torch.empty((rows, D_LATENT), dtype=torch.bfloat16, device=x.device)
        with torch.cuda.device(x.device):
            _cabi.check(_cabi.load().hgn_encoder_forward(rows, k, _cabi.ptr(x), packed.data_ptr(), _cabi.ptr(out), _cabi.stream_ptr()),
                        "hgn_encoder_forward")
        _count(int(rows > 0))    # one io_mlp_tc_kernel
        ctx.save_for_backward(x)
        ctx.packed = packed
        ctx.param_shapes = [tuple(p.shape) for p in (W0, b0, W1, b1, W2, b2, gamma, beta)]
        return out

    @staticmethod
    def backward(ctx, grad_out):
        (x,) = ctx.saved_tensors
        rows, k = x.shape
        dev = x.device
        lib = _cabi.load()
        grad_out = grad_out.contiguous().to(torch.bfloat16)
        grad_x = torch.empty_like(x) if ctx.needs_input_grad[0] else None
        gparams = [torch.empty(shape, dtype=torch.float32, device=dev) for shape in ctx.param_shapes]
        with torch.cuda.device(dev):
            ws_bytes = lib.hgn_encoder_backward_workspace_bytes(rows, k)
            ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
            _cabi.check(lib.hgn_encoder_backward(rows, k, _cabi.ptr(x), ctx.packed.data_ptr(), _cabi.ptr(grad_out), _cabi.ptr(grad_x),
                                                 *[g.data_ptr() for g in gparams], ws.data_ptr(), ws_bytes, _cabi.stream_ptr()),
                        "hgn_encoder_backward")
        _count(_io_backward_launches(rows))
        return (grad_x, None, *gparams)


class _DecoderMLP(torch.autograd.Function):
    """``W2 relu(W1 relu(W0 x + b0) + b1) + b2`` of bf16 latents ``x[N, 128]`` -> fp32 ``[N, n_out]``."""

    @staticmethod
    def forward(ctx, x, packed, W0, b0, W1, b1, W2, b2):
        rows, n_out = x.shape[0], W2.shape[0]
        out = torch.empty((rows, n_out), dtype=torch.float32, device=x.device)
        with torch.cuda.device(x.device):
            _cabi.check(_cabi.load().hgn_decoder_forward(rows, n_out, _cabi.ptr(x), packed.data_ptr(), _cabi.ptr(out), _cabi.stream_ptr()),
                        "hgn_decoder_forward")
        _count(int(rows > 0))    # one io_mlp_tc_kernel
        ctx.save_for_backward(x)
        ctx.packed = packed
        ctx.n_out = n_out
        ctx.param_shapes = [tuple(p.shape) for p in (W0, b0, W1, b1, W2, b2)]
        return out

    @staticmethod
    def backward(ctx, grad_out):
        (x,) = ctx.saved_tensors
        rows, dev = x.shape[0], x.device
        lib = _cabi.load()
        grad_out = grad_out.contiguous().to(torch.float32)
        grad_x = torch.empty_like(x)
        gparams = [torch.empty(shape, dtype=torch.float32, device=dev) for shape in ctx.param_shapes]
        with torch.cuda.device(dev):
            ws_bytes = lib.hgn_decoder_backward_workspace_bytes(rows, ctx.n_out)
            ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
            _cabi.check(lib.hgn_decoder_backward(rows, ctx.n_out, _cabi.ptr(x), ctx.packed.data_ptr(), _cabi.ptr(grad_out), _cabi.ptr(grad_x),
                                                 *[g.data_ptr() for g in gparams], ws.data_ptr(), ws_bytes, _cabi.stream_ptr()),
                        "hgn_decoder_backward")
        _count(_io_backward_launches(rows))
        return (grad_x, None, *gparams)


def encoder_mlp(params: Sequence[torch.Tensor], packed_cache: dict, x: torch.Tensor) -> torch.Tensor:
    """bf16 ``[R, 128]`` latents of raw fp32 features ``x[R, K]`` (1 <= K <= 128) through the eight tensors of a reference encoder
    MLP ``Sequential(LazyMLP([128, 128, 128]), LayerNorm(128))``."""
    _cabi.require_cuda(x)
    if x.dtype != torch.float32 or x.dim() != 2:
        raise _cabi.HgnError(f"encoder kernel takes fp32 [rows, K] features: got {x.dtype} {tuple(x.shape)}")
    k = x.shape[1]
    W0, b0, W1, b1, W2, b2, gamma, beta = params
    if not 1 <= k <= D_LATENT or W0.shape != (D_LATENT, k) or W1.shape != (D_LATENT, D_LATENT) or W2.shape != (D_LATENT, D_LATENT) \
            or any(p.shape != (D_LATENT,) for p in (b0, b1, b2, gamma, beta)):
        raise _cabi.HgnError(f"encoder kernel is specialised for 1 <= K <= 128 inputs and latent 128: got K={k}, W0 {tuple(W0.shape)}, "
                             f"W1 {tuple(W1.shape)}, W2 {tuple(W2.shape)}")
    x = x.contiguous()
    with torch.cuda.device(x.device):
        packed = io_mlp_pack(packed_cache, IO_ENCODER, k, params)
    return _EncoderMLP.apply(x, packed, *params)


def decoder_mlp(params: Sequence[torch.Tensor], packed_cache: dict, x: torch.Tensor) -> torch.Tensor:
    """fp32 ``[N, n_out]`` outputs (1 <= n_out <= 16) of bf16 latents ``x[N, 128]`` through the six tensors of a reference decoder
    MLP ``LazyMLP([128, 128, n_out])``."""
    _cabi.require_cuda(x)
    if x.dtype != torch.bfloat16 or x.dim() != 2 or x.shape[1] != D_LATENT:
        raise _cabi.HgnError(f"decoder kernel takes bf16 [rows, 128] latents: got {x.dtype} {tuple(x.shape)}")
    W0, b0, W1, b1, W2, b2 = params
    n_out = W2.shape[0]
    if not 1 <= n_out <= IO_MAX_OUT or W0.shape != (D_LATENT, D_LATENT) or W1.shape != (D_LATENT, D_LATENT) \
            or W2.shape != (n_out, D_LATENT) or b0.shape != (D_LATENT,) or b1.shape != (D_LATENT,) or b2.shape != (n_out,):
        raise _cabi.HgnError(f"decoder kernel is specialised for latent 128 and 1 <= n_out <= {IO_MAX_OUT}: got W0 {tuple(W0.shape)}, "
                             f"W1 {tuple(W1.shape)}, W2 {tuple(W2.shape)}")
    x = x.contiguous()
    with torch.cuda.device(x.device):
        packed = io_mlp_pack(packed_cache, IO_DECODER, n_out, params)
    return _DecoderMLP.apply(x, packed, *params)
