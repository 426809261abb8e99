"""Topology plans: int32 index copies and receiver-/sender-sorted CSR views of an index vector.

The reference re-expands ``receivers`` to an ``[E,128]`` int64 index on every aggregation
(src/util.py:105-110) and moves the index tensors to the device on every use (graphnet.py:25-26).
Mesh topology is constant along a trajectory, so here each distinct index tensor gets one cached
``SegmentPlan``: the int32 copy used as gather index by the MLP tile kernels, and -- built on first
need by ``hgn_csr_build`` (stable sort on the device) -- the CSR view used by the aggregation
forward and by the deterministic gather backward.
"""
from __future__ import annotations

from collections import OrderedDict
import ctypes
import os as _os
import weakref as _weakref

import torch

from . import _cabi



class SegmentSplit:
    """The long segments of a CSR (more than ``hgn_segment_split_threshold()`` elements, cut into pieces of
    ``hgn_segment_split_piece()`` perm positions) and the short CSR without them, as built by ``hgn_segment_split_build``.
    ``c`` is the ``hgn_segment_split`` the ``*_split`` entry points take; the tensors it points into are held here."""

    __slots__ = ("n_long", "n_pieces", "n_short", "long_ids", "piece_ptr", "pieces", "perm_short", "rowptr_short", "c", "nbytes")

    def __init__(self, perm: torch.Tensor, rowptr: torch.Tensor, E: int, S: int):
        lib = _cabi.load()
        dev = rowptr.device
        max_long = lib.hgn_segment_split_max_long(E, S)
        i32 = dict(dtype=torch.int32, device=dev)
        long_ids = torch.empty(max(max_long, 1), **i32)
        piece_ptr = torch.empty(max_long + 1, **i32)
        pieces = torch.empty(max(3 * lib.hgn_segment_split_max_pieces(E), 1), **i32)
        perm_short = torch.empty(max(E, 1), **i32)
        self.rowptr_short = torch.empty(S + 1, **i32)
        ws_bytes = lib.hgn_segment_split_build_workspace_bytes(E, S)
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        counts = (ctypes.c_int64 * 3)()
        with torch.cuda.device(dev):
            _cabi.check(lib.hgn_segment_split_build(perm.data_ptr(), rowptr.data_ptr(), E, S, long_ids.data_ptr(), piece_ptr.data_ptr(),
                                                    pieces.data_ptr(), perm_short.data_ptr(), self.rowptr_short.data_ptr(), counts,
                                                    ws.data_ptr(), ws_bytes, _cabi.stream_ptr()), "hgn_segment_split_build")
        self.n_long, self.n_pieces, self.n_short = int(counts[0]), int(counts[1]), int(counts[2])
        if self.n_long == 0:            # the plan keeps no split
            return
        # only what the counts cover is kept (clones: a slice would keep the bound-sized buffer alive)
        self.long_ids = long_ids[:max(self.n_long, 1)].clone()
        self.piece_ptr = piece_ptr[:self.n_long + 1].clone()
        self.pieces = pieces[:max(3 * self.n_pieces, 1)].clone()
        self.perm_short = perm_short[:max(self.n_short, 1)].clone()
        self.c = _cabi.SegmentSplit(S, E, self.n_long, self.n_pieces, self.n_short, self.long_ids.data_ptr(), self.piece_ptr.data_ptr(),
                                    self.pieces.data_ptr(), self.perm_short.data_ptr(), self.rowptr_short.data_ptr())
        self.nbytes = _tensor_bytes(self.long_ids, self.piece_ptr, self.pieces, self.perm_short, self.rowptr_short)


class SegmentPlan:
    """``ids`` with values in ``[0, num_segments)``.

    ``ids32``  int32 copy (gather index).
    ``perm``   element ids grouped by segment, ascending id inside a segment (stable).
    ``rowptr`` ``rowptr[s]:rowptr[s+1]`` delimits segment ``s`` inside ``perm``.
    ``split``  ``None`` when no segment is long, else the ``SegmentSplit`` the bf16 / width-128 segment calls run on."""

    __slots__ = ("_ids_ref", "_ids_own", "num_segments", "num_elements", "_perm", "_rowptr", "_split", "_cache_key", "ids32", "version",
                 "__weakref__")

    def __init__(self, ids: torch.Tensor, num_segments: int):
        _cabi.require_cuda(ids)
        self.version = ids._version
        # The caller's tensor is referenced weakly (the cache entry of this plan must die with it); a converted copy is ours.
        if ids.dtype == torch.int64 and ids.is_contiguous():
            self._ids_ref, self._ids_own = _weakref.ref(ids), None
        else:
            self._ids_ref, self._ids_own = None, ids.to(torch.int64).contiguous()
        self.num_segments = int(num_segments)
        self.num_elements = ids.numel()
        self.ids32 = ids.to(torch.int32).contiguous() if self.num_elements else torch.zeros(1, dtype=torch.int32, device=ids.device)
        self._perm = None
        self._rowptr = None
        self._split = False          # not built yet
        self._cache_key = None

    @property
    def ids(self) -> torch.Tensor:
        """The int64 index vector (the caller's own tensor while it is alive, else widened from ``ids32``)."""
        if self._ids_own is not None:
            return self._ids_own
        t = self._ids_ref() if self._ids_ref is not None else None
        if t is None or t._version != self.version:
            self._ids_own = self.ids32[:self.num_elements].to(torch.int64)
            return self._ids_own
        return t

    def _build_csr(self) -> None:
        lib = _cabi.load()
        ids = self.ids
        E, dev = self.num_elements, ids.device
        self._perm = torch.empty(max(E, 1), dtype=torch.int32, device=dev)
        self._rowptr = torch.empty(self.num_segments + 1, dtype=torch.int32, device=dev)
        ws_bytes = lib.hgn_csr_workspace_bytes(E, self.num_segments)
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
        with torch.cuda.device(dev):
            _cabi.check(lib.hgn_csr_build(ids.data_ptr(), E, self.num_segments, self._perm.data_ptr(),
                                          self._rowptr.data_ptr(), None, ws.data_ptr(), ws_bytes, _cabi.stream_ptr()),
                        "hgn_csr_build")

    @property
    def perm(self) -> torch.Tensor:
        if self._perm is None:
            self._build_csr()
        return self._perm

    @property
    def rowptr(self) -> torch.Tensor:
        if self._rowptr is None:
            self._build_csr()
        return self._rowptr

    @property
    def split(self) -> "SegmentSplit | None":
        """Built on first use (only the bf16 / width-128 segment bindings ask), so plans that never reach them -- fp32 parity mode, the
        connector and graph builders -- pay nothing for it."""
        if self._split is False:
            if self._rowptr is None:
                self._build_csr()
            E = self.num_elements
            split = SegmentSplit(self._perm, self._rowptr, E, self.num_segments) if E > _cabi.load().hgn_segment_split_threshold() else None
            self._split = split if split is not None and split.n_long > 0 else None
            if self._split is not None and self._cache_key is not None:
                _grow(self._cache_key, self, self._split.nbytes)
        return self._split


# ---- cache -------------------------------------------------------------------------------------------------------------------
# Keyed on the IDENTITY of the index tensor object (id + a weak reference that must still resolve to that very object) and its
# in-place version counter -- never on (data_ptr, numel): two strided views of one buffer share those, and a freed buffer's address
# is recycled.  An entry holds only a weak reference to its source tensor: when the caller drops the tensor (the reference's
# build_graph / _get_batched create fresh index tensors every step) the entry is dead and is swept at the next insertion.  Live
# entries are bounded in BYTES (HGN_PLAN_CACHE_BYTES, default 4 GiB; least recently used first), not in count.
_CACHE_BYTES = int(_os.environ.get("HGN_PLAN_CACHE_BYTES", str(4 << 30)))
_plans: "OrderedDict[tuple, tuple]" = OrderedDict()      # key -> (weakrefs to the source tensors, versions, value, bytes)
_plan_bytes = 0


def _tensor_bytes(*tensors) -> int:
    return sum(t.numel() * t.element_size() for t in tensors if isinstance(t, torch.Tensor))


def _lookup(key, sources):
    hit = _plans.get(key)
    if hit is None:
        return None
    refs, versions, value, _ = hit
    if any(r() is not t for r, t in zip(refs, sources)) or versions != tuple(t._version for t in sources):
        _forget(key)
        return None
    _plans.move_to_end(key)
    return value


def _forget(key) -> None:
    global _plan_bytes
    hit = _plans.pop(key, None)
    if hit is not None:
        _plan_bytes -= hit[3]


def _remember(key, sources, value, nbytes: int) -> None:
    global _plan_bytes
    for k in [k for k, (refs, _, _, _) in _plans.items() if any(r() is None for r in refs)]:     # sources that have died
        _forget(k)
    _forget(key)
    _plans[key] = (tuple(_weakref.ref(t) for t in sources), tuple(t._version for t in sources), value, int(nbytes))
    _plan_bytes += int(nbytes)
    while _plan_bytes > _CACHE_BYTES and len(_plans) > 1:
        _forget(next(iter(_plans)))


def _grow(key, value, nbytes: int) -> None:
    """Adds ``nbytes`` to the live entry ``key`` (when it still holds ``value``): a plan's split is sized when its CSR is built."""
    global _plan_bytes
    hit = _plans.get(key)
    if hit is None or hit[2] is not value:
        return
    _plans[key] = hit[:3] + (hit[3] + int(nbytes),)
    _plan_bytes += int(nbytes)
    while _plan_bytes > _CACHE_BYTES and len(_plans) > 1:
        _forget(next(iter(_plans)))


def plan_cache_stats() -> dict:
    return {"entries": len(_plans), "bytes": _plan_bytes, "limit_bytes": _CACHE_BYTES}


def segment_plan(ids: torch.Tensor, num_segments: int) -> SegmentPlan:
    """Cached plan for a device index tensor (see the cache notes above).  Callers with a dynamic set (``world_edges`` changes every
    step) simply pass each step's fresh tensor: its plan lives exactly as long as the tensor does."""
    key = ("plan", id(ids), int(num_segments))
    hit = _lookup(key, (ids,))
    if hit is not None:
        return hit
    plan = SegmentPlan(ids, num_segments)
    plan._cache_key = key
    # ids (int64, a private copy unless the caller's tensor already was contiguous int64) + ids32 + perm + rowptr
    # ids32 + perm + rowptr (+ a private int64 copy when the caller's tensor was not contiguous int64)
    _remember(key, (ids,), plan, ids.numel() * 8 + (int(num_segments) + 1) * 4 + (ids.numel() * 8 if plan._ids_own is not None else 0))
    return plan


def to_device_index(ids: torch.Tensor, device: torch.device) -> torch.Tensor:
    """Device copy of an index tensor, made once per source tensor object."""
    if ids.device == device:
        return ids
    key = ("h2d", id(ids), str(device))
    hit = _lookup(key, (ids,))
    if hit is not None:
        return hit
    dev_ids = ids.to(device)
    _remember(key, (ids,), dev_ids, _tensor_bytes(dev_ids))
    return dev_ids


class EdgeStorageOrder:
    """Receiver-sorted STORAGE order of one edge set (experimental, ``HGN_EDGE_STORAGE=receiver_sorted``; DESIGN.md s8 round-2 plan).

    The reference's edge order (util.py:60-69: unique (max, min) pairs, then the reversed copies) is half sender-sorted and half
    receiver-sorted.  Keeping the rows stably sorted by receiver INSIDE the processor makes every receiver's edges contiguous: the
    ``Pr[r]`` / ``grad_agg[r]`` row gathers of the edge kernels then touch ~6 distinct rows per warp instruction instead of ~17
    (scripts/analysis_gather_locality.py), and the aggregation becomes a reduction over consecutive rows (the precondition for
    fusing it into the edge kernels' epilogues).  The sort is stable, so within a segment the rows keep their ascending reference
    order: the receiver-side CSR kernels sum them in the same order, so the forward results are bitwise those of the reference
    order (the sender-side sums of the backward see another order: gradients agree to fp32 / bf16 rounding).

    ``perm[k]`` = reference id of the k-th stored row; ``inverse[i]`` = storage position of reference row i.  One instance per
    receivers tensor (cached like the segment plans); ``senders`` / ``receivers`` are the permuted int64 index tensors, created once so
    that their own segment plans stay cached across steps."""

    def __init__(self, senders: torch.Tensor, receivers: torch.Tensor):
        self.perm = torch.argsort(receivers, stable=True)
        self.inverse = torch.empty_like(self.perm)
        self.inverse[self.perm] = torch.arange(self.perm.numel(), device=self.perm.device, dtype=self.perm.dtype)
        self.senders = senders.index_select(0, self.perm).contiguous()
        self.receivers = receivers.index_select(0, self.perm).contiguous()
        self.version = (senders._version, receivers._version)

    def store(self, features: torch.Tensor) -> torch.Tensor:
        """Rows in storage order (differentiable: the backward of a permutation is the gather through its inverse)."""
        return _PermuteRows.apply(features, self._perm32(), self._inverse32())

    def restore(self, features: torch.Tensor) -> torch.Tensor:
        """Rows back in the reference order."""
        return _PermuteRows.apply(features, self._inverse32(), self._perm32())

    def _perm32(self) -> torch.Tensor:
        if getattr(self, "_p32", None) is None:
            self._p32, self._i32 = self.perm.to(torch.int32), self.inverse.to(torch.int32)
        return self._p32

    def _inverse32(self) -> torch.Tensor:
        self._perm32()
        return self._i32


class _PermuteRows(torch.autograd.Function):
    """``x[index]`` for a PERMUTATION ``index`` through the row-gather kernel, forward and backward (``torch.index_select`` would run its
    backward as an atomic ``index_add_``: ~10 x the time on a 6 M x 128 tensor).  CUDA only, like every kernel of the package; the
    host-side test of the bookkeeping installs its own stand-in for ``_permute_rows`` (tests/test_graph_building_cpu.py)."""

    @staticmethod
    def forward(ctx, x, index32, inverse32):
        ctx.inverse32, ctx.index32 = inverse32, index32
        return _permute_rows(x, index32)

    @staticmethod
    def backward(ctx, grad):
        return _permute_rows(grad.contiguous(), ctx.inverse32), None, None


def _permute_rows(x: torch.Tensor, index32: torch.Tensor) -> torch.Tensor:
    from . import _cabi
    _cabi.require_cuda(x, index32)
    x = x.contiguous()
    out = torch.empty_like(x)
    if x.shape[0]:
        with torch.cuda.device(x.device):
            _cabi.check(_cabi.load().hgn_rows_gather(_cabi.dtype_code(x.dtype), x.data_ptr(), index32.data_ptr(), x.shape[0], x.shape[1],
                                                     out.data_ptr(), _cabi.stream_ptr()), "hgn_rows_gather")
    return out


def edge_storage_order(senders: torch.Tensor, receivers: torch.Tensor) -> EdgeStorageOrder:
    """Cached per (senders, receivers) tensor pair, like ``segment_plan``."""
    key = ("order", id(senders), id(receivers))
    hit = _lookup(key, (senders, receivers))
    if hit is not None:
        return hit
    order = EdgeStorageOrder(senders, receivers)
    _remember(key, (senders, receivers), order, _tensor_bytes(order.perm, order.inverse, order.senders, order.receivers))
    return order


def clear_plan_cache() -> None:
    global _plan_bytes
    _plans.clear()
    _plan_bytes = 0
