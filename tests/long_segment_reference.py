"""Numpy restatement of the long-segment split (csrc/segment_long.cu, include/hgn_b200.h), on segment_reference.py's conventions.

A segment of more than ``T`` elements is long; it is cut into pieces of ``P`` consecutive positions of ``perm`` (the last piece may be
shorter).  For a long segment:

- piece partial ``p_k`` = fp32 sum from +0.0 of the piece's rows in ``perm`` order;
- ``total = (((0 + p_0) + p_1) + ...)`` in ascending ``k``;
- sum = ``total`` (``total + prior`` with an accumulated output), rounded once; mean = ``total * fp32(1 / count)``, rounded once;
- max / min and their winners: piece winners (first in order) combined in ascending piece order with strict comparisons, which is the
  sequential first-in-order result of ``segment_reference.segment_argext``.

Short segments keep ``segment_reference``'s sequential order.  ``T`` and ``P`` are arguments, so that the CPU tests can also check
degenerate layouts (one piece per long segment); the GPU tests pass the library's values.
"""
import numpy as np

import segment_reference as sr

F32 = np.float32


def split(perm, rowptr, T, P):
    """The split bookkeeping: dict of long_ids, piece_ptr [n_long + 1], pieces [n_pieces, 3] (segment, begin, end), perm_short,
    rowptr_short (all int64)."""
    perm, rowptr = np.asarray(perm, dtype=np.int64), np.asarray(rowptr, dtype=np.int64)
    counts = np.diff(rowptr)
    long_ids = np.flatnonzero(counts > T).astype(np.int64)
    pieces = [(s, b, min(b + P, rowptr[s + 1])) for s in long_ids for b in range(int(rowptr[s]), int(rowptr[s + 1]), P)]
    pieces = np.asarray(pieces, dtype=np.int64).reshape(-1, 3)
    n_per = (counts[long_ids] + P - 1) // P
    piece_ptr = np.concatenate([[0], np.cumsum(n_per)]).astype(np.int64)
    short_counts = np.where(counts > T, 0, counts)
    rowptr_short = np.concatenate([[0], np.cumsum(short_counts)]).astype(np.int64)
    keep = np.repeat(counts <= T, counts)                   # per perm position: does it belong to a short segment
    return dict(long_ids=long_ids, piece_ptr=piece_ptr, pieces=pieces, perm_short=perm[keep] if len(perm) else perm[:0],
                rowptr_short=rowptr_short)


def _piece_csr(perm, sp):
    """(perm, rowptr) whose segments are the pieces."""
    pieces = sp["pieces"]
    if len(pieces) == 0:
        return np.zeros(0, dtype=np.int64), np.zeros(1, dtype=np.int64)
    idx = np.concatenate([np.arange(b, e) for _, b, e in pieces])
    return np.asarray(perm, dtype=np.int64)[idx], np.concatenate([[0], np.cumsum(pieces[:, 2] - pieces[:, 1])])


def long_totals(x, perm, sp):
    """fp32 ``total`` of every long segment, [n_long, ...]."""
    x = np.asarray(x, dtype=F32)
    pperm, prow = _piece_csr(perm, sp)
    partials = sr.sequential_sum(x, pperm, prow)
    return sr.sequential_sum(partials, np.arange(len(partials), dtype=np.int64), sp["piece_ptr"])


def _sums(x, perm, rowptr, T, P):
    """fp32 segment sums: the short segments in sequential order (over the short CSR, where every long segment is empty), the long
    ones piece by piece."""
    sp = split(perm, rowptr, T, P)
    s = sr.sequential_sum(x, sp["perm_short"], sp["rowptr_short"])
    s[sp["long_ids"]] = long_totals(x, perm, sp)
    return s


def segment_sum(x, perm, rowptr, T, P, prior=None, out_dtype="float32"):
    s = _sums(x, perm, rowptr, T, P)
    if prior is not None:
        s = s + np.asarray(prior, dtype=F32)
    return sr._out(s, out_dtype)


def segment_mean(x, perm, rowptr, T, P, out_dtype="float32"):
    s = _sums(x, perm, rowptr, T, P)
    return sr._out(sr._scale_by_count(s, np.diff(rowptr), True), out_dtype)


def segment_argext(x, perm, rowptr, T, P, largest):
    """(value, arg) with the long segments' winners combined piece by piece: per piece the first-in-order winner, then across the
    segment's pieces in ascending order with a strict comparison."""
    x = np.asarray(x, dtype=F32)
    value, arg = sr.segment_argext(x, perm, rowptr, largest)
    sp = split(perm, rowptr, T, P)
    if len(sp["long_ids"]) == 0:
        return value, arg
    pperm, prow = _piece_csr(perm, sp)
    pv, pa = sr.segment_argext(x, pperm, prow, largest)
    better = np.greater if largest else np.less
    for i, s in enumerate(sp["long_ids"]):
        v = np.full(x.shape[1:], -np.inf if largest else np.inf, dtype=F32)
        a = np.full(x.shape[1:], -1, dtype=np.int64)
        for k in range(sp["piece_ptr"][i], sp["piece_ptr"][i + 1]):
            win = better(pv[k], v)
            v, a = np.where(win, pv[k], v), np.where(win, pa[k], a)
        value[s], arg[s] = v, a
    return value, arg
