"""Order-exact numpy reference of the segment kernels (csrc/segment.cu).

The kernels do only fp32 additions, one multiplication or division for 'mean', comparisons and copies, in an order the header
documents, and the library is built without fast-math.  This module does the same operations in the same order, one numpy fp32
operation at a time, so that its results can be compared with the kernels' bit for bit:

- sum: start from +0.0 and add the segment's rows in ascending position of ``perm`` (= ascending element id); with an accumulated
  output the prior value is added *after* the segment sum (``s + prior``).  The result is rounded to the output dtype once.
- mean: the fp32 segment sum, then ``s * fp32(1 / max(count, 1))`` (the vector kernels) or ``s / max(count, 1)`` (the scalar
  kernels, ``reciprocal=False``).
- max / min: the winner is the first element in ``perm`` order whose value equals the segment's extreme, and the output is the
  winner's own value (so the sign of a +-0 winner is kept).  An empty segment gives +0.0 and arg -1.
- multi-source sum: ``base`` first, then sources 0 .. k-1, each in its own ``perm`` order.
- backward: ``0 + g_sum + g_mean / count + [arg == e] g_max + [arg == e] g_min (+ prior)``, terms in that order.

Inputs are fp32 numpy arrays (bf16 tensors widened exactly); ``out_dtype='bfloat16'`` rounds the result to the nearest bf16 value,
ties to even, and returns it widened to fp32 again.  Non-finite inputs (NaN, +-inf) are outside what this module restates.
"""
import numpy as np

F32 = np.float32


def round_bf16(x):
    """fp32 -> nearest bf16 (ties to even), returned as fp32.  Finite inputs; values that round past the largest bf16 give inf."""
    u = np.ascontiguousarray(x, dtype=F32).view(np.uint32)
    u = (u + (((u >> 16) & 1) + 0x7FFF).astype(np.uint32)) & np.uint32(0xFFFF0000)
    return u.view(F32)


def _out(x, out_dtype):
    return round_bf16(x) if out_dtype == "bfloat16" else x.astype(F32, copy=False)


def csr(ids, num_segments):
    """(perm, rowptr) of the plan: element ids grouped by segment, ascending inside a segment (int64)."""
    ids = np.asarray(ids, dtype=np.int64)
    perm = np.argsort(ids, kind="stable").astype(np.int64)
    rowptr = np.zeros(num_segments + 1, dtype=np.int64)
    np.cumsum(np.bincount(ids, minlength=num_segments), out=rowptr[1:])
    return perm, rowptr


def sequential_sum(x, perm, rowptr, acc=None):
    """fp32 ``acc[s] + x[perm[rowptr[s]]] + x[perm[rowptr[s] + 1]] + ...``, one rounding per addition (acc defaults to +0.0).

    Vectorised over segments: step p adds the p-th element of every segment that has more than p elements."""
    x = np.asarray(x, dtype=F32)
    S = len(rowptr) - 1
    acc = np.zeros((S,) + x.shape[1:], dtype=F32) if acc is None else np.array(acc, dtype=F32)
    counts = np.diff(rowptr)
    order = np.argsort(-counts, kind="stable")             # segments by decreasing size: the live ones at step p are a prefix
    neg_sorted = -counts[order]
    beg = rowptr[:-1][order]
    for p in range(int(counts.max()) if S else 0):
        n = int(np.searchsorted(neg_sorted, -p, side="left"))   # segments with more than p elements
        segs = order[:n]
        acc[segs] = acc[segs] + x[perm[beg[:n] + p]]
    return acc


def segment_sum(x, perm, rowptr, prior=None, out_dtype="float32"):
    s = sequential_sum(x, perm, rowptr)
    if prior is not None:
        s = s + np.asarray(prior, dtype=F32)
    return _out(s, out_dtype)


def _scale_by_count(v, counts, reciprocal):
    c = np.maximum(counts, 1).astype(F32).reshape((-1,) + (1,) * (v.ndim - 1))
    return v * (F32(1) / c) if reciprocal else v / c


def segment_mean(x, perm, rowptr, reciprocal=True, out_dtype="float32"):
    return _out(_scale_by_count(sequential_sum(x, perm, rowptr), np.diff(rowptr), reciprocal), out_dtype)


def segment_argext(x, perm, rowptr, largest):
    """(value, arg) of max (``largest``) or min per segment and column: the first element in ``perm`` order equal to the extreme."""
    x = np.asarray(x, dtype=F32)
    S, E = len(rowptr) - 1, len(perm)
    value = np.zeros((S,) + x.shape[1:], dtype=F32)
    arg = np.full((S,) + x.shape[1:], -1, dtype=np.int64)
    counts = np.diff(rowptr)
    live = np.flatnonzero(counts)
    if E == 0 or live.size == 0:
        return value, arg
    starts = rowptr[:-1][live]
    xs = x[perm]                                            # perm order: every segment is one contiguous run
    ext = (np.maximum if largest else np.minimum).reduceat(xs, starts, axis=0)
    seg_of = np.repeat(np.arange(S), counts)
    pos = np.arange(E, dtype=np.int64).reshape((E,) + (1,) * (x.ndim - 1))
    full = np.zeros((S,) + x.shape[1:], dtype=F32)
    full[live] = ext
    cand = np.where(xs == full[seg_of], pos, E)             # == : -0.0 and +0.0 tie
    first = np.minimum.reduceat(cand, starts, axis=0)
    arg[live] = perm[first]
    value[live] = np.take_along_axis(xs, first, axis=0)
    return value, arg


def multi_segment_sum(sources, base=None, shape=None, out_dtype="float32"):
    """``sources``: [(x_k, perm_k, rowptr_k)], at most the kernel's four; ``base`` [S, D], or None for zeros of ``shape``."""
    acc = np.zeros(shape, dtype=F32) if base is None else np.asarray(base, dtype=F32)
    for x, perm, rowptr in sources:
        acc = sequential_sum(x, perm, rowptr, acc)
    return _out(acc, out_dtype)


def segment_backward(ids, rowptr, g_sum=None, g_mean=None, g_max=None, g_min=None, argmax=None, argmin=None, prior=None,
                     reciprocal=True, contract_mean=False, out_dtype="float32"):
    """grad[e] = 0 + g_sum[r] + g_mean[r] / count_r + [argmax[r] == e] g_max[r] + [argmin[r] == e] g_min[r] (+ prior[e]), r = ids[e].

    ``contract_mean``: ``(0 + g_sum) + g_mean * fp32(1 / count)`` as one fused multiply-add, rounded once, which the compiler may
    make of the vector kernels' expression (emulated in fp64, where the product is exact)."""
    ids = np.asarray(ids, dtype=np.int64)
    E = len(ids)
    some = next(g for g in (g_sum, g_mean, g_max, g_min, prior) if g is not None)
    tail = np.asarray(some).shape[1:]
    g = np.zeros((E,) + tail, dtype=F32)
    e = np.arange(E, dtype=np.int64).reshape((E,) + (1,) * len(tail))
    if g_sum is not None:
        g = g + np.asarray(g_sum, dtype=F32)[ids]
    if g_mean is not None:
        gm = np.asarray(g_mean, dtype=F32)[ids]
        if contract_mean:
            inv = F32(1) / np.maximum(np.diff(rowptr)[ids], 1).astype(F32).reshape((-1,) + (1,) * len(tail))
            g = (g.astype(np.float64) + gm.astype(np.float64) * inv.astype(np.float64)).astype(F32)
        else:
            g = g + _scale_by_count(gm, np.diff(rowptr)[ids], reciprocal)
    for gx, ax in ((g_max, argmax), (g_min, argmin)):
        if gx is not None:
            g = np.where(np.asarray(ax)[ids] == e, g + np.asarray(gx, dtype=F32)[ids], g)
    if prior is not None:
        g = g + np.asarray(prior, dtype=F32)
    return _out(g, out_dtype)
