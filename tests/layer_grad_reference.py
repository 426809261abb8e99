"""Order-exact numpy restatement of ``hgn_segment_layer_grad`` (csrc/segment.cu): the incoming gradient of e' in a fused GraphNet
layer with a 'mean' / 'max' / 'min' / 'pna' aggregator.

    agg_grad[r]  = 0 + g_sum[r] + g_mean[r] * fp32(1 / max(cnt_r, 1))                       one row per segment
    edge_grad[e] = 0 + base[e] + [argmax[r_e] == e] g_max[r_e] + [argmin[r_e] == e] g_min[r_e]

one numpy fp32 operation at a time, absent terms skipped, the product rounded before it is added (numpy never fuses a multiply and an
add), each output rounded to bf16 once.  Inputs are fp32 arrays holding bf16 values; outputs are bf16 values widened to fp32.
"""
import numpy as np

from segment_reference import F32, round_bf16


def layer_grad(perm, rowptr, num_elements, g_sum=None, g_mean=None, g_max=None, g_min=None, argmax=None, argmin=None, base=None):
    """(agg_grad [S, D], edge_grad [E, D]) over the CSR grouping (perm, rowptr) of ``num_elements`` elements."""
    perm, rowptr = np.asarray(perm, dtype=np.int64), np.asarray(rowptr, dtype=np.int64)
    counts = np.diff(rowptr)
    S, E = len(counts), int(num_elements)
    D = next(np.asarray(g).shape[1] for g in (g_sum, g_mean, g_max, g_min, base) if g is not None)
    agg = np.zeros((S, D), dtype=F32)
    if g_sum is not None:
        agg = agg + np.asarray(g_sum, dtype=F32)
    if g_mean is not None:
        inv = (F32(1) / np.maximum(counts, 1).astype(F32)).reshape(-1, 1)
        agg = agg + np.asarray(g_mean, dtype=F32) * inv
    ids = np.empty(E, dtype=np.int64)
    ids[perm] = np.repeat(np.arange(S), counts)
    edge = np.zeros((E, D), dtype=F32)
    if base is not None:
        edge = edge + np.asarray(base, dtype=F32)
    e = np.arange(E, dtype=np.int64).reshape(-1, 1)
    for gx, ax in ((g_max, argmax), (g_min, argmin)):
        if gx is not None:
            edge = np.where(np.asarray(ax)[ids] == e, edge + np.asarray(gx, dtype=F32)[ids], edge)
    return round_bf16(agg), round_bf16(edge)
