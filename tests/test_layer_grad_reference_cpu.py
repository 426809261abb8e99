"""The numpy restatement of ``hgn_segment_layer_grad`` (tests/layer_grad_reference.py) against torch on the CPU.

* Bit for bit against the same formula written with torch fp32 operations and torch's own bf16 rounding, for every combination of
  present gradient terms, ties of -0 against +0 included.
* Against the meaning of the two outputs: ``agg_grad[receivers] + edge_grad`` is the autograd gradient (fp64) of
  ``<g_sum, segment_sum(x)> + <g_mean, segment_mean(x)> + <g_max, segment_max(x)> + <g_min, segment_min(x)> + <base, x>``
  up to the two bf16 roundings.
"""
import itertools

import numpy as np
import pytest
import torch

import segment_reference as sr
from layer_grad_reference import layer_grad

TERMS = ("sum", "mean", "max", "min", "base")


def _case(seed, ties=False):
    """Segments of every size 0 .. 33 in random order, elements in random order; bf16-valued fp32 gradients and winners."""
    rng = np.random.default_rng(seed)
    degrees = np.tile(np.arange(34), 2)
    rng.shuffle(degrees)
    ids = np.repeat(np.arange(len(degrees)), degrees)
    rng.shuffle(ids)
    S, E, D = len(degrees), len(ids), 16
    perm, rowptr = sr.csr(ids, S)
    bf = lambda a: sr.round_bf16(a.astype(np.float32))
    if ties:
        x = rng.choice(np.array([-1.0, -0.0, 0.0, 1.0], dtype=np.float32), size=(E, D))
    else:
        x = bf(rng.standard_normal((E, D)))
    _, argmax = sr.segment_argext(x, perm, rowptr, True)
    _, argmin = sr.segment_argext(x, perm, rowptr, False)
    g = {k: bf(rng.standard_normal((S, D))) for k in ("sum", "mean", "max", "min")}
    if ties:                                        # signed zeros in the gradients: 0 + -0 = +0 must come out of both sides
        for k in g:
            g[k][:, ::3] = rng.choice(np.array([-0.0, 0.0], dtype=np.float32), size=g[k][:, ::3].shape)
    g["base"] = bf(rng.standard_normal((E, D)))
    g["base"][::5, ::2] = -0.0
    return ids, perm, rowptr, x, argmax, argmin, g


def _torch_formula(ids, rowptr, argmax, argmin, g, present):
    t = {k: torch.from_numpy(v) for k, v in g.items()}
    S, E, D = len(rowptr) - 1, len(ids), g["base"].shape[1]
    r = torch.from_numpy(ids)
    agg = torch.zeros(S, D)
    if "sum" in present:
        agg = agg + t["sum"]
    if "mean" in present:
        inv = 1.0 / torch.from_numpy(np.diff(rowptr)).clamp(min=1).float()
        agg = agg + t["mean"] * inv.view(-1, 1)
    edge = torch.zeros(E, D)
    if "base" in present:
        edge = edge + t["base"]
    e = torch.arange(E).view(-1, 1)
    for op, arg in (("max", argmax), ("min", argmin)):
        if op in present:
            edge = torch.where(torch.from_numpy(arg)[r] == e, edge + t[op][r], edge)
    return agg.to(torch.bfloat16).float().numpy(), edge.to(torch.bfloat16).float().numpy()


def _kwargs(g, argmax, argmin, present):
    kw = {f"g_{k}": g[k] for k in ("sum", "mean", "max", "min") if k in present}
    kw.update(argmax=argmax, argmin=argmin, base=g["base"] if "base" in present else None)
    return kw


@pytest.mark.parametrize("ties", [False, True])
def test_restatement_matches_torch_bitwise(ties):
    ids, perm, rowptr, _, argmax, argmin, g = _case(3 + ties, ties)
    for n in range(1, len(TERMS) + 1):
        for present in itertools.combinations(TERMS, n):
            agg, edge = layer_grad(perm, rowptr, len(ids), **_kwargs(g, argmax, argmin, present))
            t_agg, t_edge = _torch_formula(ids, rowptr, argmax, argmin, g, present)
            assert np.array_equal(agg.view(np.uint32), t_agg.view(np.uint32)), present
            assert np.array_equal(edge.view(np.uint32), t_edge.view(np.uint32)), present


def test_restatement_is_the_aggregate_gradient():
    ids, perm, rowptr, x, argmax, argmin, g = _case(11)
    S, E, D = len(rowptr) - 1, len(ids), x.shape[1]
    r = torch.from_numpy(ids)
    xt = torch.from_numpy(x).double().requires_grad_(True)
    total = torch.zeros(S, D, dtype=torch.float64).index_add(0, r, xt)
    count = torch.bincount(r, minlength=S).clamp(min=1).double().view(-1, 1)
    # max / min as gathers of the winners (the values have no ties here): their gradient goes to the winning element only
    pick = lambda arg: torch.cat([xt, xt.new_zeros(1, D)]).gather(0, torch.from_numpy(np.where(arg < 0, E, arg)))
    gd = {k: torch.from_numpy(v).double() for k, v in g.items()}
    loss = ((total * gd["sum"]).sum() + (total / count * gd["mean"]).sum() + (pick(argmax) * gd["max"]).sum()
            + (pick(argmin) * gd["min"]).sum() + (xt * gd["base"]).sum())
    loss.backward()
    agg, edge = layer_grad(perm, rowptr, E, **_kwargs(g, argmax, argmin, TERMS))
    got = agg[ids].astype(np.float64) + edge
    want = xt.grad.numpy()
    assert np.allclose(got, want, rtol=2 ** -7, atol=2 ** -7 * np.abs(want).max()), np.abs(got - want).max()
