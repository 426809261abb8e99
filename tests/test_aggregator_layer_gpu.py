"""The fused GraphNet layer with the 'mean', 'max', 'min' and 'pna' aggregators (``ops.graphnet_layer``) and the kernel that routes its
aggregate gradients (``hgn_segment_layer_grad``), on one B200 (``-m gpu``).

* ``hgn_segment_layer_grad`` bit for bit against the numpy restatement of tests/layer_grad_reference.py: segment sizes 0 .. 33,
  ~1e5-element segments, 2^19 + 1 segments, max / min ties (-0 against +0, single-element segments whose one edge wins both), every
  combination of NULL gradient inputs, and the argument refusals.
* The route: a one-block bf16 processor runs every aggregator through the fused layer, the change in ``ops.launch_count`` equals the
  number of ``hgn::`` kernels ``torch.profiler`` records, and both equal the per-layer formula of DESIGN.md (profiled in a process of its
  own, tests/launch_count_worker.py).
* The forward is bit-identical to the old composition ``ops.edge_update`` + ``ops.segment_aggregate`` + ``ops.node_update``.
* Gradients against the bf16 rounding-point emulation of tests/test_gpu_parity.py, globally and over the row windows of a persistent
  grid; two runs bit-identical.
* The partitioned processor at world size 1 equals the processor bit for bit over three steps, for every aggregator; with 2 and 4 GPUs
  (skipped with fewer) the 'pna' peer-memory path against the single-GPU run (tests/partition_aggregator_gpu_worker.py).
* The full cfg5 mesh, 'pna', one layer against the emulation.
"""
import json
import os
import socket
import subprocess
import sys

import numpy as np
import pytest
import torch
import torch.distributed as dist

import layer_grad_reference as lgr
from conftest import rel_err, rel_l2
from hgn_b200 import _cabi, ops, partition, synthetic
from hgn_b200.migration.graphnet import PNA_OPS
from hgn_b200.plan import segment_plan
from hgn_b200.util import EdgeSet
from test_gpu_parity import (_KernelValue, _MLP_NAMES, _bf16_emulated_aggregates, _bf16_emulated_projected_edge,
                             _bf16_emulated_projected_node, _mlp_params, _param_errs, _random_mlp_weights, _report, _row_errs)
from test_layer_schedule_gpu import _processor, _step, _whole
from test_segment_kernels_gpu import NAN, Plan, _assert_bits, _degree_ids, _fan_in_plan, _reduce, _rows, _tied_rows

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
AGGREGATORS = ("sum", "mean", "max", "min", "pna")
TERMS = ("sum", "mean", "max", "min", "base")
HGN_ERR_INVALID_ARGUMENT, HGN_ERR_UNSUPPORTED = -1, -3


def _reducers(aggregator):
    return PNA_OPS if aggregator == "pna" else (aggregator,)


# ------------------------------------------------------------------------------------------------------------------------------------
# hgn_segment_layer_grad
# ------------------------------------------------------------------------------------------------------------------------------------
def _call(plan, grads, args, base, agg, edge, dtype=_cabi.HGN_BF16, D=128, perm=True, rowptr=True):
    return _cabi.load().hgn_segment_layer_grad(
        dtype, plan.E, D, plan.perm.data_ptr() if perm else None, plan.rowptr.data_ptr() if rowptr else None, plan.S,
        *[_cabi.ptr(grads.get(k)) for k in ("sum", "mean", "max", "min")], _cabi.ptr(args.get("max")), _cabi.ptr(args.get("min")),
        _cabi.ptr(base), _cabi.ptr(agg), _cabi.ptr(edge), _cabi.stream_ptr())


def _layer_grad(plan, grads, args, base):
    """The kernel's outputs, NaN-filled before the call (every row must be written); an output is NULL when no term feeds it."""
    want_agg = "sum" in grads or "mean" in grads
    want_edge = "max" in grads or "min" in grads or base is not None
    agg = torch.full((plan.S, 128), NAN, dtype=torch.bfloat16, device="cuda") if want_agg else None
    edge = torch.full((max(plan.E, 1), 128), NAN, dtype=torch.bfloat16, device="cuda")[:plan.E] if want_edge else None
    _cabi.check(_call(plan, grads, args, base, agg, edge), "hgn_segment_layer_grad")
    return agg, edge


def _check_layer_grad(plan, x, terms, rng, tag):
    """Winners from the forward kernel on rows ``x``, random bf16 gradients; the terms in ``terms`` present, the others NULL."""
    _, am = _reduce(x, plan, ("max", "min"), "bf16")
    args = {k: am[k] for k in ("max", "min") if k in terms}
    g = {k: _rows(rng, plan.S, 128, "bf16") for k in ("sum", "mean", "max", "min") if k in terms}
    base = _rows(rng, plan.E, 128, "bf16") if "base" in terms else (None, None)
    agg, edge = _layer_grad(plan, {k: v[0] for k, v in g.items()}, args, base[0])
    want_agg, want_edge = lgr.layer_grad(plan.perm_np, plan.rowptr_np, plan.E, **{f"g_{k}": v[1] for k, v in g.items()},
                                         argmax=am["max"].cpu().numpy(), argmin=am["min"].cpu().numpy(), base=base[1])
    if agg is not None:
        _assert_bits(agg, want_agg, f"{tag} agg_grad {terms}")
    if edge is not None:
        _assert_bits(edge, want_edge, f"{tag} edge_grad {terms}")


_SUBSETS = [tuple(t for i, t in enumerate(TERMS) if m >> i & 1) for m in range(1, 1 << len(TERMS))]


@pytest.mark.parametrize("terms", _SUBSETS, ids=["+".join(t) for t in _SUBSETS])
def test_layer_grad_bit_exact(terms):
    """Every combination of present gradient terms (the others NULL, and an output NULL when no term feeds it), segment sizes 0 .. 33."""
    rng = np.random.default_rng(len(terms) * 31 + sum(map(len, terms)))
    plan = _fan_in_plan(rng)
    x, _ = _rows(rng, plan.E, 128, "bf16")
    _check_layer_grad(plan, x, terms, rng, "fan-in")


def test_layer_grad_ties():
    """Purpose-built max / min ties (first and last position, -0 against +0) and single-element segments, where the one edge wins both
    max and min in every column: the gradient goes to the first winner in perm order only, and both terms land on the single edge."""
    rng = np.random.default_rng(23)
    plan = _fan_in_plan(rng)
    x, _ = _tied_rows(rng, plan, 128, "bf16")
    assert (np.diff(plan.rowptr_np) == 1).any()
    _check_layer_grad(plan, x, TERMS, rng, "ties")
    _check_layer_grad(plan, x, ("max", "min"), rng, "ties")


def test_layer_grad_long_segments_and_grid_scale():
    """A handful of ~1e5-element segments (plus an empty one), then ~2 M elements over 2^19 + 1 segments."""
    rng = np.random.default_rng(29)
    plan = Plan(_degree_ids(rng, [100_000, 0, 99_999, 100_001, 3]), 5)
    x, _ = _rows(rng, plan.E, 128, "bf16")
    _check_layer_grad(plan, x, TERMS, rng, "long")
    S = 2 ** 19 + 1
    plan = Plan(rng.integers(0, S, size=2_000_000), S)
    x, _ = _rows(rng, plan.E, 128, "bf16")
    _check_layer_grad(plan, x, TERMS, rng, "grid scale")
    _check_layer_grad(plan, x, ("mean", "max"), rng, "grid scale")


def test_layer_grad_refusals_and_empty():
    rng = np.random.default_rng(31)
    plan = _fan_in_plan(rng, 1)
    x, _ = _rows(rng, plan.E, 128, "bf16")
    _, am = _reduce(x, plan, ("max", "min"), "bf16")
    g = _rows(rng, plan.S, 128, "bf16")[0]
    base = _rows(rng, plan.E, 128, "bf16")[0]
    agg, edge = torch.empty(plan.S, 128, dtype=torch.bfloat16, device="cuda"), torch.empty(plan.E, 128, dtype=torch.bfloat16, device="cuda")
    args = {"max": am["max"], "min": am["min"]}
    assert _call(plan, {"sum": g}, {}, None, agg, None, dtype=_cabi.HGN_F32) == HGN_ERR_UNSUPPORTED
    refused = {
        "unknown dtype": _call(plan, {"sum": g}, {}, None, agg, None, dtype=7),
        "D = 64": _call(plan, {"sum": g}, {}, None, agg, None, D=64),
        "g_max without argmax": _call(plan, {"max": g}, {}, None, None, edge),
        "g_min without argmin": _call(plan, {"min": g}, {}, None, None, edge),
        "g_sum without agg_grad": _call(plan, {"sum": g}, {}, None, None, edge),
        "g_mean without agg_grad": _call(plan, {"mean": g}, {}, None, None, None),
        "g_max without edge_grad": _call(plan, {"max": g}, args, None, agg, None),
        "base without edge_grad": _call(plan, {"sum": g}, {}, base, agg, None),
        "edge_grad aliasing base": _call(plan, {"max": g}, args, base, None, base),
        "agg_grad aliasing g_sum": _call(plan, {"sum": g}, {}, None, g, None),
        "rowptr NULL": _call(plan, {"sum": g}, {}, None, agg, None, rowptr=False),
        "perm NULL with edge_grad": _call(plan, {"max": g}, args, None, None, edge, perm=False),
    }
    assert all(rc == HGN_ERR_INVALID_ARGUMENT for rc in refused.values()), refused
    # no segments: nothing is written
    empty = Plan(np.zeros(0, dtype=np.int64), 0)
    sentinel = torch.full((4, 128), 3.0, dtype=torch.bfloat16, device="cuda")
    _cabi.check(_call(empty, {"sum": g}, {}, None, sentinel, None), "hgn_segment_layer_grad")
    # no elements: agg_grad is still written for every (empty) segment, inv = 1
    none = Plan(np.zeros(0, dtype=np.int64), 9)
    gs, gs_np = _rows(rng, 9, 128, "bf16")
    agg9, _ = _layer_grad(none, {"mean": gs}, {}, None)
    torch.cuda.synchronize()
    assert (sentinel == 3.0).all()
    _assert_bits(agg9, lgr.layer_grad(none.perm_np, none.rowptr_np, 0, g_mean=gs_np)[0], "E = 0 agg_grad")


# ------------------------------------------------------------------------------------------------------------------------------------
# route and launches
# ------------------------------------------------------------------------------------------------------------------------------------
W, H = 40, 32


@pytest.fixture(scope="module")
def mesh():
    s, r = synthetic.grid_edges_two_way(W, H)
    gen = torch.Generator().manual_seed(3)
    n, e = W * H, s.numel()
    v0, e0, coef = torch.randn(n, 128, generator=gen), torch.randn(e, 128, generator=gen), torch.randn(n, 128, generator=gen)
    return s, r, v0.cuda(), e0.cuda(), coef.cuda()


def launches_per_layer(aggregator):
    """The kernels of one fused layer, fwd + bwd (DESIGN.md section 3.0): projection, edge forward, aggregate, node forward (one table
    projection per two aggregates + the node kernel); node backward (2 + 2 per table + 1 per aggregate), the aggregate-gradient kernel
    (not 'sum'), edge backward (2), paired G0 sums (1), node-level dgrad / wgrad (4)."""
    k = len(_reducers(aggregator))
    t = (k + 1) // 2
    return (3 + t + 1) + (2 + 2 * t + k) + int(aggregator != "sum") + 2 + 1 + 4


@pytest.mark.parametrize("aggregator", AGGREGATORS)
def test_route_and_launch_count(aggregator):
    """One fwd+bwd step of a one-block processor under torch.profiler, in a process of its own (tests/launch_count_worker.py): the change
    in ops.launch_count, the hgn:: kernels the profiler records and the formula agree, and the aggregate gradient is routed by
    segment_layer_grad, never expanded by the segment backward."""
    run = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "launch_count_worker.py"), aggregator],
                         capture_output=True, text=True, timeout=600)
    assert run.returncode == 0, run.stdout[-2000:] + run.stderr[-4000:]
    res = json.loads(run.stdout.strip().splitlines()[-1])
    counted, names = res["counted"], res["kernels"]
    assert counted == len(names) == launches_per_layer(aggregator), (counted, len(names), launches_per_layer(aggregator))
    assert sum("segment_layer_grad" in n for n in names) == int(aggregator != "sum"), names
    assert not any("segment_bwd" in n or "segment_reduce_bwd" in n for n in names), names


# ------------------------------------------------------------------------------------------------------------------------------------
# forward against the old composition
# ------------------------------------------------------------------------------------------------------------------------------------
_SIZES = [(1, 5), (63, 40), (129, 33), ("grid 40x40", 1600), (200000, 40000)]


def _edges(rows, n_nodes, seed):
    if rows == "grid 40x40":
        return tuple(t.cuda() for t in synthetic.grid_edges_two_way(40, 40))
    torch.manual_seed(seed)
    return torch.randint(0, n_nodes, (rows,), device="cuda"), torch.randint(0, n_nodes, (rows,), device="cuda")


@pytest.mark.parametrize("rows,n_nodes", _SIZES)
@pytest.mark.parametrize("aggregator", AGGREGATORS)
def test_forward_equals_composition_bitwise(aggregator, rows, n_nodes):
    """v' and e' of the fused layer equal edge_update + segment_aggregate (or the edge update's own 'sum') + node_update bit for bit,
    with and without gradients required (the winners are recorded only in the first case)."""
    s, r = _edges(rows, n_nodes, 1000 + n_nodes)
    reducers = _reducers(aggregator)
    we, wn = _random_mlp_weights(3, 11), _random_mlp_weights(1 + len(reducers), 13)
    v0 = torch.randn(n_nodes, 128, device="cuda").to(torch.bfloat16)
    e0 = torch.randn(s.numel(), 128, device="cuda").to(torch.bfloat16)
    sp, rp = segment_plan(s, n_nodes), segment_plan(r, n_nodes)
    for grad in (True, False):
        pe, pn = _mlp_params(we), _mlp_params(wn)
        v, e = v0.clone().requires_grad_(grad), e0.clone().requires_grad_(grad)
        with torch.set_grad_enabled(grad):
            fused = ops.graphnet_layer(pe, {}, pn, {}, v, e, sp, rp, aggregator)
            e_new, agg = ops.edge_update(pe, {}, v, e, sp, rp, aggregator == "sum")
            aggs = [agg] if aggregator == "sum" else ops.segment_aggregate(e_new, rp, reducers)
            v_new = ops.node_update(pn, {}, v, aggs)
        assert torch.equal(fused[0], v_new) and torch.equal(fused[1], e_new), (aggregator, rows, grad)


# ------------------------------------------------------------------------------------------------------------------------------------
# gradients against the emulation
# ------------------------------------------------------------------------------------------------------------------------------------
def _layer_vs_emulation(aggregator, s, r, n_nodes, loss, seed, repeat=True):
    """ops.graphnet_layer against the emulated edge update, aggregation (each aggregate rounded as the kernels store it, max / min taken
    on the kernel's own e' so the winners agree) and node update, at the bounds of the fused 'sum' layer's test.  ``loss``: 'both'
    outputs, only 'nodes' (v') or only 'edges' (e').  ``repeat``: run twice and require bit-identical results."""
    torch.manual_seed(seed)
    reducers = _reducers(aggregator)
    rows = s.numel()
    we, wn = _random_mlp_weights(3, 11), _random_mlp_weights(1 + len(reducers), 13)
    v0 = torch.randn(n_nodes, 128, device="cuda").to(torch.bfloat16)
    e0 = torch.randn(rows, 128, device="cuda").to(torch.bfloat16)
    gv = torch.randn(n_nodes, 128, device="cuda").to(torch.bfloat16)
    ge = torch.randn(rows, 128, device="cuda").to(torch.bfloat16)
    sp, rp = segment_plan(s, n_nodes), segment_plan(r, n_nodes)
    pick = {"both": (0, 1), "nodes": (0,), "edges": (1,)}[loss]
    runs = []
    for _ in range(2 if repeat else 1):
        pe, pn = _mlp_params(we), _mlp_params(wn)
        v, e = v0.clone().requires_grad_(True), e0.clone().requires_grad_(True)
        outs = ops.graphnet_layer(pe, {}, pn, {}, v, e, sp, rp, aggregator)
        torch.autograd.backward([outs[i] for i in pick], [(gv, ge)[i] for i in pick])
        runs.append([outs[0].detach(), outs[1].detach(), v.grad, e.grad] + [p.grad for p in pe + pn])
        del outs
    if repeat:
        for i, (a, b) in enumerate(zip(*runs)):
            assert torch.equal(a, b), i
    v_new, e_new, v_grad, e_grad = runs[-1][:4]
    del runs[:-1]
    rd = lambda t: t.to(torch.bfloat16).float()
    wer, wnr = [p.detach().clone().requires_grad_(True) for p in pe], [p.detach().clone().requires_grad_(True) for p in pn]
    vf, ef = v0.float().requires_grad_(True), e0.float().requires_grad_(True)
    e_ref = rd(_bf16_emulated_projected_edge(vf, ef, s, r, wer))
    e_used = _KernelValue.apply(e_ref, e_new)
    v_ref = _bf16_emulated_projected_node(vf, _bf16_emulated_aggregates(e_used, r, n_nodes, reducers), wnr)
    torch.autograd.backward([(v_ref, e_used)[i] for i in pick], [(gv.float(), ge.float())[i] for i in pick])
    checks = {"v'": (*_row_errs(v_new.float(), v_ref.detach(), rel_err), 1e-2), "e'": (*_row_errs(e_new.float(), e_ref.detach(), rel_err), 1e-2),
              "grad e": (*_row_errs(e_grad.float(), ef.grad, rel_l2), 1e-2), "grad v": (*_row_errs(v_grad.float(), vf.grad, rel_l2), 1.5e-2)}
    err, name = _param_errs(pe + pn, wer + wnr, [f"edge {n}" for n in _MLP_NAMES] + [f"node {n}" for n in _MLP_NAMES])
    checks[f"weights (worst {name})"] = (err, 0.0, 1.5e-2)
    _report(f"{aggregator} layer, {rows} edges / {n_nodes} nodes, loss on {loss}", checks)


_GRAD_CASES = [(a, rows, n, "both") for a in AGGREGATORS[1:] for rows, n in _SIZES]
_GRAD_CASES += [(a, "grid 40x40", 1600, loss) for a in AGGREGATORS[1:] for loss in ("nodes", "edges")]


@pytest.mark.parametrize("aggregator,rows,n_nodes,loss", _GRAD_CASES)
def test_layer_vs_bf16_emulation(aggregator, rows, n_nodes, loss):
    seed = (1600 if rows == "grid 40x40" else rows) + 10 * AGGREGATORS.index(aggregator) + ["both", "nodes", "edges"].index(loss)
    s, r = _edges(rows, n_nodes, seed)
    _layer_vs_emulation(aggregator, s, r, n_nodes, loss, seed)


def test_cfg5_full_mesh_pna_layer_vs_bf16_emulation():
    """The 'pna' layer on the full cfg5 mesh (1 000 000 nodes, 5 992 002 edges), both outputs in the loss; prints the peak device
    memory of the test."""
    s, r = (t.cuda() for t in synthetic.grid_edges_two_way(1000, 1000))
    torch.cuda.empty_cache()
    torch.cuda.reset_peak_memory_stats()
    _layer_vs_emulation("pna", s, r, 1_000_000, "both", seed=9, repeat=False)
    print(f"cfg5 pna layer vs emulation: peak device memory {torch.cuda.max_memory_allocated() / 2 ** 30:.1f} GiB")
    torch.cuda.empty_cache()


# ------------------------------------------------------------------------------------------------------------------------------------
# partitioned processor
# ------------------------------------------------------------------------------------------------------------------------------------
LAYERS = 3


@pytest.mark.parametrize("aggregator", AGGREGATORS[1:])
def test_world1_partitioned_equals_processor_bitwise(aggregator, mesh, tmp_path):
    """World size 1 (gloo; a PeerHalo without peers): the peer fast path runs the fused layer of every aggregator, and over three steps
    (both table parities) its outputs, input gradients and parameter gradients equal the processor's on the whole graph bit for bit."""
    s, r, v0, e0, coef = mesh
    dist.init_process_group("gloo", store=dist.FileStore(str(tmp_path / "store"), 1), rank=0, world_size=1)
    try:
        dev = torch.device("cuda", torch.cuda.current_device())
        lg = partition.build_local_graph(s, r, partition.block_partition(W * H, 1), 0, 1)
        peer = partition.PeerHalo(lg, LAYERS, dev)
        try:
            proc = _processor(aggregator, LAYERS)
            model = partition.PartitionedProcessor(proc, partition.HaloPlan(lg, dev), peer)
            s_loc, r_loc = lg.senders.to(dev), lg.receivers.to(dev)
            assert model._fast_path(v0.to(torch.bfloat16), [EdgeSet("mesh_edges", e0.to(torch.bfloat16), s_loc, r_loc)])

            def run_split(v, e):
                out_v, out_sets = model(v, [EdgeSet("mesh_edges", e, s_loc, r_loc)])
                return out_v, out_sets[0].features
            run_whole, params = _whole(proc, s, r), list(proc.parameters())
            for step in range(3):
                whole = _step(run_whole, params, v0, e0, coef, 0.01 * step)
                parted = _step(run_split, params, v0, e0, coef, 0.01 * step)
                for i, (a, b) in enumerate(zip(parted, whole)):
                    assert torch.equal(a, b), (step, i)
        finally:
            peer.close()
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world", [2, 4])
def test_partitioned_pna_peer_path_matches_single_gpu(world):
    if torch.cuda.device_count() < world:
        pytest.skip(f"needs {world} GPUs, {torch.cuda.device_count()} visible")
    with socket.socket() as sock:
        sock.bind(("127.0.0.1", 0))
        port = sock.getsockname()[1]
    run = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}", "--master-addr", "127.0.0.1",
                          "--master-port", str(port), os.path.join(ROOT, "tests", "partition_aggregator_gpu_worker.py"), "pna"],
                         capture_output=True, text=True, timeout=900)
    assert run.returncode == 0 and run.stdout.count("PARTITION-AGG-GPU-OK") == world, run.stdout[-3000:] + run.stderr[-5000:]
    print("\n" + "\n".join(ln for ln in run.stdout.splitlines() if "PARTITION-AGG-GPU-OK" in ln))
