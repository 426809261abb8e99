"""Parity above one tile and at the benchmarked sizes (``-m gpu``), plus the empty-edge-set edge case.

* empty ``world_edges`` (deforming_plate frames without contact, plate.py:86-110 -> E = 0) through GraphNet / HyperGraphNet /
  HeteroGraphNet, forward and backward, both precision modes: equals the oracle, the set's weight gradients are exactly zero;
* 15 message-passing layers forward + backward at the flag_simple shape (BASELINE.json configs[1]) against the oracle;
* a 1000 x 125 slab (125 000 nodes / 745 752 edges, 5 826 tiles = 39 per CTA), 2 layers forward + backward against the oracle;
* the FULL cfg5 mesh (1 000 000 nodes / 5 992 002 edges, 317 tiles per CTA), one layer: sampled edge rows, the aggregation of
  sampled receivers and sampled node rows against the oracle's arithmetic on exactly those rows; the bf16 (tcgen05) and fp32
  (FFMA) backward passes against each other; run-to-run bit identity.
Tolerances: fp32 1e-5 / bf16 2e-2 on forward quantities (max metric); gradients: relative L2 in bf16, and in fp32 above ~10^5 rows x
layers (the max metric below that), with the bound = the measured figure x 2 (printed by the tests; see GRAD_L2).
"""
import numpy as np
import pytest
import torch

import hgn_oracle as orc
from conftest import GoldenCase, rel_err, rel_l2
from hgn_b200 import synthetic
from hgn_b200 import util as hutil
from hgn_b200.migration.meshgraphnet import MeshGraphNet

pytestmark = pytest.mark.gpu

TOL = {"fp32": 1e-5, "bf16": 2e-2}
GRAD_MAX_FP32 = 1e-4            # max metric, small graphs (a few thousand rows)
# Above ~10^5 rows x layers gradients are compared in relative L2, in BOTH modes: the forward latents of two correct fp32
# implementations agree to ~1e-6, so of the ~10^8 hidden units a few hundred have a pre-activation closer to zero than that and
# their ReLU takes the other branch -- isolated rows then differ by O(10 %), which the max metric reports as 1e-2 .. 5e-2 (measured:
# slab 1.8e-2 / 2.5e-2, 15 layers 2.7e-2 / 4.8e-2) while the L2 metric stays at the share of affected rows.  With 'pna' the same
# happens to max / min winners (tests/test_gpu_parity.py: fp32_grad_check).  Bounds = the figures measured on the B200 (printed by
# the tests; profiles/r2_scale_parity.txt) x 2:
#   fp32: slab 2 layers 1.84e-4 / 3.09e-4 / 3.33e-4 (v, e, worst weight), 15 layers 1.45e-3 / 1.53e-3 / 3.52e-3 (one B200, 1000 W power
#   limit; the fp32 kernels themselves are held to 5e-5 in the max metric against float64 up to 1.5 M rows by tests/test_mlp_f32_gpu.py);
#   bf16 (vs the fp32 oracle): slab 5.2e-2 / 8.8e-2 / 9.5e-2 (v, e, worst weight),
#   15 layers 1.24e-1 / 1.41e-1 / 1.79e-1, cfg5 one layer (vs our fp32 kernels) 4.2e-2 / 8.3e-2 / 1.0e-1.
# The bf16 kernels themselves are pinned much tighter (1.5e-2) against an emulation with the same rounding points, at the full
# cfg5 size too (test_cfg5_full_mesh_edge_kernels_vs_bf16_emulation).
GRAD_L2 = {"fp32": {"slab": 6.7e-4, "deep": 7.1e-3}, "bf16": {"slab": 0.18, "deep": 0.36, "cfg5": 0.2, "small": 0.3}}


def _processor(arch, aggregator, layers, edge_sets, weights, precision):
    shell = MeshGraphNet(3, 128, 2, aggregator, layers, arch, edge_sets)
    proc = shell.processor
    if weights is not None:
        proc.load_state_dict({k[len("processor."):]: t for k, t in weights.items()})
    proc = proc.cuda()
    proc.precision = precision
    return proc


def _weight_grad_checks(proc, wo, precision, tag):
    worst = 0.0
    for key, p in proc.named_parameters():
        ref = wo["processor." + key].grad
        if ref is None:
            assert p.grad is None or float(p.grad.abs().max()) == 0.0, key
            continue
        assert p.grad is not None, key
        if float(ref.norm()) == 0.0:
            assert float(p.grad.abs().max()) == 0.0, f"{tag}: {key} should have an exactly-zero gradient"
            continue
        err = rel_l2(p.grad, ref)
        worst = max(worst, err)
    return worst


# ------------------------------------------------------------------------------------------------------------------
# empty edge set
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("arch", ["none", "hyper", "hetero"])
def test_empty_world_edges_forward_backward(arch, precision):
    case = GoldenCase("mgn_pna_L1" if arch == "none" else "hgn_hyper_pna_L1")
    g = case.graph(orc.MultiGraph, orc.EdgeSet)
    n_rows = [int(x.shape[0]) for x in g.node_features]
    names = [es.name for es in g.edge_sets] + ["world_edges"]
    index_sets = [(es.name, es.senders, es.receivers) for es in g.edge_sets]
    index_sets.append(("world_edges", torch.zeros(0, dtype=torch.int64), torch.zeros(0, dtype=torch.int64)))
    proc = _processor(arch, "pna", 1, names, None, precision)
    v_cpu = [synthetic.seeded_tensor(f"ev{i}", (n, 128), 3) for i, n in enumerate(n_rows)]
    e_cpu = {nm: synthetic.seeded_tensor(f"ee{nm}", (s.numel(), 128), 3) for nm, s, _ in index_sets}

    def graph(mod, dev, grad):
        nodes = [t.clone().to(dev).requires_grad_(grad) for t in v_cpu]
        sets = [mod.EdgeSet(nm, e_cpu[nm].clone().to(dev).requires_grad_(grad), s, r) for nm, s, r in index_sets]
        return mod.MultiGraph(nodes, sets)

    with torch.no_grad():                       # materialises the lazy linears -- with E = 0 for world_edges
        proc(graph(hutil, "cuda", False))
    shapes = {"processor." + k: tuple(v.shape) for k, v in proc.state_dict().items()}
    w = synthetic.seeded_state_dict(shapes, 31)
    proc.load_state_dict({k[len("processor."):]: t for k, t in w.items()})
    wo = {k: t.clone().requires_grad_(True) for k, t in w.items()}
    go = graph(orc, "cpu", True)
    # the reference iterates {'mesh_edges', 'world_edges'}.intersection(...) -- a set, hash-seed dependent (hypergraphnet.py:31,44); the
    # oracle takes the order this process produces, which is the one hgn_b200's blocks see too
    # -- evaluated like the reference does, against the block's ModuleDict keys: set.intersection(<keys view>) inserts in key order,
    # set.intersection(<set>) in the smaller set's own order, and the two differ when the two names share a hash slot (1 process in ~16)
    block_keys = proc.graphnet_blocks[0].edge_models.keys()
    set_order = {"mesh": list({"mesh_edges", "world_edges"}.intersection(block_keys)),
                 "inter": list({"inter_cluster", "inter_cluster_world"}.intersection(block_keys))}
    ref = orc.processor(wo, "pna", arch, go, set_order=set_order)
    coefs = [synthetic.seeded_tensor(f"ec{i}", t.shape, 4) for i, t in enumerate(ref.node_features)]
    sum((t * c).sum() for t, c in zip(ref.node_features, coefs)).backward()

    gg = graph(hutil, "cuda", True)
    leaves = list(gg.node_features)             # the blocks replace the list's entries in place (graphnet.py:48)
    out = proc(gg)
    sum((t * c.cuda()).sum() for t, c in zip(out.node_features, coefs)).backward()
    for i, (a, b) in enumerate(zip(out.node_features, ref.node_features)):
        assert rel_err(a, b) < TOL[precision], f"node latents {i}"
    world = next(es for es in out.edge_sets if es.name == "world_edges")
    assert world.features.shape == (0, 128)
    for a, b in zip(leaves, go.node_features):
        err = rel_err(a.grad, b.grad) if precision == "fp32" else rel_l2(a.grad, b.grad)
        assert err < (GRAD_MAX_FP32 if precision == "fp32" else GRAD_L2["bf16"]["small"]), err
    zero_keys = [k for k, p in proc.named_parameters() if ".edge_models.world_edges." in k]
    assert zero_keys
    for k, p in proc.named_parameters():
        if k in zero_keys:                      # the reference's autograd gives exact zeros for an MLP that saw no rows
            assert p.grad is not None and float(p.grad.abs().max()) == 0.0, k
    _weight_grad_checks(proc, wo, precision, f"empty world edges {arch}")


# ------------------------------------------------------------------------------------------------------------------
# depth: 15 layers forward + backward at the flag_simple shape
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_processor_15_layers_forward_backward_flag_shape(precision):
    s, r = synthetic.grid_edges_two_way(40, 40)
    n, E, L = 1600, s.numel(), 15
    w = synthetic.seeded_state_dict(synthetic.processor_shapes(L, ["mesh_edges"], "pna"), 21)
    v0 = synthetic.seeded_tensor("v0", (n, 128), 1)
    e0 = synthetic.seeded_tensor("e0", (E, 128), 1)
    wo = {k: t.clone().requires_grad_(True) for k, t in w.items()}
    vo, eo = v0.clone().requires_grad_(True), e0.clone().requires_grad_(True)
    ref = orc.processor(wo, "pna", "none", orc.MultiGraph([vo], [orc.EdgeSet("mesh_edges", eo, s, r)]))
    coef = synthetic.seeded_tensor("c15", (n, 128), 2)
    (ref.node_features[0] * coef).sum().backward()

    proc = _processor("none", "pna", L, ["mesh_edges"], w, precision)
    v, e = v0.cuda().requires_grad_(True), e0.cuda().requires_grad_(True)
    out = proc(hutil.MultiGraph([v], [hutil.EdgeSet("mesh_edges", e, s, r)]))
    (out.node_features[0] * coef.cuda()).sum().backward()
    fwd = rel_err(out.node_features[0], ref.node_features[0])
    fwd_e = rel_err(out.edge_sets[0].features, ref.edge_sets[0].features)
    gv, ge = rel_l2(v.grad, vo.grad), rel_l2(e.grad, eo.grad)
    gw = _weight_grad_checks(proc, wo, precision, "15 layers")
    print(f"\n15 layers [{precision}]: latents {fwd:.2e} / {fwd_e:.2e}, gradients (L2): v {gv:.2e}, e {ge:.2e}, worst weight {gw:.2e}; "
          f"max metric v {rel_err(v.grad, vo.grad):.2e}, e {rel_err(e.grad, eo.grad):.2e}")
    assert fwd < TOL[precision] and fwd_e < TOL[precision]
    bound = GRAD_L2[precision]["deep"]
    assert gv < bound and ge < bound and gw < bound


# ------------------------------------------------------------------------------------------------------------------
# width: 1000 x 125 slab, two layers, forward + backward
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_slab_1000x125_two_layers_forward_backward(precision):
    W, H, L = 1000, 125, 2
    s, r = synthetic.grid_edges_two_way(W, H)
    n, E = W * H, s.numel()
    w = synthetic.seeded_state_dict(synthetic.processor_shapes(L, ["mesh_edges"], "sum"), 22)
    v0 = synthetic.seeded_tensor("sv", (n, 128), 1)
    e0 = synthetic.seeded_tensor("se", (E, 128), 1)
    wo = {k: t.clone().requires_grad_(True) for k, t in w.items()}
    vo, eo = v0.clone().requires_grad_(True), e0.clone().requires_grad_(True)
    ref = orc.processor(wo, "sum", "none", orc.MultiGraph([vo], [orc.EdgeSet("mesh_edges", eo, s, r)]))
    coef = synthetic.seeded_tensor("sc", (n, 128), 2)
    (ref.node_features[0] * coef).sum().backward()

    proc = _processor("none", "sum", L, ["mesh_edges"], w, precision)
    v, e = v0.cuda().requires_grad_(True), e0.cuda().requires_grad_(True)
    out = proc(hutil.MultiGraph([v], [hutil.EdgeSet("mesh_edges", e, s, r)]))
    (out.node_features[0] * coef.cuda()).sum().backward()
    fwd = rel_err(out.node_features[0], ref.node_features[0])
    fwd_e = rel_err(out.edge_sets[0].features, ref.edge_sets[0].features)
    gv, ge = rel_l2(v.grad, vo.grad), rel_l2(e.grad, eo.grad)
    gw = _weight_grad_checks(proc, wo, precision, "slab")
    print(f"\nslab 1000x125 [{precision}]: latents {fwd:.2e} / {fwd_e:.2e}, gradients (L2): v {gv:.2e}, e {ge:.2e}, worst weight {gw:.2e}; "
          f"max metric v {rel_err(v.grad, vo.grad):.2e}, e {rel_err(e.grad, eo.grad):.2e}")
    assert fwd < TOL[precision] and fwd_e < TOL[precision]
    bound = GRAD_L2[precision]["slab"]
    assert gv < bound and ge < bound and gw < bound


# ------------------------------------------------------------------------------------------------------------------
# the benchmarked configuration itself: cfg5 full mesh, one layer
# ------------------------------------------------------------------------------------------------------------------
def _cfg5():
    s, r = synthetic.grid_edges_two_way(1000, 1000)
    n, E = 1_000_000, s.numel()
    assert E == 5_992_002
    g = torch.Generator().manual_seed(5)
    v0 = torch.randn(n, 128, generator=g)
    e0 = torch.randn(E, 128, generator=g)
    w = synthetic.seeded_state_dict(synthetic.processor_shapes(1, ["mesh_edges"], "sum"), 23)
    return s, r, n, E, v0, e0, w


def test_cfg5_full_mesh_sampled_rows_and_cross_mode_gradients():
    s, r, n, E, v0, e0, w = _cfg5()
    rng = np.random.default_rng(9)
    # sampled edges: the first and last tile, a tile boundary, and 1 500 random rows
    edge_rows = np.unique(np.concatenate([np.arange(0, 130), np.arange(E - 130, E), np.arange(128 * 148 * 100 - 3, 128 * 148 * 100 + 3),
                                          rng.integers(0, E, 1500)]))
    node_rows = np.unique(np.concatenate([np.arange(0, 130), np.arange(n - 130, n), rng.integers(0, n, 800)]))
    er, nr = torch.from_numpy(edge_rows), torch.from_numpy(node_rows)
    pre = "processor.graphnet_blocks.0"
    x = torch.cat([v0[s[er]], v0[r[er]], e0[er]], -1)
    edge_ref = e0[er] + orc.mlp(w, f"{pre}.edge_models.mesh_edges", x)
    order = torch.sort(r, stable=True).indices
    rowptr = torch.zeros(n + 1, dtype=torch.int64)
    rowptr[1:] = torch.bincount(r, minlength=n).cumsum(0)
    coef = torch.randn(n, 128, generator=torch.Generator().manual_seed(6))
    results = {}
    for precision in ("fp32", "bf16"):
        proc = _processor("none", "sum", 1, ["mesh_edges"], w, precision)
        proc.restore_edge_dtype = True
        v, e = v0.cuda().requires_grad_(True), e0.cuda().requires_grad_(True)
        out = proc(hutil.MultiGraph([v], [hutil.EdgeSet("mesh_edges", e, s, r)]))
        (out.node_features[0] * coef.cuda()).sum().backward()
        new_e = out.edge_sets[0].features.detach()
        got_e = new_e[er.cuda()].float().cpu()
        err_e = rel_err(got_e, edge_ref)
        # aggregation + node update of the sampled receivers from the GPU's own e' (checks the 6 M-row CSR pass) and the oracle MLP
        agg = torch.stack([new_e[order[rowptr[j]:rowptr[j + 1]].cuda()].float().sum(0).cpu() for j in node_rows.tolist()])
        node_ref = v0[nr] + orc.mlp(w, f"{pre}.node_model_cross", torch.cat([v0[nr], agg], -1))
        err_v = rel_err(out.node_features[0].detach()[nr.cuda()].cpu(), node_ref)
        print(f"\ncfg5 full mesh [{precision}]: sampled edge rows {err_e:.2e} ({len(edge_rows)}), sampled node rows {err_v:.2e} ({len(node_rows)})")
        assert err_e < TOL[precision] and err_v < TOL[precision]
        grads = {k: p.grad.detach().clone() for k, p in proc.named_parameters()}
        results[precision] = (v.grad.detach().clone(), e.grad.detach().clone(), grads)
        if precision == "bf16":                 # run-to-run bit identity at the full size (no float atomics anywhere)
            proc.zero_grad()
            v2, e2 = v0.cuda().requires_grad_(True), e0.cuda().requires_grad_(True)
            out2 = proc(hutil.MultiGraph([v2], [hutil.EdgeSet("mesh_edges", e2, s, r)]))
            (out2.node_features[0] * coef.cuda()).sum().backward()
            assert torch.equal(out2.node_features[0], out.node_features[0]) and torch.equal(v2.grad, v.grad) and torch.equal(e2.grad, e.grad)
            for k, p in proc.named_parameters():
                assert torch.equal(p.grad, grads[k]), k
        del proc, v, e, out
        torch.cuda.empty_cache()
    # the tcgen05 backward against the FFMA backward (which is pinned to the oracle at 1e-4 on the smaller meshes above)
    gv = rel_l2(results["bf16"][0], results["fp32"][0])
    ge = rel_l2(results["bf16"][1], results["fp32"][1])
    gw = max(rel_l2(results["bf16"][2][k], results["fp32"][2][k]) for k in results["fp32"][2])
    print(f"cfg5 full mesh: bf16 vs fp32 backward, relative L2: grad v {gv:.2e}, grad e {ge:.2e}, worst weight grad {gw:.2e}")
    assert max(gv, ge, gw) < GRAD_L2["bf16"]["cfg5"]


def test_cfg5_full_mesh_edge_kernels_vs_bf16_emulation():
    """The projected edge update (node projection, fused forward kernel, receiver aggregate, fused backward kernel with the
    aggregate's gradient gathered inside, G0 segment sums, node-level dgrad / wgrad) on the FULL cfg5 mesh -- 5 992 002 edges,
    46 813 tiles, 317 per CTA -- against torch arithmetic with the same rounding points (tests/test_gpu_parity.py pins the same
    comparison at up to 200 k rows).  Forward 1e-2 (bf16 output rounding), gradients 1.5e-2 in relative L2."""
    from hgn_b200 import ops
    from hgn_b200.plan import segment_plan
    from test_gpu_parity import _bf16_emulated_projected_edge, _random_mlp_weights
    s, r = (t.cuda() for t in synthetic.grid_edges_two_way(1000, 1000))
    n, E = 1_000_000, s.numel()
    torch.manual_seed(7)
    w = _random_mlp_weights(3, 11)
    params = [w[f"m.0.layers.linear_{k}.{p}"].cuda().requires_grad_(True) for k in range(3) for p in ("weight", "bias")]
    params += [w["m.1.weight"].cuda().requires_grad_(True), w["m.1.bias"].cuda().requires_grad_(True)]
    v = torch.randn(n, 128, device="cuda").to(torch.bfloat16).requires_grad_(True)
    e = torch.randn(E, 128, device="cuda").to(torch.bfloat16).requires_grad_(True)
    gup = torch.randn(E, 128, device="cuda").to(torch.bfloat16)
    gagg = torch.randn(n, 128, device="cuda").to(torch.bfloat16)
    sp, rp = segment_plan(s, n), segment_plan(r, n)
    out, agg = ops.edge_update(params, {}, v, e, sp, rp, True)
    torch.autograd.backward([out, agg], [gup, gagg])
    wr = [p.detach().clone().requires_grad_(True) for p in params]
    vf, ef = v.detach().float().requires_grad_(True), e.detach().float().requires_grad_(True)
    ref = _bf16_emulated_projected_edge(vf, ef, s, r, wr)
    ref_agg = torch.zeros(n, 128, device="cuda").index_add_(0, r, ref)
    torch.autograd.backward([ref, ref_agg], [gup.float(), gagg.float()])
    errs = {"out": rel_err(out.float(), ref), "agg": rel_err(agg.float(), ref_agg), "grad_e": rel_l2(e.grad.float(), ef.grad),
            "grad_v": rel_l2(v.grad.float(), vf.grad), "grad_w": max(rel_l2(a.grad, b.grad) for a, b in zip(params, wr))}
    print("\ncfg5 full mesh, edge kernels vs bf16 emulation: " + ", ".join(f"{k} {x:.2e}" for k, x in errs.items()))
    assert errs["out"] < 1e-2 and errs["agg"] < 1e-2
    assert errs["grad_e"] < 1e-2 and errs["grad_v"] < 1.5e-2 and errs["grad_w"] < 1.5e-2


def test_cfg5_full_mesh_sum_layer_vs_bf16_emulation():
    """The fused 'sum' block (ops.graphnet_sum_layer, what bench.py times) on the FULL cfg5 mesh, both outputs in the loss, against the
    composed emulation of tests/test_gpu_parity.py: globally and over the first tile, the last tile and the first wrap of the grid."""
    from test_gpu_parity import _sum_layer_vs_emulation
    s, r = (t.cuda() for t in synthetic.grid_edges_two_way(1000, 1000))
    _sum_layer_vs_emulation(s, r, 1_000_000, "both", seed=8, repeat=False)
    torch.cuda.empty_cache()


def test_tile_kernel_multi_slab_backward_vs_bf16_emulation():
    """Above 2^21 rows the tile kernels' backward runs in slabs: the tile kernel at a row offset slab0, the workspaces addressed with
    slab-local rows, the weight-gradient partials and the bias / LayerNorm column sums accumulated from the second slab on.  A node update
    of 6 chunks ('sum' over five edge sets) on 2^21 + 401 mesh rows -- two slabs, the last tile partial -- against the emulation, with
    an extra window across the slab boundary.  A slab dropped or overwritten moves the parameter gradients by O(1)."""
    from test_gpu_parity import _node_update_tile_kernel_vs_emulation
    slab = 1 << 21
    torch.cuda.empty_cache()
    torch.cuda.reset_peak_memory_stats()
    _node_update_tile_kernel_vs_emulation(6, "mesh", slab + 401, 16, True, extra_windows={"slab boundary": (slab - 128, slab + 128)})
    print(f"multi-slab backward: peak device memory {torch.cuda.max_memory_allocated() / 2**30:.1f} GiB")
    torch.cuda.empty_cache()
