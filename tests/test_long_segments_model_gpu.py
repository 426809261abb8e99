"""bf16 HyperGraphNet and HeteroGraphNet processors whose cluster segments are long, with the split against the same step on the
existing segment kernels.

The remote edge sets come from ``rmp.hierarchical_connector.connector_indices`` over a grid mesh (``synthetic.grid_edges_two_way``)
clustered into bands of consecutive node ids: every cluster is one segment of ~N/C elements in the pooling (receivers) and in the
broadcast (senders).  One step (forward, backward of a random projection of every output) runs three times: twice with the split and
once with every plan's split bypassed (``ops._split_of`` returning None, so every binding calls the existing kernels).  The two split
runs must be bit-identical; split against existing kernels is held to test_gpu_parity.py's emulation bounds and row windows (forward
1e-2 in the max metric, gradients 1e-2 / 1.5e-2 in relative L2 over the whole tensor and over the first tile, the last tile and the
grid wrap).  The only difference between the two is the summation order of the long segments' sums and means; the pooled rows are
chosen so that the forward sums are exact (see _run_case), which leaves the backward's long sums as the difference.

Every call of ``ops._split_of`` is recorded: the split must be taken by the forward and the backward bindings of the remote sets, and
no call may see a plan with a split but a different segment or element count (that would fall back to the existing kernels).
"""
import pytest
import torch

from conftest import rel_err, rel_l2
from hgn_b200 import ops, synthetic
from hgn_b200.migration.meshgraphnet import MeshGraphNet
from hgn_b200.util import EdgeSet, MultiGraph

pytestmark = pytest.mark.gpu


def _windows(rows):
    if rows <= 128:
        return []
    wins = [(0, 128), ((rows - 1) // 128 * 128, rows)]
    wrap = torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count * 128
    if wrap < rows:
        wins.append((wrap - 64, min(wrap + 64, rows)))
    return wins


def _errs(got, want, metric):
    got, want = got.float(), want.float()
    return metric(got, want), max((rel_l2(got[lo:hi], want[lo:hi]) for lo, hi in _windows(got.shape[0])), default=0.0)


class _Spy:
    """Records (binding, split taken) for every ``ops._split_of`` call, and every call that saw a plan's split but did not take it."""

    def __init__(self, monkeypatch, bypass):
        self.calls, self.mismatched = [], []
        orig = ops._split_of

        def split_of(plan, S, E):
            import inspect
            caller = inspect.stack()[1].function
            sp = None if bypass else orig(plan, S, E)
            if not bypass and sp is None and plan.split is not None:
                self.mismatched.append((caller, S, E, plan.num_segments, plan.num_elements))
            self.calls.append((caller, sp is not None))
            return sp
        monkeypatch.setattr(ops, "_split_of", split_of)


def _step(proc, inputs, edges, grads_out, monkeypatch, bypass):
    spy = _Spy(monkeypatch, bypass)
    proc.zero_grad(set_to_none=True)
    v = [t.detach().clone().requires_grad_(True) for t in inputs["nodes"]]
    e = {nm: t.detach().clone().requires_grad_(True) for nm, t in inputs["edges"].items()}
    graph = MultiGraph(list(v), [EdgeSet(nm, e[nm], s, r) for nm, (s, r) in edges.items()])
    out = proc(graph)
    sets = list(out.edge_sets)                  # a HyperGraphNet block returns them in its phase order
    outs = list(out.node_features) + [x.features for x in sets]
    n_fwd = len(spy.calls)
    torch.autograd.backward(outs, grads_out["nodes"] + [grads_out["edges"][x.name] for x in sets])
    torch.cuda.synchronize()
    res = {f"out node {i}": t.detach() for i, t in enumerate(out.node_features)}
    res.update({f"out {x.name}": x.features.detach() for x in sets})
    res.update({f"grad node {i}": t.grad for i, t in enumerate(v)})
    res.update({f"grad {nm}": t.grad for nm, t in e.items()})
    res.update({f"grad {n}": p.grad for n, p in proc.named_parameters() if p.grad is not None})
    monkeypatch.undo()
    return res, spy, spy.calls[:n_fwd], spy.calls[n_fwd:]


def _run_case(arch, agg, width, height, clusters, layers, monkeypatch):
    torch.manual_seed(11)
    edges = {nm: (s.cuda(), r.cuda()) for nm, (s, r) in synthetic.hyper_grid_edges(width, height, clusters).items()}
    n = width * height
    w = synthetic.seeded_state_dict(synthetic.hyper_processor_shapes(arch, agg, layers), 5)
    proc = MeshGraphNet(3, 128, 2, agg, layers, arch, list(synthetic.HYPER_EDGE_SETS)).processor
    # The pooled rows are made exact in any summation order: the pooling edge model's LayerNorm has zero gain and bias, so its e' is
    # its input e, eighths of integers in [-4, 4] (sums of up to 2^21 / 32 such rows are exact in fp32).  So the two paths give the
    # same forward, bit for bit, and no ReLU unit of the few hyper rows switches between them (with one row per cluster, one such
    # switch moves a hyper MLP's weight gradient by O(10 %), a property of bf16 training, not of the kernels).  The backward still
    # sums inexact rows over the long segments (G0 of the pooling and broadcast edges by hyper node), in the split's order.
    for k in w:
        if ".edge_models.intra_cluster_to_cluster.1." in k:
            w[k] = torch.zeros_like(w[k])
    proc.load_state_dict({k[len("processor."):]: t for k, t in w.items()})
    proc = proc.cuda()
    proc.precision = "bf16"
    inputs = {"nodes": [torch.randn(n, 128, device="cuda"), torch.randn(clusters, 128, device="cuda")],
              "edges": {nm: torch.randn(s.numel(), 128, device="cuda") for nm, (s, _) in edges.items()}}
    pooled = inputs["edges"]["intra_cluster_to_cluster"]
    pooled.copy_(torch.randint(-32, 33, pooled.shape, device="cuda").float() / 8)
    grads_out = {"nodes": [torch.randn(n, 128, device="cuda"), torch.randn(clusters, 128, device="cuda")],
                 "edges": {nm: torch.randn(s.numel(), 128, device="cuda").to(torch.bfloat16) for nm, (s, _) in edges.items()}}

    new, spy, fwd, bwd = _step(proc, inputs, edges, grads_out, monkeypatch, bypass=False)
    again, _, _, _ = _step(proc, inputs, edges, grads_out, monkeypatch, bypass=False)
    old, _, _, _ = _step(proc, inputs, edges, grads_out, monkeypatch, bypass=True)

    assert not spy.mismatched, f"bindings saw a split plan with other sizes: {spy.mismatched}"
    taken_fwd = sorted({c for c, t in fwd if t})
    taken_bwd = sorted({c for c, t in bwd if t})
    print(f"\n{arch} {agg} {n} nodes / {clusters} clusters: split taken forward by {taken_fwd}, backward by {taken_bwd}")
    assert taken_fwd and taken_bwd, "the long cluster segments did not reach the split"

    for k in new:
        assert torch.equal(new[k].view(torch.int16) if new[k].dtype == torch.bfloat16 else new[k],
                           again[k].view(torch.int16) if again[k].dtype == torch.bfloat16 else again[k]), f"{k}: two runs differ"
    checks = {}
    for k, t in new.items():
        if k.startswith("out"):
            assert torch.equal(t, old[k]), f"{k}: the forward differs from the existing kernels' although its long sums are exact"
            checks[k] = (*_errs(t, old[k], rel_err), 1e-2)
        else:
            bound = 1e-2 if k[len("grad "):] in edges else 1.5e-2     # edge latents 1e-2; node latents and weights 1.5e-2
            checks[k] = (*_errs(t, old[k], rel_l2), bound)
    worst = max(checks.items(), key=lambda kv: max(kv[1][0], kv[1][1]))
    differ = sum(not torch.equal(new[k], old[k]) for k in new)
    print(f"{differ} of {len(new)} tensors differ from the existing kernels' bits; worst: {worst[0]} {worst[1][0]:.2e} / windows "
          f"{worst[1][1]:.2e}")
    bad = [k for k, (g, win, b) in checks.items() if not (g < b and win < b)]
    assert not bad, f"beyond the bound: {[(k, checks[k]) for k in bad]}"


@pytest.mark.parametrize("agg", ["sum", "pna"])
@pytest.mark.parametrize("arch", ["hyper", "hetero"])
def test_processor_split_vs_existing_kernels(arch, agg, monkeypatch):
    _run_case(arch, agg, 448, 448, 8, 2, monkeypatch)           # ~200 k nodes, clusters of ~25 000


def test_processor_split_vs_existing_kernels_1000x1000(monkeypatch):
    _run_case("hyper", "sum", 1000, 1000, 16, 1, monkeypatch)   # 62 500 nodes per cluster
