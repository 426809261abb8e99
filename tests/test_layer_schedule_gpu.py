"""One schedule for the one-GPU and the partitioned GraphNet layer (``ops._GraphNetSumLayer``), and ``ops.launch_count`` against the
kernels that actually run (``-m gpu``, one B200).

* The partitioned processor at world size 1 (gloo; ``PeerHalo`` without peers, so its exchanges launch nothing) owns every node and
  edge in their original order: over three steps (both table parities) its outputs and every gradient equal the processor's on the
  whole graph bit for bit.
* For one fwd+bwd step after a warm-up step, the change in ``ops.launch_count`` equals the number of ``hgn::`` kernels
  ``torch.profiler`` records: the fused 'sum' layer, a bf16 'pna' block (node update with 4 aggregates), the partitioned layer.
"""
import pytest
import torch
import torch.distributed as dist

from hgn_b200 import ops, partition, synthetic
from hgn_b200.migration.meshgraphnet import MeshGraphNet
from hgn_b200.util import EdgeSet, MultiGraph

pytestmark = pytest.mark.gpu

W, H, LAYERS = 40, 32, 3


@pytest.fixture(scope="module")
def mesh():
    s, r = synthetic.grid_edges_two_way(W, H)
    gen = torch.Generator().manual_seed(0)
    n, e = W * H, s.numel()
    v0, e0, coef = torch.randn(n, 128, generator=gen), torch.randn(e, 128, generator=gen), torch.randn(n, 128, generator=gen)
    return s, r, v0.cuda(), e0.cuda(), coef.cuda()


def _processor(aggregator, layers):
    weights = synthetic.seeded_state_dict(synthetic.processor_shapes(layers, ["mesh_edges"], aggregator), seed=17)
    proc = MeshGraphNet(3, 128, 2, aggregator, layers, "none", ["mesh_edges"]).processor
    proc.load_state_dict({k[len("processor."):]: t for k, t in weights.items()})
    proc = proc.cuda()
    proc.precision = "bf16"
    return proc


def _whole(proc, s, r):
    s, r = s.cuda(), r.cuda()

    def run(v, e):
        out = proc(MultiGraph([v], [EdgeSet("mesh_edges", e, s, r)]))
        return out.node_features[0], out.edge_sets[0].features
    return run


def _step(run, params, v0, e0, coef, shift=0.0):
    """One fwd+bwd step: outputs, both input gradients and every parameter gradient."""
    for p in params:
        p.grad = None
    v = (v0 + shift).requires_grad_(True)
    e = e0.clone().requires_grad_(True)
    out_v, out_e = run(v, e)
    ((out_v * coef).sum() + (out_e.float() ** 2).sum() * 1e-3).backward()
    return [out_v.detach(), out_e.detach(), v.grad, e.grad] + [p.grad.clone() for p in params]


@pytest.fixture
def split(tmp_path, mesh):
    """The 3-layer bf16 'sum' processor and its world-size-1 partitioned wrapper; the pool and the process group go away after."""
    s, r, v0, e0, _ = mesh
    dist.init_process_group("gloo", store=dist.FileStore(str(tmp_path / "store"), 1), rank=0, world_size=1)
    dev = torch.device("cuda", torch.cuda.current_device())
    lg = partition.build_local_graph(s, r, partition.block_partition(W * H, 1), 0, 1)
    peer = partition.PeerHalo(lg, LAYERS, dev)
    proc = _processor("sum", LAYERS)
    model = partition.PartitionedProcessor(proc, partition.HaloPlan(lg, dev), peer)
    s_loc, r_loc = lg.senders.to(dev), lg.receivers.to(dev)
    assert model._fast_path(v0.to(torch.bfloat16), [EdgeSet("mesh_edges", e0.to(torch.bfloat16), s_loc, r_loc)])

    def run(v, e):
        out_v, out_sets = model(v, [EdgeSet("mesh_edges", e, s_loc, r_loc)])
        return out_v, out_sets[0].features
    try:
        yield proc, run
    finally:
        peer.close()
        dist.destroy_process_group()


def test_world1_partitioned_equals_processor_bitwise(split, mesh):
    s, r, v0, e0, coef = mesh
    proc, run_split = split
    run_whole = _whole(proc, s, r)
    params = list(proc.parameters())
    for step in range(3):
        shift = 0.01 * step
        whole = _step(run_whole, params, v0, e0, coef, shift)
        parted = _step(run_split, params, v0, e0, coef, shift)
        for i, (a, b) in enumerate(zip(parted, whole)):
            assert torch.equal(a, b), (step, i)


def _launches(run, params, v0, e0, coef):
    """(change in ops.launch_count, hgn:: kernels in the profiler) over one step after a warm-up step."""
    _step(run, params, v0, e0, coef)
    torch.cuda.synchronize()
    before = ops.launch_count
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        _step(run, params, v0, e0, coef)
        torch.cuda.synchronize()
    counted = ops.launch_count - before
    return counted, sum(1 for ev in prof.events() if "hgn::" in ev.name)


@pytest.mark.parametrize("aggregator", ["sum", "pna"])
def test_launch_count_one_gpu(aggregator, mesh):
    s, r, v0, e0, coef = mesh
    proc = _processor(aggregator, 1)
    counted, kernels = _launches(_whole(proc, s, r), list(proc.parameters()), v0, e0, coef)
    assert kernels > 0 and counted == kernels, (counted, kernels)


def test_launch_count_partitioned(split, mesh):
    _, _, v0, e0, coef = mesh
    proc, run_split = split
    counted, kernels = _launches(run_split, list(proc.parameters()), v0, e0, coef)
    assert kernels > 0 and counted == kernels, (counted, kernels)
