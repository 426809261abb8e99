"""The partitioned HyperGraphNet processor on one GPU, and on 2 and 4 GPUs of one box.

* ``hgn_segment_partials`` (fp32, unrounded) followed by the one-rank ``hgn_cluster_combine`` equals the existing segment kernels bit for
  bit after bf16 rounding, for segment sizes 0 .. 33 and for segments longer than the split threshold (the split route).
* World size 1 (gloo, a ``PeerHalo`` and a cluster pool without peers): over three steps and for every aggregator, the forward (owned
  latents, hyper rows, edge latents) equals the one-GPU HyperGraphNet processor bit for bit, the gradients are within relative L2 2e-2
  (the fused mesh layer adds its two partial gradients of v in fp32; the pooling's 'mean' term and max / min winners are added to the
  edge gradient in another rounding order), and two runs are bit-identical.
* 2 and 4 GPUs: ``tests/partition_hyper_gpu_worker.py`` under torch.distributed.run (skipped with fewer GPUs)."""
import os
import socket
import subprocess
import sys

import pytest
import torch
import torch.distributed as dist

from conftest import ROOT, rel_l2
from hgn_b200 import _cabi, ops, partition, synthetic
from hgn_b200._cabi import HgnError
from hgn_b200.migration.meshgraphnet import MeshGraphNet
from hgn_b200.plan import segment_plan
from hgn_b200.util import EdgeSet, MultiGraph

pytestmark = pytest.mark.gpu
AGGREGATORS = ["sum", "mean", "max", "min", "pna"]


def _bits(t):
    return t.view(torch.int16) if t.dtype == torch.bfloat16 else t


def _partials_case(sizes, seed):
    gen = torch.Generator().manual_seed(seed)
    S = len(sizes)
    ids = torch.repeat_interleave(torch.arange(S), torch.tensor(sizes))
    ids = ids[torch.randperm(ids.numel(), generator=gen)].cuda()         # segment members spread over the rows
    data = torch.randn(ids.numel(), 128, generator=gen).cuda().to(torch.bfloat16)
    return data, segment_plan(ids, S), ids


@pytest.mark.parametrize("sizes", [list(range(34)), [0, 2049, 1, 5000, 33, 7000, 0, 2304, 2048]], ids=["short", "long"])
def test_partials_and_one_rank_combine_equal_existing_kernels(sizes):
    data, plan, ids = _partials_case(sizes, 3)
    S = len(sizes)
    if max(sizes) > 2048:
        assert plan.split is not None and plan.split.n_long == sum(n > 2048 for n in sizes)
    want_sum, want_mean, want_max, want_min = ops.segment_aggregate(data.detach().requires_grad_(True), plan, ["sum", "mean", "max", "min"])
    only_sum = ops.segment_aggregate(data, plan, ["sum"])[0]
    # the winners of the existing kernels, through their own binding
    am, an = torch.empty((S, 128), dtype=torch.int32, device="cuda"), torch.empty((S, 128), dtype=torch.int32, device="cuda")
    ops._segment_reduce(data, plan, [None, None, torch.empty_like(want_max), torch.empty_like(want_min)], am, an)
    for minmax in (False, True):
        part = torch.empty((S, _cabi.HGN_SEGMENT_PARTIAL_WIDTH), dtype=torch.float32, device="cuda")
        pam = torch.empty((S, 128), dtype=torch.int32, device="cuda") if minmax else None
        pan = torch.empty((S, 128), dtype=torch.int32, device="cuda") if minmax else None
        ops._segment_partials(data, plan, part, minmax, pam, pan)
        counts = part[:, 384].view(torch.int32)
        assert torch.equal(counts.cpu(), torch.tensor(sizes, dtype=torch.int32))
        assert torch.equal(_bits(part[:, :128].to(torch.bfloat16)), _bits(want_sum)) and torch.equal(_bits(want_sum), _bits(only_sum))
        outs = [torch.empty_like(want_sum) for _ in range(4)] if minmax else [torch.empty_like(want_sum), torch.empty_like(want_sum), None, None]
        count = torch.empty(S, dtype=torch.int32, device="cuda")
        ops._cluster_combine(part[None], 1, 0, outs, pam, pan, count)
        assert torch.equal(count, counts)
        assert torch.equal(_bits(outs[0]), _bits(want_sum)) and torch.equal(_bits(outs[1]), _bits(want_mean))
        if minmax:
            assert torch.equal(_bits(outs[2]), _bits(want_max)) and torch.equal(_bits(outs[3]), _bits(want_min))
            assert torch.equal(pam, am) and torch.equal(pan, an)


def test_combine_skips_ranks_without_members_and_sums_in_rank_order():
    """Two ranks' partial rows: a rank with count 0 takes no part in max / min (its -inf / +inf rows are not values), a cluster empty
    on both yields 0, sums are added in rank order from +0, and the winners of the other rank are cleared."""
    W = _cabi.HGN_SEGMENT_PARTIAL_WIDTH
    slots = torch.zeros((2, 3, W), dtype=torch.float32, device="cuda")
    gen = torch.Generator().manual_seed(5)
    vals = torch.randn(2, 3, 3, 128, generator=gen).cuda()
    slots[..., :384] = vals.reshape(2, 3, 384)
    cnt = torch.tensor([[4, 0, 0], [2, 3, 0]], dtype=torch.int32, device="cuda")
    slots[..., 384] = cnt.view(torch.float32)
    slots[1, 2, 128:256], slots[1, 2, 256:384] = -float("inf"), float("inf")
    slots[0, 1, 128:256], slots[0, 1, 256:384] = 1e30, -1e30          # rank 0 has no member of cluster 1: its rows are not values
    outs = [torch.empty((3, 128), dtype=torch.bfloat16, device="cuda") for _ in range(4)]
    for rank in (0, 1):
        am = torch.full((3, 128), 7, dtype=torch.int32, device="cuda")
        an = torch.full((3, 128), 7, dtype=torch.int32, device="cuda")
        count = torch.empty(3, dtype=torch.int32, device="cuda")
        ops._cluster_combine(slots, 2, rank, outs, am, an, count)
        assert count.tolist() == [6, 3, 0]
        s = (slots[0, :, :128] + slots[1, :, :128])
        assert torch.equal(_bits(outs[0]), _bits(s.to(torch.bfloat16)))
        mx0, mx1 = slots[0, 0, 128:256], slots[1, 0, 128:256]
        assert torch.equal(outs[2][0], torch.maximum(mx0, mx1).to(torch.bfloat16))
        assert torch.equal(outs[2][1], slots[1, 1, 128:256].to(torch.bfloat16)) and torch.equal(outs[3][1], slots[1, 1, 256:384].to(torch.bfloat16))
        assert (outs[2][2] == 0).all() and (outs[3][2] == 0).all()
        won0 = mx0 >= mx1                                               # strict comparisons: rank 0 keeps a tie
        keep = won0 if rank == 0 else ~won0
        assert torch.equal(am[0] == 7, keep) and (am[1] == (7 if rank == 1 else -1)).all() and (am[2] == -1).all()
    g = torch.randn(3, 3, 128, generator=gen).cuda().to(torch.bfloat16)
    out = torch.empty((3, 128), dtype=torch.bfloat16, device="cuda")
    ops._cluster_grad_sum(g, out)
    assert torch.equal(_bits(out), _bits(((g[0].float() + g[1].float()) + g[2].float()).to(torch.bfloat16)))


# ---- world size 1 ----------------------------------------------------------------------------------------------------------------
LAYERS = 2


def _hyper_graph(width, height, clusters):
    sets = synthetic.hyper_grid_edges(width, height, clusters)
    return sets, width * height


def _hyper_processor(agg, layers=LAYERS, seed=5):
    w = synthetic.seeded_state_dict(synthetic.hyper_processor_shapes("hyper", agg, layers), seed)
    proc = MeshGraphNet(3, 128, 2, agg, layers, "hyper", list(synthetic.HYPER_EDGE_SETS)).processor
    proc.load_state_dict({k[len("processor."):]: t for k, t in w.items()})
    proc = proc.cuda()
    proc.precision = "bf16"
    return proc


def _inputs(sets, n, clusters, seed=1):
    gen = torch.Generator().manual_seed(seed)
    v = torch.randn(n, 128, generator=gen)
    h = torch.randn(clusters, 128, generator=gen)
    e = {nm: torch.randn(s.numel(), 128, generator=gen) for nm, (s, _) in sets.items()}
    cv, ch = torch.randn(n, 128, generator=gen), torch.randn(clusters, 128, generator=gen)
    return [t.cuda() for t in (v, h, cv, ch)] + [{nm: t.cuda() for nm, t in e.items()}]


def _loss(v, h, e, cv, ch):
    return (v * cv).sum() + (h * ch).sum() + sum((x.float() ** 2).sum() for x in e.values()) * 1e-3


def _one_gpu_step(proc, sets, inp, shift):
    v0, h0, cv, ch, e0 = inp
    proc.zero_grad(set_to_none=True)
    v = (v0 + shift).requires_grad_(True)
    h = h0.clone().requires_grad_(True)
    e = {nm: t.clone().requires_grad_(True) for nm, t in e0.items()}
    out = proc(MultiGraph([v, h], [EdgeSet(nm, e[nm], s.cuda(), r.cuda()) for nm, (s, r) in sets.items()]))
    oe = {es.name: es.features for es in out.edge_sets}
    _loss(out.node_features[0], out.node_features[1], oe, cv, ch).backward()
    res = {"v": out.node_features[0].detach(), "h": out.node_features[1].detach(), **{f"e {k}": t.detach() for k, t in oe.items()}}
    grads = {"grad v": v.grad, "grad h": h.grad, **{f"grad e {k}": t.grad for k, t in e.items()}}
    grads.update({f"grad {n}": p.grad.clone() for n, p in proc.named_parameters() if p.grad is not None})
    return res, grads


def _parted_step(model, proc, sets, inp, shift):
    v0, h0, cv, ch, e0 = inp
    proc.zero_grad(set_to_none=True)
    v = (v0 + shift).requires_grad_(True)
    h = h0.clone().requires_grad_(True)
    e = {nm: t.clone().requires_grad_(True) for nm, t in e0.items()}
    ov, oes, oh = model(v, [EdgeSet(nm, e[nm], s.cuda(), r.cuda()) for nm, (s, r) in sets.items()], h)
    oe = {es.name: es.features for es in oes}
    _loss(ov, oh, oe, cv, ch).backward()           # one rank: nothing to all-reduce
    res = {"v": ov.detach(), "h": oh.detach(), **{f"e {k}": t.detach() for k, t in oe.items()}}
    grads = {"grad v": v.grad, "grad h": h.grad, **{f"grad e {k}": t.grad for k, t in e.items()}}
    grads.update({f"grad {n}": p.grad.clone() for n, p in proc.named_parameters() if p.grad is not None})
    return res, grads


@pytest.fixture
def world1(tmp_path):
    dist.init_process_group("gloo", store=dist.FileStore(str(tmp_path / "store"), 1), rank=0, world_size=1)
    yield
    dist.destroy_process_group()


@pytest.mark.parametrize("mesh", [(96, 64, 4), (128, 96, 4)], ids=["short_clusters", "long_clusters"])
@pytest.mark.parametrize("agg", AGGREGATORS)
def test_world1_hyper_forward_bitwise_gradients_close(agg, mesh, world1):
    width, height, clusters = mesh
    sets, n = _hyper_graph(width, height, clusters)
    dev = torch.device("cuda", torch.cuda.current_device())
    lh = partition.build_local_hyper_graph(sets, n, clusters, partition.block_partition(n, 1), 0, 1)
    local = {"mesh_edges": (lh.mesh.senders, lh.mesh.receivers), **{nm: (x.senders, x.receivers) for nm, x in lh.remote.items()}}
    for nm, (s, r) in sets.items():                 # one rank: the local lists are the global ones
        assert torch.equal(local[nm][0], s) and torch.equal(local[nm][1], r)
    peer = partition.PeerHalo(lh.mesh, LAYERS, dev)
    proc = _hyper_processor(agg)
    model = partition.PartitionedProcessor(proc, partition.HaloPlan(lh.mesh, dev), peer, hyper=lh)
    try:
        inp = _inputs(sets, n, clusters)
        first = None
        for step in range(3):
            shift = 0.01 * step
            want, want_g = _one_gpu_step(proc, sets, inp, shift)
            got, got_g = _parted_step(model, proc, sets, inp, shift)
            for k in want:
                assert torch.equal(_bits(got[k]), _bits(want[k])), (step, k)
            errs = {k: rel_l2(got_g[k].float(), want_g[k].float()) for k in want_g}
            worst = max(errs.items(), key=lambda kv: kv[1])
            assert worst[1] < 2e-2, (step, worst)
            if first is None:
                first = (got, got_g)
        again, again_g = _parted_step(model, proc, sets, inp, 0.0)     # a fourth step repeats the first: bit-identical
        for k in first[0]:
            assert torch.equal(_bits(again[k]), _bits(first[0][k])), k
        for k in first[1]:
            assert torch.equal(again_g[k], first[1][k]), k
        print(f"\n{agg} {mesh}: forward bitwise over 3 steps; worst gradient {worst[0]} {worst[1]:.2e}")
    finally:
        model.close()
        peer.close()


def test_world1_hyper_refuses_fp32(world1):
    sets, n = _hyper_graph(32, 16, 2)
    dev = torch.device("cuda", torch.cuda.current_device())
    lh = partition.build_local_hyper_graph(sets, n, 2, partition.block_partition(n, 1), 0, 1)
    peer = partition.PeerHalo(lh.mesh, 1, dev)
    proc = _hyper_processor("sum", layers=1)
    proc.precision = "fp32"
    model = partition.PartitionedProcessor(proc, partition.HaloPlan(lh.mesh, dev), peer, hyper=lh)
    try:
        v0, h0, _, _, e0 = _inputs(sets, n, 2)
        with pytest.raises(HgnError, match="fp32 parity mode"):
            model(v0, [EdgeSet(nm, e0[nm], s.cuda(), r.cuda()) for nm, (s, r) in sets.items()], h0)
    finally:
        model.close()
        peer.close()


# ---- 2 and 4 GPUs ----------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("world", [2, 4])
def test_partitioned_hyper_matches_whole_graph(world):
    if torch.cuda.device_count() < world:
        pytest.skip(f"needs {world} GPUs, {torch.cuda.device_count()} visible")
    with socket.socket() as sock:
        sock.bind(("127.0.0.1", 0))
        port = sock.getsockname()[1]
    run = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}", "--master-addr", "127.0.0.1",
                          "--master-port", str(port), os.path.join(ROOT, "tests", "partition_hyper_gpu_worker.py")],
                         capture_output=True, text=True, timeout=1500)
    assert run.returncode == 0 and run.stdout.count("PARTITION-HYPER-GPU-OK") == world, run.stdout[-4000:] + run.stderr[-6000:]
    print("\n" + "\n".join(ln for ln in run.stdout.splitlines() if "PARTITION-HYPER" in ln))
