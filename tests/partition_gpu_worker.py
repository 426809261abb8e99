"""TEST INFRASTRUCTURE -- one rank of tests/test_partition_gpu.py (launched with torch.distributed.run, NCCL, one GPU per rank).

The partitioned processor on its two paths -- halo rows through NVLink peer memory (``partition.PeerHalo``, csrc/peer.cu) and the
generic path (node latents by NCCL grouped send/recv before every block) -- against each other and, on rank 0, against the SAME
bf16 processor run on the whole mesh on one GPU: latents of the owned rows, their gradients, edge latents and gradients, and the
all-reduced weight gradients.  Three consecutive steps, so that both table parities and the flag epochs are exercised."""
import os
import sys

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "hyper-graph-nets_b200"))
from hgn_b200 import partition, synthetic  # noqa: E402
from hgn_b200.migration.meshgraphnet import MeshGraphNet  # noqa: E402
from hgn_b200.util import EdgeSet, MultiGraph  # noqa: E402

rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
dev = torch.device("cuda", int(os.environ["LOCAL_RANK"]))
torch.cuda.set_device(dev)
dist.init_process_group("nccl", device_id=dev)
W, H, L = 160, 96, 3
s, r = synthetic.grid_edges_two_way(W, H)
n, e_total = W * H, s.numel()
part = partition.block_partition(n, world)
lg = partition.build_local_graph(s, r, part, rank, world)
gen = torch.Generator().manual_seed(0)
v_full, e_full, coef_full = (torch.randn(n, 128, generator=gen), torch.randn(e_total, 128, generator=gen), torch.randn(n, 128, generator=gen))
v0, e0, coef = v_full[lg.owned].to(dev), e_full[lg.edge_ids].to(dev), coef_full[lg.owned].to(dev)
weights = synthetic.seeded_state_dict(synthetic.processor_shapes(L, ["mesh_edges"], "sum"), seed=17)
proc = MeshGraphNet(3, 128, 2, "sum", L, "none", ["mesh_edges"]).processor
proc.load_state_dict({k[len("processor."):]: t for k, t in weights.items()})
proc = proc.to(dev)
proc.precision = "bf16"
plan = partition.HaloPlan(lg, dev)
peer = partition.PeerHalo(lg, L, dev)
fast = partition.PartitionedProcessor(proc, plan, peer)
generic = partition.PartitionedProcessor(proc, plan, None)
s_loc, r_loc = lg.senders.to(dev), lg.receivers.to(dev)
params = list(proc.parameters())


def run(model, shift):
    for p in params:
        p.grad = None
    v = (v0 + shift).requires_grad_(True)
    ed = e0.clone().requires_grad_(True)
    out_v, out_sets = model(v, [EdgeSet("mesh_edges", ed, s_loc, r_loc)])
    loss = (out_v * coef).sum() + (out_sets[0].features.float() ** 2).sum() * 1e-3
    loss.backward()
    partition.allreduce_gradients(proc)
    torch.cuda.synchronize()
    return [out_v.detach(), out_sets[0].features.detach().float(), v.grad, ed.grad] + [p.grad.clone() for p in params]


def rel(x, y):
    return float((x.double() - y.double()).norm() / y.double().norm().clamp_min(1e-30))


assert fast._fast_path(v0.to(torch.bfloat16), [EdgeSet("mesh_edges", e0.to(torch.bfloat16), s_loc, r_loc)])
worst_paths = worst_single = 0.0
for step in range(3):
    shift = 0.01 * step
    a, b = run(fast, shift), run(generic, shift)
    errs = [rel(x, y) for x, y in zip(a, b)]
    worst_paths = max(worst_paths, max(errs))
    # the peer path is the fused layer (the node update's share of d loss / d v is added in fp32 inside the dgrad kernel), the NCCL path the
    # generic block on [owned | ghost] rows (two bf16 partial gradients added by autograd): one rounding point differs per layer
    # (measured 6.4e-3 worst over 5 layers)
    assert max(errs) < 2e-2, (step, errs)
    if rank == 0:                                   # the whole mesh on this one GPU
        for p in params:
            p.grad = None
        vf = (v_full.to(dev) + shift).requires_grad_(True)
        ef = e_full.to(dev).requires_grad_(True)
        out = proc(MultiGraph([vf], [EdgeSet("mesh_edges", ef, s.to(dev), r.to(dev))]))
        ((out.node_features[0] * coef_full.to(dev)).sum() + (out.edge_sets[0].features.float() ** 2).sum() * 1e-3).backward()
        own, eid = lg.owned.to(dev), lg.edge_ids.to(dev)
        single = [out.node_features[0].detach()[own], out.edge_sets[0].features.detach().float()[eid], vf.grad[own], ef.grad[eid]] + [p.grad.clone() for p in params]
        errs1 = [rel(x, y) for x, y in zip(a, single)]
        worst_single = max(worst_single, max(errs1))
        assert max(errs1) < 5e-3, (step, errs1)     # same kernels, same rounding points; the ghost contributions are summed in another order
    dist.barrier()
print(f"PARTITION-GPU-OK rank {rank}/{world}: {lg.n_own} owned, {lg.n_ghost} ghosts, {lg.senders.numel()} edges; peer vs nccl path {worst_paths:.2e}"
      + (f"; vs the whole mesh on one GPU {worst_single:.2e}" if rank == 0 else ""), flush=True)
peer.close()
dist.destroy_process_group()
