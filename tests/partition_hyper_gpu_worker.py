"""TEST INFRASTRUCTURE -- one rank of tests/test_partition_hyper_gpu.py::test_partitioned_hyper_matches_whole_graph (launched with
torch.distributed.run, NCCL, one GPU per rank).

A HyperGraphNet processor partitioned in row slabs over a 448 x 448 grid (~200 k nodes), for the 'sum', 'pna' and 'max' aggregators.
The clusters are laid out so that the pooling meets every case of the cross-rank combine: column bands that straddle every rank
boundary (local segments longer than the split threshold), clusters held by rank 0 alone (the other ranks own no member), and clusters
whose share on a second rank is a short segment.  Over three consecutive steps (both table parities) rank 0 compares its owned rows,
the hyper rows, its local edge latents, the input gradients and the all-reduced weight gradients against
* the same schedule on the whole graph on rank 0 alone (a one-rank group: no halo, a one-rank combine): the forward bit for bit for
  'max' (every reduction of the forward is exact in any order), else within 5e-3 (same rounding points, another summation order); the
  gradients within 2e-2, because each rank rounds its share of the hyper rows' gradient to bf16 before the rank-ordered sum;
* the unmodified one-GPU processor: within 2e-2.
Every rank checks that the hyper rows, their input gradient and the replicated modules' gradients are bit-identical on all ranks, and
a repeated step reproduces the first bit for bit."""
import os
import sys

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "hyper-graph-nets_b200"))
from hgn_b200 import partition, synthetic  # noqa: E402
from hgn_b200.migration.meshgraphnet import MeshGraphNet  # noqa: E402
from hgn_b200.rmp.hierarchical_connector import connector_indices  # noqa: E402
from hgn_b200.util import EdgeSet, MultiGraph  # noqa: E402

rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
# one GPU per rank over NCCL; with fewer GPUs than ranks (run by hand: the test skips then) the ranks share the devices over gloo, which
# checks the exchanges' logic, not their speed
shared = torch.cuda.device_count() < world
dev = torch.device("cuda", int(os.environ["LOCAL_RANK"]) % torch.cuda.device_count())
torch.cuda.set_device(dev)
dist.init_process_group("gloo" if shared else "nccl", **({} if shared else {"device_id": dev}))
alone = dist.new_group([0])
W = H = 448
L = 2
n = W * H
y, x = torch.arange(n) // W, torch.arange(n) % W
cl = (x * 6) // W                                          # 0..5: column bands across every rank
top = y < H // 4                                           # inside rank 0's slab at 2 and 4 ranks
cl[top] = torch.where(x[top] < W // 2, 6, 7)
cl[top & (x >= W - 20)] = 8                                # 112 x 20 nodes, rank 0 only
cl[(y == H // 4) & (x < 50)] = 6                           # short spill into the next slab at 4 ranks
cl[(y == H // 2) & (x < 30)] = 7                           # short spill into the next slab at 2 ranks (at 4: rank 2)
C = 9
clusters = [torch.nonzero(cl == c).flatten() for c in range(C)]
sets = {"mesh_edges": synthetic.grid_edges_two_way(W, H), **connector_indices(clusters, [], n, fully_connect=True)}
part = partition.block_partition(n, world)
lh = partition.build_local_hyper_graph(sets, n, C, part, rank, world)
lh_whole = partition.build_local_hyper_graph(sets, n, C, partition.block_partition(n, 1), 0, 1) if rank == 0 else None
up_sizes = torch.bincount(lh.remote["intra_cluster_to_cluster"].receivers - lh.n_own, minlength=C).tolist()

gen = torch.Generator().manual_seed(0)
v_full, h_full = torch.randn(n, 128, generator=gen), torch.randn(C, 128, generator=gen)
e_full = {nm: torch.randn(s.numel(), 128, generator=gen) for nm, (s, _) in sets.items()}
cv_full, ch = torch.randn(n, 128, generator=gen), torch.randn(C, 128, generator=gen).to(dev)
local_idx = {"mesh_edges": (lh.mesh.edge_ids, lh.mesh.senders, lh.mesh.receivers),
             **{nm: (x_.edge_ids, x_.senders, x_.receivers) for nm, x_ in lh.remote.items()}}


def rel(a, b):
    return float((a.double() - b.double()).norm() / b.double().norm().clamp_min(1e-30))


def bits(t):
    return t.view(torch.int16) if t.dtype == torch.bfloat16 else t


def run(model, proc, owned, eids, idx, shift, exclude):
    """One step of a partitioned model on (owned node ids, edge ids per set, local indices per set)."""
    for p in proc.parameters():
        p.grad = None
    v = (v_full[owned].to(dev) + shift).requires_grad_(True)
    h = h_full.to(dev).requires_grad_(True)
    e = {nm: e_full[nm][eids[nm]].to(dev).requires_grad_(True) for nm in sets}
    ov, oes, oh = model(v, [EdgeSet(nm, e[nm], idx[nm][0].to(dev), idx[nm][1].to(dev)) for nm in sets], h)
    oe = {es.name: es.features for es in oes}
    loss = (ov * cv_full[owned].to(dev)).sum() + (oh * ch).sum() + sum((t.float() ** 2).sum() for t in oe.values()) * 1e-3
    loss.backward()
    if exclude is not None:
        partition.allreduce_gradients(proc, group=exclude[0], exclude=exclude[1])
    torch.cuda.synchronize()
    out = {"v": ov.detach(), "h": oh.detach(), **{f"e {k}": t.detach().float() for k, t in oe.items()},
           "grad v": v.grad, "grad h": h.grad, **{f"grad e {k}": t.grad.float() for k, t in e.items()}}
    out.update({f"grad {nm}": p.grad.clone() for nm, p in proc.named_parameters()})
    return out


worst = {}
for agg in ("sum", "pna", "max"):
    weights = synthetic.seeded_state_dict(synthetic.hyper_processor_shapes("hyper", agg, L), seed=17)
    proc = MeshGraphNet(3, 128, 2, agg, L, "hyper", list(synthetic.HYPER_EDGE_SETS)).processor
    proc.load_state_dict({k[len("processor."):]: t for k, t in weights.items()})
    proc = proc.to(dev)
    proc.precision = "bf16"
    peer = partition.PeerHalo(lh.mesh, L, dev)
    model = partition.PartitionedProcessor(proc, partition.HaloPlan(lh.mesh, dev), peer, hyper=lh)
    repl = {id(p) for p in model.replicated_parameters()}
    repl_names = [nm for nm, p in proc.named_parameters() if id(p) in repl]
    if rank == 0:
        peer_w = partition.PeerHalo(lh_whole.mesh, L, dev, group=alone)
        whole = partition.PartitionedProcessor(proc, partition.HaloPlan(lh_whole.mesh, dev, group=alone), peer_w, hyper=lh_whole)
        whole_idx = {"mesh_edges": (lh_whole.mesh.senders, lh_whole.mesh.receivers),
                     **{nm: (x_.senders, x_.receivers) for nm, x_ in lh_whole.remote.items()}}
    eids = {nm: t[0] for nm, t in local_idx.items()}
    idx = {nm: (t[1], t[2]) for nm, t in local_idx.items()}
    first = None
    for step in range(3):
        shift = 0.01 * step
        got = run(model, proc, lh.mesh.owned, eids, idx, shift, (None, model.replicated_parameters()))
        if first is None:
            first = got
        # bit-identical replicated state on every rank
        for k in ["h", "grad h"] + [f"grad {nm}" for nm in repl_names]:
            mine = got[k].contiguous()
            every = [torch.empty_like(mine) for _ in range(world)]
            dist.all_gather(every, mine)
            assert all(torch.equal(bits(t), bits(mine)) for t in every), (agg, step, k)
        if rank == 0:
            all_eids = {nm: torch.arange(s.numel()) for nm, (s, _) in sets.items()}
            ref = run(whole, proc, torch.arange(n), all_eids, whole_idx, shift, None)
            own = lh.mesh.owned.to(dev)
            sel = {"v": own, "grad v": own, **{f"e {nm}": eids[nm].to(dev) for nm in sets}, **{f"grad e {nm}": eids[nm].to(dev) for nm in sets}}
            pick = lambda d, k: d[k][sel[k]] if k in sel else d[k]
            errs = {k: rel(got[k], pick(ref, k)) for k in got}
            if agg == "max":
                for k in ["v", "h"] + [f"e {nm}" for nm in sets]:
                    assert torch.equal(bits(got[k]), bits(pick(ref, k))), (agg, step, k, errs[k])
            # forward: the same rounding points in another summation order.  Gradients: each rank rounds its share of the hyper rows'
            # gradient to bf16 before the rank-ordered sum, one more rounding point per rank than the whole graph has
            bad = {k: v_ for k, v_ in errs.items() if v_ >= (2e-2 if k.startswith("grad") else 5e-3)}
            assert not bad, (agg, step, bad)
            # the unmodified one-GPU processor
            for p in proc.parameters():
                p.grad = None
            vf = (v_full.to(dev) + shift).requires_grad_(True)
            hf = h_full.to(dev).requires_grad_(True)
            ef = {nm: t.to(dev).requires_grad_(True) for nm, t in e_full.items()}
            out = proc(MultiGraph([vf, hf], [EdgeSet(nm, ef[nm], s.to(dev), r.to(dev)) for nm, (s, r) in sets.items()]))
            oe = {es.name: es.features for es in out.edge_sets}
            ((out.node_features[0] * cv_full.to(dev)).sum() + (out.node_features[1] * ch).sum()
             + sum((t.float() ** 2).sum() for t in oe.values()) * 1e-3).backward()
            single = {"v": out.node_features[0].detach(), "h": out.node_features[1].detach(),
                      **{f"e {k}": t.detach().float() for k, t in oe.items()}, "grad v": vf.grad, "grad h": hf.grad,
                      **{f"grad e {k}": t.grad.float() for k, t in ef.items()}}
            single.update({f"grad {nm}": p.grad.clone() for nm, p in proc.named_parameters()})
            errs1 = {k: rel(got[k], pick(single, k)) for k in got}
            bad = {k: v_ for k, v_ in errs1.items() if v_ >= 2e-2}
            assert not bad, (agg, step, "vs one-GPU processor", bad)
            worst[agg] = tuple(max(p_, q_) for p_, q_ in zip(worst.get(agg, (0.0, 0.0)), (max(errs.values()), max(errs1.values()))))
            del out, vf, hf, ef, single, ref
        dist.barrier()
    again = run(model, proc, lh.mesh.owned, eids, idx, 0.0, (None, model.replicated_parameters()))
    for k in first:
        assert torch.equal(bits(again[k]), bits(first[k])), (agg, "repeat", k)
    dist.barrier()
    model.close()
    peer.close()
    if rank == 0:
        whole.close()
        peer_w.close()
    dist.barrier()
print(f"PARTITION-HYPER-GPU-OK rank {rank}/{world}: {lh.n_own} owned, {lh.mesh.n_ghost} ghosts, up segments {up_sizes}"
      + (f"; worst vs same schedule on the whole graph / vs one-GPU processor: "
         + ", ".join(f"{a} {w[0]:.2e} / {w[1]:.2e}" for a, w in worst.items()) if rank == 0 else ""), flush=True)
dist.destroy_process_group()
