"""A HyperGraphNet processor partitioned across the GPUs of one box (run under torch.distributed.run, one process per GPU).

Workload: a W x H triangulated grid mesh (default 1000 x 1000) in C = 16 clusters, 5 layers, bf16 forward + backward, per aggregator
(default 'sum' and 'pna').  The clusters are column bands and the parts are row slabs (``partition.block_partition``), so every cluster
straddles every rank boundary: each rank holds a long segment of every cluster, the cross-rank combine's worst case.

Per aggregator it records: ms per step (CUDA events, max over the ranks) and edge updates per second (edges of all four sets x layers);
the per-kernel times of the cross-rank exchanges and of the partial / combine kernels from a second pass with the library's per-launch
CUDA events (``HGN_TIMED`` names); the peak allocation of each rank; a partition check (rank 0 reruns one step on the whole graph with the
unmodified processor and reports relative L2); and, unless --no-single, the one-GPU processor timed on rank 0 in the same run.  With
--no-single / --no-check the whole-graph legs are skipped (a mesh that does not fit one GPU).

Appends one JSON record per run to --out (a JSON list), with the card's name and power limit.
"""
import argparse
import json
import os
import subprocess
import sys

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "hyper-graph-nets_b200"))
from hgn_b200 import _cabi, partition, synthetic  # noqa: E402
from hgn_b200.migration.meshgraphnet import MeshGraphNet  # noqa: E402
from hgn_b200.rmp.hierarchical_connector import connector_indices  # noqa: E402
from hgn_b200.util import EdgeSet, MultiGraph  # noqa: E402

EXCHANGE_KERNELS = ("halo_push", "halo_wait", "cluster_combine", "cluster_grad_sum", "cluster_mean_grad", "segment_partials",
                    "segment_partials_long", "segment_long_partial")


def _card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", str(torch.cuda.current_device())],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name()


def _processor(agg, layers, dev):
    w = synthetic.seeded_state_dict(synthetic.hyper_processor_shapes("hyper", agg, layers), seed=17)
    proc = MeshGraphNet(3, 128, 2, agg, layers, "hyper", list(synthetic.HYPER_EDGE_SETS)).processor
    proc.load_state_dict({k[len("processor."):]: t for k, t in w.items()})
    proc = proc.to(dev)
    proc.precision = "bf16"
    return proc


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--width", type=int, default=1000)
    ap.add_argument("--height", type=int, default=1000)
    ap.add_argument("--clusters", type=int, default=16)
    ap.add_argument("--layers", type=int, default=5)
    ap.add_argument("--aggregators", default="sum,pna")
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--no-single", action="store_true", help="do not time the one-GPU processor on rank 0")
    ap.add_argument("--no-check", action="store_true", help="do not rerun a step on the whole graph on rank 0")
    ap.add_argument("--out", required=True)
    args = ap.parse_args()

    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    dev = torch.device("cuda", int(os.environ["LOCAL_RANK"]))
    torch.cuda.set_device(dev)
    dist.init_process_group("nccl", device_id=dev)
    W, H, C, L = args.width, args.height, args.clusters, args.layers
    n = W * H
    col = torch.arange(n) % W
    clusters = [torch.nonzero((col * C) // W == c).flatten() for c in range(C)]
    sets = {"mesh_edges": synthetic.grid_edges_two_way(W, H), **connector_indices(clusters, [], n, fully_connect=True)}
    edges_total = sum(s.numel() for s, _ in sets.values())
    lh = partition.build_local_hyper_graph(sets, n, C, partition.block_partition(n, world), rank, world)
    local = {"mesh_edges": (lh.mesh.edge_ids, lh.mesh.senders, lh.mesh.receivers),
             **{nm: (x.edge_ids, x.senders, x.receivers) for nm, x in lh.remote.items()}}
    gen = torch.Generator().manual_seed(0)
    v_full, h_full = torch.randn(n, 128, generator=gen), torch.randn(C, 128, generator=gen)
    e_full = {nm: torch.randn(s.numel(), 128, generator=gen) for nm, (s, _) in sets.items()}
    cv_full, ch = torch.randn(n, 128, generator=gen), torch.randn(C, 128, generator=gen).to(dev)
    v0 = v_full[lh.mesh.owned].to(dev).to(torch.bfloat16)
    e0 = {nm: e_full[nm][local[nm][0]].to(dev).to(torch.bfloat16) for nm in sets}
    idx = {nm: (local[nm][1].to(dev), local[nm][2].to(dev)) for nm in sets}
    cv, h0 = cv_full[lh.mesh.owned].to(dev), h_full.to(dev)
    card = _card()
    records = []

    def timed(fn, steps):
        dist.barrier()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(steps):
            fn()
        b.record()
        torch.cuda.synchronize()
        ms = torch.tensor([a.elapsed_time(b) / steps], device=dev)
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms)

    for agg in args.aggregators.split(","):
        proc = _processor(agg, L, dev)
        peer = partition.PeerHalo(lh.mesh, L, dev)
        model = partition.PartitionedProcessor(proc, partition.HaloPlan(lh.mesh, dev), peer, hyper=lh)
        repl = model.replicated_parameters()
        kept = {}

        def step(keep=False):
            for p in proc.parameters():
                p.grad = None
            v = v0.detach().requires_grad_(True)
            h = h0.detach().requires_grad_(True)
            e = {nm: t.detach().requires_grad_(True) for nm, t in e0.items()}
            ov, oes, oh = model(v, [EdgeSet(nm, e[nm], *idx[nm]) for nm in sets], h)
            loss = (ov * cv).sum() + (oh * ch).sum() + sum(es.features.float().sum() for es in oes) * 1e-3
            loss.backward()
            partition.allreduce_gradients(proc, exclude=repl)
            if keep:
                kept.update(v=ov.detach(), h=oh.detach(), grad_v=v.grad, grads=[p.grad.clone() for p in proc.parameters()])

        for _ in range(args.warmup):
            step()
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats(dev)
        ms = timed(step, args.steps)
        peak = torch.tensor([torch.cuda.max_memory_allocated(dev) / 2**30], device=dev)
        peaks = [torch.zeros_like(peak) for _ in range(world)]
        dist.all_gather(peaks, peak)
        _cabi.profile(True)
        timed(step, args.steps)
        kernels = _cabi.profile_report()
        _cabi.profile(False)
        ex = {k["name"]: round(k["ms"] / args.steps, 4) for k in kernels if k["name"] in EXCHANGE_KERNELS}
        step(keep=True)
        torch.cuda.synchronize()
        model.close()
        peer.close()
        dist.barrier()
        rec = {"aggregator": agg, "n_gpus": world, "nodes": n, "clusters": C, "layers": L, "edges": edges_total,
               "ms_per_step": ms, "edge_updates_per_s": edges_total * L / (ms * 1e-3),
               "peak_gib_per_rank": [round(float(p), 2) for p in peaks], "exchange_kernels_ms_per_step_rank0": ex,
               "kernels_ms_per_step_rank0": {k["name"]: round(k["ms"] / args.steps, 4) for k in kernels}}
        if rank == 0 and not (args.no_single and args.no_check):
            del model, peer
            torch.cuda.empty_cache()
            vf = v_full.to(dev).requires_grad_(True)
            hf = h_full.to(dev).requires_grad_(True)
            ef = {nm: t.to(dev).requires_grad_(True) for nm, t in e_full.items()}
            full_sets = [EdgeSet(nm, ef[nm], s.to(dev), r.to(dev)) for nm, (s, r) in sets.items()]

            def single(keep=False):
                for p in proc.parameters():
                    p.grad = None
                out = proc(MultiGraph([vf, hf], list(full_sets)))
                ((out.node_features[0] * cv_full.to(dev)).sum() + (out.node_features[1] * ch).sum()
                 + sum(es.features.float().sum() for es in out.edge_sets) * 1e-3).backward()
                if keep:
                    return out
            if not args.no_check:
                vf.grad = hf.grad = None
                out = single(keep=True)
                own = lh.mesh.owned.to(dev)
                rel = lambda a, b: float((a.double() - b.double()).norm() / b.double().norm().clamp_min(1e-30))
                check = {"latents_owned_rows": rel(kept["v"], out.node_features[0].detach()[own]),
                         "hyper_rows": rel(kept["h"], out.node_features[1].detach()),
                         "latent_gradients_owned_rows": rel(kept["grad_v"], vf.grad[own]),
                         "weight_gradients_worst": max(rel(a, p.grad) for a, p in zip(kept["grads"], proc.parameters())),
                         "metric": "relative L2, partitioned vs the unmodified bf16 processor on the whole graph on one GPU"}
                rec["partition_check"] = check
                del out
            if not args.no_single:
                for _ in range(args.warmup):
                    single()
                torch.cuda.synchronize()
                torch.cuda.reset_peak_memory_stats(dev)
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                for _ in range(args.steps):
                    single()
                b.record()
                torch.cuda.synchronize()
                one = a.elapsed_time(b) / args.steps
                rec["one_gpu_processor"] = {"ms_per_step": one, "edge_updates_per_s": edges_total * L / (one * 1e-3),
                                            "peak_gib": round(torch.cuda.max_memory_allocated(dev) / 2**30, 2)}
                rec["speedup_vs_one_gpu"] = one / ms
            del vf, hf, ef, full_sets
            torch.cuda.empty_cache()
        dist.barrier()
        records.append(rec)
        del proc
        torch.cuda.empty_cache()
    if rank == 0:
        run = {"card": card, "world": world, "workload": f"{W} x {H} grid, {C} column-band clusters vs {world} row slabs, {L} HyperGraphNet "
               "layers, bf16 forward + backward", "steps": args.steps, "warmup": args.warmup, "records": records}
        print(json.dumps(run))
        old = json.load(open(args.out)) if os.path.exists(args.out) else []
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(old + [run], f, indent=1)
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
