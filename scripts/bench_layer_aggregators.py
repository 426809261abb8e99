"""Time one GraphNet layer (fwd + bwd, bf16, one edge set) per aggregator on the cfg5 mesh (1000 x 1000 triangulated grid: 1 000 000
nodes, 5 992 002 edges), comparing

* fused:    ops.graphnet_layer -- one autograd node per layer;
* composed: ops.edge_update + ops.segment_aggregate (the edge update's own 'sum' aggregate for 'sum') + ops.node_update -- four
            autograd nodes, the aggregate gradient expanded to [E,128] by the segment backward and added to d e' by autograd.

Both run the same forward kernels.  Each timed step is forward + backward with d v' and d e' given; CUDA events around ``--steps``
steps after ``--warmup`` steps, repeated ``--repeats`` times alternating the two paths (median reported).  The latents (1.8 GB
per layer) are larger than L2.  Prints the GPU's name and power limit, then one JSON line per aggregator.

    python scripts/bench_layer_aggregators.py [--aggregators sum,mean,max,min,pna] [--steps 10] [--warmup 3] [--repeats 3]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "hyper-graph-nets_b200"))

import torch  # noqa: E402

from hgn_b200 import ops, synthetic  # noqa: E402
from hgn_b200.plan import segment_plan  # noqa: E402

PNA_OPS = ("sum", "mean", "max", "min")


def _params(n_chunks, seed, dev):
    w = synthetic.seeded_state_dict(synthetic.mlp_shapes("m", 128 * n_chunks), seed)
    keys = [f"m.0.layers.linear_{k}.{p}" for k in range(3) for p in ("weight", "bias")] + ["m.1.weight", "m.1.bias"]
    return [w[k].to(dev).requires_grad_(True) for k in keys]


def _gpu_info(dev):
    name = torch.cuda.get_device_name(dev)
    try:
        out = subprocess.run(["nvidia-smi", f"--id={dev.index}", "--query-gpu=power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        out = "unknown"
    return name, out or "unknown"


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--aggregators", default="sum,mean,max,min,pna")
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--grid", type=int, default=1000, help="grid side (1000 = cfg5)")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_layer_aggregators.py measures on the GPU: no CUDA device visible")
    dev = torch.device("cuda", torch.cuda.current_device())
    name, power = _gpu_info(dev)
    s, r = (t.to(dev) for t in synthetic.grid_edges_two_way(args.grid, args.grid))
    n, E = args.grid * args.grid, s.numel()
    sp, rp = segment_plan(s, n), segment_plan(r, n)
    gen = torch.Generator(device=dev).manual_seed(0)
    v = torch.randn(n, 128, device=dev, generator=gen).to(torch.bfloat16).requires_grad_(True)
    e = torch.randn(E, 128, device=dev, generator=gen).to(torch.bfloat16).requires_grad_(True)
    gv = torch.randn(n, 128, device=dev, generator=gen).to(torch.bfloat16)
    ge = torch.randn(E, 128, device=dev, generator=gen).to(torch.bfloat16)
    print(json.dumps({"gpu": name, "power_limit": power, "nodes": n, "edges": E, "steps": args.steps, "warmup": args.warmup,
                      "repeats": args.repeats}), flush=True)
    for agg in args.aggregators.split(","):
        reducers = PNA_OPS if agg == "pna" else (agg,)
        pe, pn = _params(3, 11, dev), _params(1 + len(reducers), 13, dev)
        ce, cn = {}, {}

        def fused():
            return ops.graphnet_layer(pe, ce, pn, cn, v, e, sp, rp, agg)

        def composed():
            e_new, a = ops.edge_update(pe, ce, v, e, sp, rp, agg == "sum")
            aggs = [a] if agg == "sum" else ops.segment_aggregate(e_new, rp, reducers)
            return ops.node_update(pn, cn, v, aggs), e_new

        def step(path):
            for t in [v, e] + pe + pn:
                t.grad = None
            out_v, out_e = path()
            torch.autograd.backward([out_v, out_e], [gv, ge])

        def timed(path):
            for _ in range(args.warmup):
                step(path)
            torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            launches = ops.launch_count
            a.record()
            for _ in range(args.steps):
                step(path)
            b.record()
            torch.cuda.synchronize()
            return a.elapsed_time(b) / args.steps, (ops.launch_count - launches) // args.steps

        ms = {"fused": [], "composed": []}
        launches = {}
        for _ in range(args.repeats):
            for label, path in (("fused", fused), ("composed", composed)):
                t, launches[label] = timed(path)
                ms[label].append(t)
        med = {k: statistics.median(x) for k, x in ms.items()}
        print(json.dumps({"aggregator": agg, "fused_ms": round(med["fused"], 3), "composed_ms": round(med["composed"], 3),
                          "speedup": round(med["composed"] / med["fused"], 3), "fused_ms_all": [round(x, 3) for x in ms["fused"]],
                          "composed_ms_all": [round(x, 3) for x in ms["composed"]], "launches_per_layer": launches,
                          "peak_gib": round(torch.cuda.max_memory_allocated(dev) / 2 ** 30, 1)}), flush=True)
        del pe, pn, ce, cn
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
