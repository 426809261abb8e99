"""Encoder / decoder MLPs on one GPU: torch (fp32 Linear / ReLU / LayerNorm, then the conversion the bf16 processor does) against the
bf16 tcgen05 kernels (hgn_b200.ops.encoder_mlp / decoder_mlp), and the whole bf16 MeshGraphNet training step with the switch off
and on, at the cfg5 shape: 1 000 000 mesh nodes (K = 5 raw features), 5 992 002 mesh edges (K = 7), 3 outputs, 15 'sum' layers.

    python scripts/bench_io_mlp.py [--steps 20] [--warmup 5] [--out profiles/io_mlp_b200.json]

Timing: CUDA events around each arm's forward + backward, the two arms alternated call by call inside one process after every shape
was warmed up; inputs are larger than the 126 MB L2 (the raw edge features alone are 168 MB, a latent tensor 1.5-3 GB).  Peak memory
is torch.cuda.max_memory_allocated over one step after a reset.  The card's name and power limit are printed with the numbers.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "hyper-graph-nets_b200"))

N_NODES, N_EDGES, K_NODE, K_EDGE, N_OUT, LAYERS = 1_000_000, 5_992_002, 5, 7, 3, 15


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clock = [s.strip() for s in q.split(",")]
        return {"name": name, "power_limit": power, "sm_max_clock": clock}
    except Exception as exc:                      # the numbers stay valid; say that the card could not be read
        return {"name": torch.cuda.get_device_name(), "power_limit": f"unreadable ({type(exc).__name__})"}


def timed(fn, steps):
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for _ in range(steps):
        fn()
    stop.record()
    torch.cuda.synchronize()
    return start.elapsed_time(stop) / steps


def alternate(arms, steps, warmup, rounds=4):
    """ms per call of each arm: warm-up of every arm, then `rounds` alternating windows of steps / rounds calls each (median window)."""
    for fn in arms.values():
        for _ in range(warmup):
            fn()
    torch.cuda.synchronize()
    per = max(1, steps // rounds)
    samples = {k: [] for k in arms}
    for _ in range(rounds):
        for k, fn in arms.items():
            samples[k].append(timed(fn, per))
    return {k: {"ms": sorted(v)[len(v) // 2], "windows_ms": [round(x, 3) for x in v]} for k, v in samples.items()}


def mlp_bench(steps, warmup):
    from hgn_b200 import ops
    from hgn_b200.migration.decoder import _decoder_parameters
    from hgn_b200.migration.graphnet import _mlp_parameters
    from hgn_b200.migration.meshgraphnet import MeshGraphNet
    dev = torch.device("cuda")
    torch.manual_seed(0)
    shell = MeshGraphNet(N_OUT, 128, 2, "sum", 1, "none", ["mesh_edges"]).to(dev)
    out = {}
    for what, rows, k in (("node encoder", N_NODES, K_NODE), ("edge encoder", N_EDGES, K_EDGE)):
        model = shell.encoder.node_model if what == "node encoder" else shell.encoder.edge_models["mesh_edges"]
        x = torch.randn(rows, k, device=dev)
        params = _mlp_parameters(model, k, x)
        gup = torch.randn(rows, 128, device=dev).to(torch.bfloat16)
        cache = {}

        def torch_arm():
            y = model(x).to(torch.bfloat16)          # Processor.forward converts the fp32 latents on entry
            y.backward(gup)

        def kernel_arm():
            ops.encoder_mlp(params, cache, x).backward(gup)

        res = alternate({"torch": torch_arm, "kernels": kernel_arm}, steps, warmup)
        res["shape"] = f"[{rows}, {k}] fp32 -> [{rows}, 128] bf16, forward + backward (no raw-feature gradient)"
        out[what] = res
    x = torch.randn(N_NODES, 128, device=dev).to(torch.bfloat16).requires_grad_(True)
    model = shell.decoder.model
    params = _decoder_parameters(model, x)
    gup = torch.randn(N_NODES, N_OUT, device=dev)
    cache = {}

    def torch_dec():
        model(x.to(torch.float32)).backward(gup)     # Processor.forward returns the node latents in the encoder's dtype (fp32)

    def kernel_dec():
        ops.decoder_mlp(params, cache, x).backward(gup)

    res = alternate({"torch": torch_dec, "kernels": kernel_dec}, steps, warmup)
    res["shape"] = f"[{N_NODES}, 128] bf16 -> [{N_NODES}, {N_OUT}] fp32, forward + backward (input gradient included)"
    out["decoder"] = res
    return out


def model_bench(steps, warmup):
    """One bf16 MeshGraphNet training step at cfg5 (encoder, 15 'sum' layers, decoder, loss, backward), switch off vs on."""
    import hgn_b200
    from hgn_b200 import synthetic, util
    from hgn_b200.migration.meshgraphnet import MeshGraphNet
    dev = torch.device("cuda")
    hgn_b200.set_precision("bf16")
    s, r = synthetic.grid_edges_two_way(1000, 1000)
    assert s.numel() == N_EDGES
    gen = torch.Generator().manual_seed(1)
    nf = torch.randn(N_NODES, K_NODE, generator=gen).to(dev)
    ef = torch.randn(N_EDGES, K_EDGE, generator=gen).to(dev)
    s, r = s.to(dev), r.to(dev)
    coef = torch.randn(N_NODES, N_OUT, generator=gen).to(dev)
    torch.manual_seed(0)
    m = MeshGraphNet(N_OUT, 128, 2, "sum", LAYERS, "none", ["mesh_edges"]).to(dev)

    def step():
        g = util.MultiGraph([nf], [util.EdgeSet("mesh_edges", ef, s, r)])
        loss = (m(g) * coef).sum()
        loss.backward()
        return loss

    arms, peaks = {}, {}
    for on in (False, True):
        def arm(on=on):
            hgn_b200.set_io_kernels(on)
            step()
        arms["kernels" if on else "torch"] = arm
    res = alternate(arms, steps, warmup, rounds=2)
    for name, fn in arms.items():
        for p in m.parameters():
            p.grad = None
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats()
        base = torch.cuda.memory_allocated()
        fn()
        torch.cuda.synchronize()
        peaks[name] = {"peak_allocated_GB": round(torch.cuda.max_memory_allocated() / 1e9, 3), "resident_before_step_GB": round(base / 1e9, 3)}
    hgn_b200.set_io_kernels(False)
    # the two arms' losses on the same weights (the kernels round at other points: same to bf16 accuracy)
    with torch.no_grad():
        g = util.MultiGraph([nf], [util.EdgeSet("mesh_edges", ef, s, r)])
        hgn_b200.set_io_kernels(False)
        l_off = float((m(g) * coef).sum())
        hgn_b200.set_io_kernels(True)
        l_on = float((m(g) * coef).sum())
        hgn_b200.set_io_kernels(False)
    for name in res:
        res[name].update(peaks[name])
    res["loss_torch_vs_kernels_relative"] = abs(l_on - l_off) / max(abs(l_off), 1e-30)
    res["shape"] = f"MeshGraphNet bf16, {N_NODES} nodes (K={K_NODE}), {N_EDGES} edges (K={K_EDGE}), {LAYERS} 'sum' layers, n_out={N_OUT}: forward + loss + backward"
    return res


def flag_bench():
    """bench.py's flag-shape FlagModel legs (graphed rollout and training iteration) with the switch on; needs the reference tree."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import reference_shim
    if not reference_shim.available():
        return {"value": None, "note": "not measured: no reference tree (FlagModel) on this machine"}
    import hgn_b200
    sys.path.insert(0, ROOT)
    import bench
    hgn_b200.set_io_kernels(True)
    try:
        return bench.rollout_bench(torch.device("cuda"))
    finally:
        hgn_b200.set_io_kernels(False)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_io_mlp.py measures the GPU: no CUDA device")
    t0 = time.time()
    res = {"card": card(), "torch": torch.__version__}
    res["mlps"] = mlp_bench(args.steps, args.warmup)
    torch.cuda.empty_cache()
    res["meshgraphnet_cfg5_step"] = model_bench(max(2, args.steps // 4), 2)
    torch.cuda.empty_cache()
    res["flag_with_io_kernels"] = flag_bench()
    res["wall_s"] = round(time.time() - t0, 1)
    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
