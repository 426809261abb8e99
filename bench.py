#!/usr/bin/env python
"""Headline benchmark: edge-updates/sec per message-passing layer (forward + backward).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

Workload (BASELINE.json configs[4], SURVEY.md s8 cfg 5): synthetic 1000 x 1000 triangulated grid,
N = 1 000 000 nodes, E = 5 992 002 directed mesh edges, latent 128, 15 unshared GraphNet layers, `sum`
aggregator, processor only (latents in, latents out), bf16 tcgen05 mode.  One step = Processor.forward
+ backward of a seeded linear loss w.r.t. all latents and weights.

value   : E * L / t with the inputs resident in HBM (CUDA events, max over ranks)
e2e     : the same through the public module API with pinned HOST inputs: H2D copy of the fp32 latents,
          forward + backward, D2H read of the loss, all inside the timed region
roofline: the dominant kernel's algorithmic FLOPs per launch / its mean launch time (CUDA events recorded
          inside the library around every launch during the timed region) against MEASURED_PEAKS.json
cpu_baseline / --impl reference: the oracle port of the reference's torch path (oracle/hgn_oracle.py)
          on the host cores, on a bounded sub-mesh of the same workload.
With --gpus N > 1 (torchrun) the mesh is edge-cut partitioned into N row slabs with a halo exchange of
boundary node latents per layer (strong scaling: the total mesh is fixed).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(ROOT, "hyper-graph-nets_b200"))

# The reference arm runs the UNMODIFIED reference on the host cores.  Its modules capture `src.util.device` at import time
# (src/util.py:9: cuda when available), so that arm must not see a GPU: hide them before torch is imported.
_REFERENCE_ARM = any(a == "reference" and i > 0 and sys.argv[i - 1] == "--impl" for i, a in enumerate(sys.argv)) or "--impl=reference" in sys.argv
if _REFERENCE_ARM:
    os.environ["CUDA_VISIBLE_DEVICES"] = ""
    os.environ.setdefault("WANDB_MODE", "disabled")

import torch  # noqa: E402

GRID_W, GRID_H = 1000, 1000
LAYERS = 15
# --workload: the headline (cfg5) plus the small-mesh training shapes of BASELINE.json configs[1] and [3] (SURVEY.md s8 cfg 2 / cfg 4:
# a batch of B disjoint trajectories' meshes per step, src/algorithms/MeshSimulator.py:158-234).  Only cfg5 is the bench line the
# driver reads; the others are reported under profiles/.
#            name: (grid w, grid h, batch, layers, aggregator, CPU sample (w, h, batch, layers), description)
WORKLOADS = {
    "cfg5": (1000, 1000, 1, 15, "sum", (1000, 125, 1, 1), "cfg5: 1M-node / 5 992 002-edge triangulated mesh"),
    "cfg2": (40, 40, 21, 15, "pna", (40, 40, 21, 15), "cfg2: flag_simple-shaped cloth (40x40 grid, 1 600 nodes / 9 282 edges) x batch 21"),
    "cfg4": (48, 40, 21, 5, "pna", (48, 40, 21, 5), "cfg4: cylinder_flow-shaped 2-D mesh (48x40 grid, 1 920 nodes / 11 158 edges) x batch 21, one rank's share"),
}
LATENT = 128
METRIC = "edge-updates/sec per MP layer (fwd+bwd)"
UNIT = "edge-updates/s"
F_EDGE = 10 * LATENT * LATENT           # GEMM flops per edge, forward (SURVEY.md s8d)
F_NODE_SUM = 2 * (2 + 2) * LATENT * LATENT


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return {"hbm_gbs": p["hbm_gbs"], "bf16_tflops": p["bf16_tflops"], "bf16_tflops_sustained": p["bf16_tflops_sustained"],
                "source": "measured (MEASURED_PEAKS.json)"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback (B200_PROFILING.md)"}


class ClockSampler:
    """SM clock and clock-event (throttle) reasons of one GPU sampled while the timed region runs: through NVML inside this process
    every 20 ms (a timed region of a few hundred ms at N = 8 is over before an `nvidia-smi -lms` child has printed its first line),
    falling back to an `nvidia-smi -lms 200` child where the NVML bindings are missing."""

    FIELDS = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    NVML_REASONS = ((0x8, "hw_slowdown"), (0x40, "hw_thermal_slowdown"), (0x20, "sw_thermal_slowdown"), (0x4, "sw_power_cap"))

    def __init__(self, index: int):
        self.index, self.rows, self.proc, self.thread = index, [], None, None
        self.nvml, self.handle, self.stop = None, None, threading.Event()

    def _nvml_handle(self):
        import pynvml
        pynvml.nvmlInit()
        try:
            uuid = str(torch.cuda.get_device_properties(self.index).uuid)
            uuid = uuid if uuid.startswith("GPU-") else "GPU-" + uuid
            handle = pynvml.nvmlDeviceGetHandleByUUID(uuid.encode() if hasattr(uuid, "encode") else uuid)
        except Exception:
            handle = pynvml.nvmlDeviceGetHandleByIndex(self.index)      # no CUDA_VISIBLE_DEVICES remapping: same numbering
        return pynvml, handle

    def _sample_nvml(self):
        nv, h = self.nvml, self.handle
        try:
            sm = float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM))
            mx = float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))
            try:
                mask = int(nv.nvmlDeviceGetCurrentClocksEventReasons(h))
            except Exception:
                mask = int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(h))
            self.rows.append([sm, mx] + ["Active" if mask & bit else "Not Active" for bit, _ in self.NVML_REASONS])
        except Exception:
            pass

    def _loop_nvml(self):
        while not self.stop.is_set():
            self._sample_nvml()
            self.stop.wait(0.02)

    def __enter__(self):
        try:
            self.nvml, self.handle = self._nvml_handle()
            self.thread = threading.Thread(target=self._loop_nvml, daemon=True)
            self.thread.start()
            return self
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.FIELDS}",
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def __exit__(self, *exc):
        if self.nvml is not None:
            self._sample_nvml()                                  # one more at the end of the region (the GPU is still busy or just done)
            self.stop.set()
            self.thread.join(timeout=2)
            return
        if self.proc is not None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except subprocess.TimeoutExpired:
                self.proc.kill()

    def summary(self):
        sm, mx, reasons = [], [], set()
        names = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")
        for row in self.rows:
            try:
                sm.append(float(row[0])); mx.append(float(row[1]))
            except (ValueError, IndexError):
                continue
            for name, val in zip(names, row[2:6]):
                if str(val).lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm),
                "via": "nvml" if self.nvml is not None else "nvidia-smi"}


# ------------------------------------------------------------------------------------------------------
# workload
# ------------------------------------------------------------------------------------------------------
def build_inputs(width, height, layers, seed=0, aggregator="sum", batch=1):
    """Host-side (pinned) latents, int64 edge lists and the seeded processor weights.  `batch` > 1: that many disjoint copies of the
    mesh in one index space, graph i's nodes offset by i * N (MeshSimulator._get_batched, src/algorithms/MeshSimulator.py:196-217)."""
    from hgn_b200 import synthetic
    senders, receivers = synthetic.grid_edges_two_way(width, height)
    if batch > 1:
        offs = (torch.arange(batch, dtype=senders.dtype) * (width * height)).repeat_interleave(senders.numel())
        senders, receivers = senders.repeat(batch) + offs, receivers.repeat(batch) + offs
    n, e = width * height * batch, senders.numel()
    gen = torch.Generator().manual_seed(seed)
    v0 = torch.randn(n, LATENT, generator=gen)
    e0 = torch.randn(e, LATENT, generator=gen)
    coef_v = torch.randn(n, LATENT, generator=gen)
    weights = synthetic.seeded_state_dict(synthetic.processor_shapes(layers, ["mesh_edges"], aggregator), seed=17)
    return {"senders": senders, "receivers": receivers, "v0": v0, "e0": e0, "coef_v": coef_v, "weights": weights, "n": n, "e": e}


def make_processor(weights, layers, precision, device, aggregator="sum"):
    from hgn_b200.migration.meshgraphnet import MeshGraphNet
    shell = MeshGraphNet(3, LATENT, 2, aggregator, layers, "none", ["mesh_edges"])
    proc = shell.processor
    proc.load_state_dict({k[len("processor."):]: t for k, t in weights.items()})
    proc = proc.to(device)
    proc.precision = precision
    return proc


DUMP_ROWS = 16384                        # rows kept per latent / latent-gradient array by --dump-outputs
DUMP_SEED = 7
DUMP_BYTES_MAX = 64 << 20


def dump_rows(n):
    """The fixed sample of `n` rows that --dump-outputs keeps: all of them up to DUMP_ROWS, else DUMP_ROWS seeded rows in order."""
    if n <= DUMP_ROWS:
        return torch.arange(n)
    return torch.randperm(n, generator=torch.Generator().manual_seed(DUMP_SEED))[:DUMP_ROWS].sort().values


def dump_outputs(out_dir, loss, out, v, ed, named_params):
    """--dump-outputs: what one step hands its caller, as float32 ``<out_dir>/<name>.npy`` -- the loss, the output node and edge
    latents and the gradients of the input latents (each on the fixed row sample of `dump_rows`), and every parameter gradient in
    full (``grad.<parameter name>.npy``).  The inputs are seeded, so two builds run with the same arguments can be compared array by
    array."""
    import numpy as np
    arrays = {"loss": loss.detach().reshape(())}
    for name, t in (("node_latents", out.node_features[0]), ("edge_latents", out.edge_sets[0].features),
                    ("node_latents_grad", v.grad), ("edge_latents_grad", ed.grad)):
        arrays[name] = t.detach()[dump_rows(t.shape[0]).to(t.device)]
    for name, p in named_params:
        if p.grad is not None:
            arrays["grad." + name] = p.grad.detach()
    total = sum(t.numel() * 4 for t in arrays.values())
    if total > DUMP_BYTES_MAX:
        raise SystemExit(f"--dump-outputs: {total} bytes exceed the {DUMP_BYTES_MAX}-byte limit")
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.float().cpu().numpy())


def fp32_parity_mode(dev):
    """The 1e-5 parity mode (`precision = "fp32"`: fp32 storage, FFMA kernels) beside the bf16 headline, against an fp32 denominator
    measured here the way MEASURED_PEAKS.json measures bf16 (SURVEY.md s8d): torch.matmul fp32 8192^3 with TF32 off, best of 10 and a
    1.5 s back-to-back loop; then the processor on a 1000 x 250 slab of the cfg5 mesh, 3 layers, fwd+bwd.  Not a roofline target."""
    from hgn_b200.util import EdgeSet, MultiGraph
    tf32 = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        a = torch.randn(8192, 8192, device=dev); b = torch.randn(8192, 8192, device=dev)
        for _ in range(3):
            a @ b
        torch.cuda.synchronize()
        best = 0.0
        for _ in range(10):
            t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0.record(); a @ b; t1.record(); torch.cuda.synchronize()
            best = max(best, 2 * 8192 ** 3 / (t0.elapsed_time(t1) * 1e-3) / 1e12)
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        reps, wall = 0, time.perf_counter()
        t0.record()
        while time.perf_counter() - wall < 1.5:
            for _ in range(10):
                a @ b
            reps += 10
            torch.cuda.synchronize()
        t1.record(); torch.cuda.synchronize()
        sustained = reps * 2 * 8192 ** 3 / (t0.elapsed_time(t1) * 1e-3) / 1e12
        del a, b
    finally:
        torch.backends.cuda.matmul.allow_tf32 = tf32
    W, H, L = 1000, 250, 3
    data = build_inputs(W, H, L)
    proc = make_processor(data["weights"], L, "fp32", dev)
    params = list(proc.parameters())
    s_, r_ = data["senders"].to(dev), data["receivers"].to(dev)
    v0, e0, coef = data["v0"].to(dev), data["e0"].to(dev), data["coef_v"].to(dev)

    def step():
        for p in params:
            p.grad = None
        v, ed = v0.detach().requires_grad_(True), e0.detach().requires_grad_(True)
        out = proc(MultiGraph([v], [EdgeSet("mesh_edges", ed, s_, r_)]))
        ((out.node_features[0] * coef).sum() + out.edge_sets[0].features.sum() * 1e-3).backward()

    for _ in range(2):
        step()
    torch.cuda.synchronize()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(3):
        step()
    t1.record(); torch.cuda.synchronize()
    ms = t0.elapsed_time(t1) / 3
    flops = 3 * (data["e"] * F_EDGE + data["n"] * F_NODE_SUM) * L
    return {"edge_updates_per_s": data["e"] * L / (ms * 1e-3), "ms_per_step": ms, "algorithmic_tflops": flops / (ms * 1e-3) / 1e12,
            "fp32_matmul_tflops_sustained": sustained, "fp32_matmul_tflops_best": best, "frac": flops / (ms * 1e-3) / 1e12 / sustained,
            "mesh": f"{W}x{H} slab of the cfg5 mesh ({data['n']} nodes, {data['e']} directed edges), {L} layers, sum, fwd+bwd",
            "what": "precision = 'fp32': the 1e-5 parity mode (FFMA kernels), not a roofline target; peak = torch.matmul fp32, TF32 off, measured in this run"}


def data_parallel_cfg4_leg(world, rank, dev, steps=20):
    """BASELINE.json configs[3] beside the partitioned cfg5 line of an N > 1 run: cylinder_flow-shaped batches (48x40 mesh x 21,
    GraphNet pna, 5 layers, bf16), every rank a replica with its own batch (seed = rank), one flat fp32 gradient all-reduce per step
    (partition.allreduce_gradients) -- trajectory data parallelism, weak scaling.  Returns the JSON sub-object (rank 0) or None."""
    import torch.distributed as dist
    from hgn_b200 import partition
    from hgn_b200.util import EdgeSet, MultiGraph
    gw, gh, batch, layers, agg, _, wl_text = WORKLOADS["cfg4"]
    data = build_inputs(gw, gh, layers, seed=rank, aggregator=agg, batch=batch)
    proc = make_processor(data["weights"], layers, "bf16", dev, agg)
    params = list(proc.parameters())
    senders, receivers = data["senders"].to(dev), data["receivers"].to(dev)
    v_dev, e_dev, coef = data["v0"].to(dev).to(torch.bfloat16), data["e0"].to(dev).to(torch.bfloat16), data["coef_v"].to(dev)

    def step():
        for p in params:
            p.grad = None
        v, ed = v_dev.detach().requires_grad_(True), e_dev.detach().requires_grad_(True)
        out = proc(MultiGraph([v], [EdgeSet("mesh_edges", ed, senders, receivers)]))
        ((out.node_features[0] * coef).sum() + out.edge_sets[0].features.sum() * 1e-3).backward()
        partition.allreduce_gradients(proc)

    for _ in range(5):
        step()
    dist.barrier()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(steps):
        step()
    b.record()
    dist.barrier()
    torch.cuda.synchronize()
    ms = torch.tensor([a.elapsed_time(b) / steps], device=dev)
    dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    if rank != 0:
        return None
    ms = float(ms)
    return {"value": data["e"] * layers * world / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms, "steps": steps, "scaling": "weak",
            "workload": f"{wl_text}, {layers} GraphNet layers, {agg}, processor fwd+bwd + gradient all-reduce; one batch per rank",
            "edges_per_rank": data["e"]}


def run_ours(args):
    from hgn_b200 import _cabi, ops, partition
    from hgn_b200.util import EdgeSet, MultiGraph
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.dump_outputs and world > 1:
        raise SystemExit("--dump-outputs: single-GPU runs only")
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1 and args.workload == "cfg5":
        from hgn_b200 import partition
        args.aggregator = args.aggregator or "sum"
        return partition.bench_partitioned(args, world, rank, dev, GRID_W, GRID_H, LAYERS, METRIC, UNIT, load_peaks(), ClockSampler,
                                           dominant_kernel_roofline, extra_leg=data_parallel_cfg4_leg)

    gw, gh, batch, layers, default_agg, cpu_sample, wl_text = WORKLOADS[args.workload]
    args.aggregator = args.aggregator or default_agg
    # world > 1 with a small-mesh workload: trajectory data parallelism (BASELINE.json configs[3], SURVEY.md s8e) -- every rank a
    # replica with its own batch (seed = rank), one flat fp32 gradient all-reduce per step, weak scaling
    data = build_inputs(gw, gh, layers, seed=rank, aggregator=args.aggregator, batch=batch)
    n, e = data["n"], data["e"]
    f_node = 2 * ((1 + (4 if args.aggregator == "pna" else 1)) + 2) * LATENT * LATENT
    proc = make_processor(data["weights"], layers, "bf16", dev, args.aggregator)
    params = [p for p in proc.parameters()]
    senders, receivers = data["senders"].to(dev), data["receivers"].to(dev)
    v0_host, e0_host = data["v0"].pin_memory(), data["e0"].pin_memory()
    coef_v = data["coef_v"].to(dev)
    # resident inputs: the latents as they sit in HBM between two processor calls of a bf16 pipeline, i.e. in the dtype the path
    # computes in (no per-step fp32 -> bf16 pass); the end-to-end leg below starts from fp32 HOST buffers and pays for the conversion
    v_dev = v0_host.to(dev).to(torch.bfloat16)
    e_dev = e0_host.to(dev).to(torch.bfloat16)
    loss_host = torch.empty(1, dtype=torch.float32).pin_memory()

    def step(v_in, e_in, keep=None):
        for p in params:
            p.grad = None
        v = v_in.requires_grad_(True)
        ed = e_in.requires_grad_(True)
        out = proc(MultiGraph([v], [EdgeSet("mesh_edges", ed, senders, receivers)]))
        loss = (out.node_features[0] * coef_v).sum() + out.edge_sets[0].features.sum() * 1e-3
        loss.backward()
        if world > 1:
            partition.allreduce_gradients(proc)
        if keep is not None:                    # the step whose results --dump-outputs writes
            keep.update(loss=loss, out=out, v=v, ed=ed)
        return loss

    def max_over_ranks(ms):
        if world == 1:
            return ms
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t)

    def fence():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def step_resident(keep=None):
        return step(v_dev.detach(), e_dev.detach(), keep)

    copy_stream = torch.cuda.Stream(device=dev)

    def upload():
        """H2D copy of one step's fp32 inputs from pinned host memory on the copy stream (an input pipeline's prefetch)."""
        with torch.cuda.stream(copy_stream):
            v = v0_host.to(dev, non_blocking=True)
            ed = e0_host.to(dev, non_blocking=True)
            ready = torch.cuda.Event()
            ready.record(copy_stream)
        return v, ed, ready

    def run_e2e(steps):
        """`steps` end-to-end steps: every step's inputs cross PCIe inside the region (step i+1's copy overlaps step i's
        compute, the way a training loop prefetches its next batch) and every step's loss is read back to the host."""
        nxt = upload()
        for i in range(steps):
            v, ed, ready = nxt
            if i + 1 < steps:
                nxt = upload()
            torch.cuda.current_stream().wait_event(ready)
            v.record_stream(torch.cuda.current_stream()); ed.record_stream(torch.cuda.current_stream())
            loss = step(v, ed)
            loss_host.copy_(loss.detach().reshape(1), non_blocking=True)
            torch.cuda.current_stream().synchronize()

    for _ in range(max(args.warmup, 3)):
        step_resident()
    fence()

    # ---- timed region: inputs resident in HBM --------------------------------------------------------
    _cabi.profile(True)
    launches0 = ops.launch_count
    last = {} if args.dump_outputs else None
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local_rank) as clocks:
        fence()
        start.record()
        for i in range(args.steps):
            step_resident(last if i == args.steps - 1 else None)
        stop.record()
        fence()
    ms_per_step = max_over_ranks(start.elapsed_time(stop) / args.steps)
    launches = ops.launch_count - launches0
    kernels = _cabi.profile_report()
    _cabi.profile(False)
    value = e * layers * world / (ms_per_step * 1e-3)
    if last is not None:
        dump_outputs(args.dump_outputs, last["loss"], last["out"], last["v"], last["ed"], proc.named_parameters())
        del last

    # ---- end to end: pinned host inputs -> H2D -> fwd+bwd -> D2H loss ---------------------------------
    run_e2e(3)                                  # warm-up: two input sets are alive at a time, let the allocator cache both
    fence()
    # --steps steps, every one of them with its own H2D copy and loss read-back inside the region; the first step's copy has nothing
    # to hide behind (65 ms of PCIe time at cfg5), so its share of the quote shrinks as --steps grows
    e2e_steps = args.steps
    t0 = torch.cuda.Event(enable_timing=True); t1 = torch.cuda.Event(enable_timing=True)
    t0.record()                                 # on the compute stream, which waits for every copy it consumes
    run_e2e(e2e_steps)
    t1.record()
    fence()
    e2e_ms = max_over_ranks(t0.elapsed_time(t1) / e2e_steps)
    e2e_value = e * layers * world / (e2e_ms * 1e-3)

    # ---- small meshes: the same resident step (forward + backward) captured in ONE CUDA graph -------------
    graphed = None
    if args.workload != "cfg5" and world == 1:
        graphed = graphed_step(step_resident, params, args.steps, e * layers)

    # ---- roofline of the dominant kernel ----------------------------------------------------------------
    peaks = load_peaks()
    roofline = dominant_kernel_roofline(kernels, args.steps, e, n, peaks)

    # ---- CPU baseline: oracle port on a bounded sub-mesh ------------------------------------------------
    cpu = (cpu_baseline(steps=1, sample=cpu_sample, aggregator=args.aggregator, workload=args.workload)
           if world == 1 and not os.environ.get("HGN_BENCH_NO_CPU") else None)
    if rank != 0:
        dist.barrier()
        return

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak" if world > 1 else "strong", "vs_baseline": None,
        "dtype": "bf16", "data": f"synthetic (seeded {gw}x{gh} triangulated grid" + (f" x {batch}" if batch > 1 else "") + ", seeded weights)",
        "config": {"workload": f"{wl_text}, {layers} GraphNet layers, {args.aggregator} aggregator, "
                               "processor fwd+bwd", "nodes": n, "edges": e, "layers": layers, "latent": LATENT,
                   "l2_policy": ("inputs larger than L2 (1.8 GB of bf16 latents per layer)" if args.workload == "cfg5" else
                                 "small mesh: the whole step's working set is L2-resident by construction (launch-bound shape)"),
                   "partitioning": "none", "backward": "recompute",
                   "resident_inputs": "bf16 latents in HBM (value); e2e: fp32 pinned host buffers, converted on the device",
                   "parallelism": (f"dp{world}: one replica and one batch (seed = rank) per GPU, one flat fp32 gradient all-reduce (NCCL) per "
                                   "step; value = all ranks' edge updates / max-over-ranks time") if world > 1 else "single GPU"},
        "e2e": {"value": e2e_value, "unit": UNIT, "ms_per_step": e2e_ms, "steps": e2e_steps,
                "pipeline": "H2D of step i+1 on a copy stream overlaps step i (the first copy of the region is exposed); loss D2H + stream sync every step",
                "h2d_bytes_per_step": int(v0_host.numel() * 4 + e0_host.numel() * 4) * world, "d2h_bytes_per_step": 4 * world},
        "gpu_launches": launches,
        "clocks": clocks.summary(),
        "roofline": roofline,
        "layer_roofline": {"tensor_ms_per_layer": 3 * (e * F_EDGE + n * f_node) / (load_peaks()["bf16_tflops_sustained"] * 1e12) * 1e3,
                           "measured_ms_per_layer": ms_per_step / layers,
                           "frac": 3 * (e * F_EDGE + n * f_node) / (load_peaks()["bf16_tflops_sustained"] * 1e12) * 1e3 / (ms_per_step / layers)},
        "kernels": [{"name": k["name"], "launches": k["launches"], "ms_per_step": k["ms"] / args.steps} for k in kernels],
        "cpu_baseline": cpu,
    }
    if graphed is not None:
        line["cuda_graph"] = graphed
    if args.workload == "cfg5" and args.aggregator == "sum" and not os.environ.get("HGN_BENCH_NO_ROLLOUT"):
        line["rollout"] = rollout_bench(dev)         # the metric's second half, BASELINE.json configs[1]
    if world == 1 and not os.environ.get("HGN_BENCH_NO_TORCH_REFERENCE"):
        del proc, params, v_dev, e_dev
        torch.cuda.empty_cache()
        line["torch_cuda_reference"] = torch_cuda_reference(dev, data, args.aggregator, layers if args.workload != "cfg5" else 1)
        if args.workload == "cfg5":
            torch.cuda.empty_cache()
            line["fp32_parity_mode"] = fp32_parity_mode(dev)
    print(json.dumps(line))
    if world > 1:
        dist.barrier()


# ------------------------------------------------------------------------------------------------------
# --workload cfg3: HeteroGraphNet on a plateCluster-shaped batch (BASELINE.json configs[2], SURVEY.md s8 cfg 3).
# WRITTEN AFTER THE ROUND'S GPU BUDGET WAS SPENT: not yet run on a GPU.  Not the driver's bench line.
# ------------------------------------------------------------------------------------------------------
CFG3_PLATE, CFG3_OBSTACLE, CFG3_BATCH, CFG3_LAYERS = (21, 20, 3), (4, 4, 4), 16, 5     # 1 260 plate + 64 obstacle nodes (plate.yaml: batch 16, 5 layers)
CFG3_SETS = ["mesh_edges", "world_edges", "intra_cluster_to_mesh", "intra_cluster_to_cluster", "inter_cluster"]   # plate.py:49-57 + connector.initialize


def plate_block_clusters(dims, block=(7, 2, 3)):
    """Block clustering of the plate lattice (node id = (k * ny + j) * nx + i): the host-side stand-in for the reference's sklearn
    clustering (out of scope).  Returns the clusters (index tensors) and the face-adjacent cluster pairs."""
    nx, ny, nz = dims
    bx, by, bz = (-(-nx // block[0]), -(-ny // block[1]), -(-nz // block[2]))
    ids = torch.arange(nx * ny * nz).reshape(nz, ny, nx)
    clusters, neighbors = [], []
    for cz in range(bz):
        for cy in range(by):
            for cx in range(bx):
                sub = ids[cz * block[2]:(cz + 1) * block[2], cy * block[1]:(cy + 1) * block[1], cx * block[0]:(cx + 1) * block[0]]
                clusters.append(sub.reshape(-1).clone())
                k = (cz * by + cy) * bx + cx
                if cx + 1 < bx:
                    neighbors.append(torch.tensor([k, k + 1]))
                if cy + 1 < by:
                    neighbors.append(torch.tensor([k, k + bx]))
                if cz + 1 < bz:
                    neighbors.append(torch.tensor([k, k + bx * by]))
    return clusters, neighbors


def build_plate_batch(dev, seed=0):
    """One batched plateCluster-shaped latent graph: two-body plate frame -> tetra mesh edges, world edges (cell-list kernel),
    hierarchical connector index lists over a block clustering of the plate body, 128-wide seeded latents, batch of 16 through the
    reference's own batching rule (hgn_b200.batching.get_batched, hyper-index quirk included)."""
    from hgn_b200 import synthetic
    from hgn_b200 import util as hutil
    from hgn_b200.batching import get_batched
    from hgn_b200.rmp.hierarchical_connector import connector_indices
    from hgn_b200.world_edges import world_edges
    frame = synthetic.plate_frame(plate=CFG3_PLATE, obstacle=CFG3_OBSTACLE, seed=seed)
    n = frame["world_pos"].shape[0]
    ms, mr = hutil.triangles_to_edges(frame["cells"].long(), deform=True)["two_way_connectivity"]
    ws, wr = world_edges(frame["world_pos"].to(dev), frame["node_type"].to(dev), ms.to(dev), mr.to(dev))
    clusters, neighbors = plate_block_clusters(CFG3_PLATE)
    idx = connector_indices(clusters, neighbors, n, False)
    index_lists = {"mesh_edges": (ms, mr), "world_edges": (ws.cpu(), wr.cpu()), "intra_cluster_to_cluster": idx["intra_cluster_to_cluster"],
                   "intra_cluster_to_mesh": idx["intra_cluster_to_mesh"], "inter_cluster": idx["inter_cluster"]}
    gen = torch.Generator().manual_seed(seed)
    data = []
    for _ in range(CFG3_BATCH):
        nodes = [torch.randn(n, LATENT, generator=gen), torch.randn(len(clusters), LATENT, generator=gen)]
        sets = [hutil.EdgeSet(name, torch.randn(s_.numel(), LATENT, generator=gen), s_, r_) for name, (s_, r_) in index_lists.items()]
        data.append((hutil.MultiGraph(nodes, sets), {}))
    (graph, _), = get_batched(data, CFG3_BATCH)
    return graph, {"nodes": n * CFG3_BATCH, "hyper_nodes": len(clusters) * CFG3_BATCH,
                   "edges": {es.name: int(es.senders.numel()) for es in graph.edge_sets}}


def run_cfg3(args):
    """HeteroGraphNet processor (pna, 5 layers, 5 edge sets, mesh + hyper nodes) fwd+bwd on the batched plate graph: edge-updates/s
    over ALL edge sets, the per-kernel table, the CPU oracle and the torch-CUDA reference beside it."""
    from hgn_b200 import _cabi, ops
    from hgn_b200.migration.meshgraphnet import MeshGraphNet
    from hgn_b200.util import MultiGraph
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    graph_host, sizes = build_plate_batch(dev)
    e_total = sum(sizes["edges"].values())
    torch.manual_seed(0)
    proc = MeshGraphNet(3, LATENT, 2, "pna", CFG3_LAYERS, "hetero", CFG3_SETS).processor.to(dev)
    proc.precision = "bf16"
    nodes_dev = [t.to(dev) for t in graph_host.node_features]
    sets_dev = [es._replace(features=es.features.to(dev), senders=es.senders.to(dev), receivers=es.receivers.to(dev)) for es in graph_host.edge_sets]
    coef = torch.randn(nodes_dev[0].shape, generator=torch.Generator().manual_seed(5)).to(dev)

    def step():
        for p in proc.parameters():
            p.grad = None
        nodes = [t.detach().requires_grad_(True) for t in nodes_dev]
        sets = [es._replace(features=es.features.detach().requires_grad_(True)) for es in sets_dev]
        out = proc(MultiGraph(nodes, sets))
        loss = (out.node_features[0] * coef).sum() + sum(es.features.float().sum() for es in out.edge_sets) * 1e-3
        loss.backward()
        return loss

    for _ in range(max(args.warmup, 3)):
        step()
    torch.cuda.synchronize()
    _cabi.profile(True)
    launches0 = ops.launch_count
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(0) as clocks:
        torch.cuda.synchronize()
        start.record()
        for _ in range(args.steps):
            step()
        stop.record()
        torch.cuda.synchronize()
    ms = start.elapsed_time(stop) / args.steps
    launches = ops.launch_count - launches0
    kernels = _cabi.profile_report()
    _cabi.profile(False)
    d2 = LATENT * LATENT
    k_aggr = 4 * len(CFG3_SETS)
    flops = 3 * (e_total * F_EDGE + (sizes["nodes"] + sizes["hyper_nodes"]) * 2 * ((1 + k_aggr) + 2) * d2) * CFG3_LAYERS   # SURVEY.md s8d
    peak = load_peaks()["bf16_tflops_sustained"]
    graphed = graphed_step(step, list(proc.parameters()), args.steps, e_total * CFG3_LAYERS)
    # baselines: the oracle port on the host cores and on the GPU through torch's own kernels (same weights, same graph)
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import hgn_oracle as orc
    weights = {"processor." + k: v.detach().float() for k, v in proc.state_dict().items()}

    def oracle_pass(device):
        w = {k: v.to(device).requires_grad_(True) for k, v in weights.items()}
        nodes = [t.to(device).clone().requires_grad_(True) for t in graph_host.node_features]
        sets = [orc.EdgeSet(es.name, es.features.to(device).clone().requires_grad_(True), es.senders.to(device), es.receivers.to(device))
                for es in graph_host.edge_sets]
        out = orc.processor(w, "pna", "hetero", orc.MultiGraph(nodes, sets))
        ((out.node_features[0] * coef.to(device)).sum() + sum(es.features.sum() for es in out.edge_sets) * 1e-3).backward()

    torch.set_num_threads(os.cpu_count() or 1)
    t0 = time.perf_counter()
    oracle_pass("cpu")                              # one pass (~15-20 s: the pna aggregates of five edge sets); no separate warm-up
    cpu_s = time.perf_counter() - t0
    oracle_pass(dev); oracle_pass(dev)
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(3):
        oracle_pass(dev)
    b.record()
    torch.cuda.synchronize()
    ref_ms = a.elapsed_time(b) / 3
    print(json.dumps({
        "metric": METRIC, "value": e_total * CFG3_LAYERS / (ms * 1e-3), "unit": UNIT, "n_gpus": 1, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "bf16",
        "data": "synthetic (seeded two-body plate lattice, block clustering, seeded latents and weights)",
        "config": {"workload": f"cfg3: plateCluster-shaped deforming plate ({sizes['nodes'] // CFG3_BATCH} nodes x batch {CFG3_BATCH}), HeteroGraphNet, "
                               f"{CFG3_LAYERS} layers, pna, edge sets {sizes['edges']}, {sizes['hyper_nodes']} hyper nodes, processor fwd+bwd",
                   "l2_policy": "small mesh: the step's working set is L2-resident by construction (launch-bound shape)"},
        "gpu_launches": launches, "clocks": clocks.summary(),
        "layer_roofline": {"tensor_ms_per_layer": flops / CFG3_LAYERS / (peak * 1e12) * 1e3, "measured_ms_per_layer": ms / CFG3_LAYERS,
                           "frac": flops / (peak * 1e12) * 1e3 / ms},
        "kernels": [{"name": k["name"], "launches": k["launches"], "ms_per_step": k["ms"] / args.steps} for k in kernels],
        "cuda_graph": graphed,
        "cpu_baseline": {"value": e_total * CFG3_LAYERS / cpu_s, "unit": UNIT, "cores": torch.get_num_threads(), "kind": "port", "seconds_per_pass": cpu_s,
                         "sample": "the same batched graph and weights, fwd+bwd, fp32, oracle/hgn_oracle.py (block_hetero)"},
        "torch_cuda_reference": {"value": e_total * CFG3_LAYERS / (ref_ms * 1e-3), "unit": UNIT, "ms_per_pass": ref_ms, "kind": "port on torch CUDA ops"},
    }))


def graphed_step(step_fn, params, steps, edge_updates_per_step):
    """The resident step replayed as one CUDA graph (the small-mesh shapes are launch-bound: ~1 100 launches of a few
    microseconds each per step).  Whole-step capture in the usual PyTorch way: warm up on a side stream, drop the gradients so that
    the captured backward allocates them in the graph's pool, capture forward + backward, replay."""
    try:
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(3):
                step_fn()
        torch.cuda.current_stream().wait_stream(side)
        for p in params:
            p.grad = None
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            step_fn()
        for _ in range(3):
            graph.replay()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        reps = steps
        a.record()
        for _ in range(reps):
            graph.replay()
        b.record()
        torch.cuda.synchronize()
        ms = a.elapsed_time(b) / reps
        return {"ms_per_step": ms, "value": edge_updates_per_step / (ms * 1e-3), "unit": UNIT, "steps": reps,
                "what": "forward + backward of the resident step captured once, replayed"}
    except Exception as exc:                         # capture is an optimisation of the host side only
        return {"value": None, "error": f"{type(exc).__name__}: {exc}"[:300]}


def ncu_traffic(kernel_name):
    path = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    try:
        with open(path) as f:
            entry = json.load(f).get("kernels", {}).get(kernel_name)
        return float(entry["dram_bytes_per_launch"]) if entry else None
    except (OSError, ValueError, KeyError, TypeError):
        return None


def dominant_kernel_roofline(kernels, steps, e, n, peaks):
    """Algorithmic FLOPs per launch (SURVEY.md s8d: GEMM flops of the reference's arithmetic, backward = 2x forward,
    recompute earns no credit) over the mean launch time of the kernel that takes the most time in the step.
    `executed` is what the kernel really issues: the node-side pre-projection removes 4 D^2 of the 10 D^2 per edge."""
    if not kernels:
        return None
    top = max(kernels, key=lambda k: k["ms"])
    mean_ms = top["ms"] / top["launches"]
    d2 = LATENT * LATENT
    # name -> (rows per launch, algorithmic flops per row, executed flops per row)
    tensor = {
        "edge_fwd_tc": (e, F_EDGE, 6 * d2), "edge_bwd_tc": (e, 2 * F_EDGE, 18 * d2),
        "node_fwd_tc": (n, F_NODE_SUM, 6 * d2), "node_bwd_tc": (n, 2 * F_NODE_SUM, 18 * d2),
        "mlp_tile_tc_fwd": (n, F_NODE_SUM, F_NODE_SUM), "mlp_tile_tc_bwd": (n, F_NODE_SUM, 2 * F_NODE_SUM),
        "mlp_wgrad_tc": (n, F_NODE_SUM, F_NODE_SUM),
    }.get(top["name"])
    # dram__bytes_read.sum + dram__bytes_write.sum per launch at the full cfg5 size: read from profiles/ncu_traffic.json, which
    # scripts/ncu_summary.py --json writes from an `ncu --set full` capture (kernel, bytes, source report, commit); null when that
    # file has no entry for the kernel or the launch is not the cfg5 size
    traffic = ncu_traffic(top["name"]) if e == 5992002 else None
    if tensor is not None:
        rows, algo_row, exec_row = tensor
        achieved = rows * algo_row / (mean_ms * 1e-3) / 1e12
        peak = peaks["bf16_tflops_sustained"]
        return {"kernel": top["name"], "bound": "tensor", "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak,
                "traffic": traffic, "mean_launch_ms": mean_ms, "launches_per_step": top["launches"] / steps,
                "algorithmic_flops_per_launch": rows * algo_row, "executed_tflops": rows * exec_row / (mean_ms * 1e-3) / 1e12,
                "share_of_step": top["ms"] / sum(k["ms"] for k in kernels),
                "peak_source": peaks["source"] + ", sustained bf16"}
    # an HBM-bound helper kernel dominates: report its bytes (reads + writes of 128-wide bf16 rows)
    bytes_launch = {"segment_reduce": (e + n) * 256 + e * 4, "segment_reduce_bwd": (e + n) * 256 + e * 4,
                    "multi_segment_sum": (2 * e + n) * 256 + 2 * e * 4, "colsum": e * 256}.get(top["name"], 0)
    achieved = bytes_launch / (mean_ms * 1e-3) / 1e9
    return {"kernel": top["name"], "bound": "hbm", "achieved": achieved, "peak": peaks["hbm_gbs"], "unit": "GB/s",
            "frac": achieved / peaks["hbm_gbs"], "traffic": traffic, "mean_launch_ms": mean_ms,
            "share_of_step": top["ms"] / sum(k["ms"] for k in kernels), "peak_source": peaks["source"]}


# ------------------------------------------------------------------------------------------------------
# second half of the metric: rollout steps/sec (BASELINE.json configs[1]: flag_simple-shaped cloth, 15 MP layers, 400 steps)
# ------------------------------------------------------------------------------------------------------
ROLLOUT_W, ROLLOUT_H, ROLLOUT_STEPS = 40, 40, 400      # 1 600 nodes / 9 282 directed edges ~ flag_simple (1 579 / 9 212)


def _cloth_features(world, prev, mesh_pos, pinned_type, senders, receivers):
    """FlagModel.build_graph (src/model/flag.py:65-128) on device tensors: velocity + node-type one-hot, relative world / mesh
    positions and their norms."""
    node_features = torch.cat((world - prev, pinned_type), dim=-1)
    rel_world = world[senders] - world[receivers]
    rel_mesh = mesh_pos[senders] - mesh_pos[receivers]
    edge_features = torch.cat((rel_world, rel_world.pow(2).sum(-1, keepdim=True).sqrt(),
                               rel_mesh, rel_mesh.pow(2).sum(-1, keepdim=True).sqrt()), dim=-1)
    return node_features, edge_features


def flag_model_params(aggregation="pna", steps=LAYERS):
    """The model section of configs/flag.yaml without remote message passing (BASELINE.json configs[1]: MeshGraphNets, 15 MP layers)."""
    return {"size": 3, "aggregation": aggregation, "message_passing_steps": steps,
            "rmp": {"num_clusters": 10, "hyper_noise": "none", "hyper_node_features": True, "frequency": 1, "clustering": "none",
                    "connector": "none", "fully_connect": False,
                    "intra_cluster_sampling": {"enabled": False, "alpha": 0.1, "spotter_threshold": 0},
                    "hdbscan": {"max_cluster_size": 50, "min_cluster_size": 20, "min_samples": 1, "spotter_threshold": 0.9}},
            "graph_balancer": {"algorithm": "none", "frequency": 1, "remove_edges": True, "ricci": {"loops": 150, "tau": 150},
                               "random": {"edge_amount": 100}}}


def rollout_model_and_trajectory(FlagModel, dev, steps):
    """The reference's own ``FlagModel`` (src/model/flag.py; on whatever ``src.migration`` modules are installed in this process) with
    seeded weights and normaliser statistics, and a synthetic ``[T, N, .]`` trajectory dict for ``model.rollout``."""
    from hgn_b200 import synthetic
    torch.manual_seed(0)
    model = FlagModel(flag_model_params())
    base = synthetic.cloth_frame(ROLLOUT_W, ROLLOUT_H, seed=1)
    n = ROLLOUT_W * ROLLOUT_H
    drift = synthetic.seeded_tensor("rollout_drift", (n, 3), 2)
    pos = [base["world_pos"] + 0.002 * t * drift for t in range(-1, 4)]
    frames = [{**base, "prev|world_pos": pos[t], "world_pos": pos[t + 1], "target|world_pos": pos[t + 2]} for t in range(3)]
    frames = [{k: v.to(dev) for k, v in f.items()} for f in frames]
    model.train()
    for f in frames:                                     # normaliser statistics (flag.py:96, 115, 192)
        g = model.build_graph(f, True)
        model.get_target(f, True)
    with torch.no_grad():
        model(g)
    net = model.learned_model
    shapes = {k: tuple(v.shape) for k, v in net.state_dict().items()}
    net.load_state_dict({k: v.to(dev) for k, v in synthetic.seeded_state_dict(shapes, 29).items()})
    model.eval()
    traj = {k: v.unsqueeze(0).expand(steps, *v.shape).contiguous() for k, v in frames[0].items()}
    return model, traj


def rollout_bench(dev):
    """The metric's second half (BASELINE.json configs[1]): 400 closed-loop steps of a flag_simple-shaped cloth, GraphNet pna, 15 layers.

    `value` / `via`: the reference's OWN ``FlagModel.rollout`` (src/model/flag.py:194-246: build_graph with its normalisers, predict,
    second-order integrate, pin the handle nodes, every step) running unchanged on the installed hgn_b200 modules, bf16 processor.
    `cuda_graph`: the same step (same model object, same normalisers, same arithmetic) captured once in a CUDA graph and replayed --
    what hgn_b200.graphed offers on top of the drop-in.  `cpu_reference`: FlagModel.rollout of the unmodified reference on the host
    cores (GPU-less child process), bounded to a few steps."""
    import hgn_b200
    shim = _reference_shim()
    out = {"unit": "rollout steps/s", "steps": ROLLOUT_STEPS,
           "config": f"{ROLLOUT_W}x{ROLLOUT_H} flag-style cloth ({ROLLOUT_W * ROLLOUT_H} nodes), FlagModel: encoder + {LAYERS} GraphNet layers (pna, bf16 "
                     f"processor) + decoder, normalisers, {ROLLOUT_STEPS} closed-loop steps"}
    if not shim.available():
        out["value"] = None
        out["via"] = "unavailable: no reference tree (oracle/_ref not staged)"
        return out
    shim._install_stub_modules()
    if shim.REFERENCE_ROOT not in sys.path:
        sys.path.insert(0, shim.REFERENCE_ROOT)
    os.environ.setdefault("WANDB_MODE", "disabled")
    hgn_b200.install_as_reference_modules()
    from src.model.flag import FlagModel
    prev_precision = hgn_b200.precision()
    hgn_b200.set_precision("bf16")
    try:
        model, traj = rollout_model_and_trajectory(FlagModel, dev, ROLLOUT_STEPS)
        model.rollout({k: v[:5] for k, v in traj.items()}, 5)                   # plans, packed weights
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        _, mse = model.rollout(traj, ROLLOUT_STEPS)
        torch.cuda.synchronize()
        out["value"] = ROLLOUT_STEPS / (time.perf_counter() - t0)
        out["via"] = "FlagModel.rollout"
        out["finite"] = bool(torch.isfinite(mse).all())
        try:
            from hgn_b200 import graphed
            out["cuda_graph"] = graphed.flag_rollout_steps_per_second(model, traj, ROLLOUT_STEPS)
        except Exception as exc:                         # capture is an optimisation of the host side only
            out["cuda_graph"] = None
            out["cuda_graph_error"] = f"{type(exc).__name__}: {exc}"[:300]
    finally:
        hgn_b200.set_precision(prev_precision)
    ref = _reference_subprocess(["--steps", "1", "--warmup", "1", "--rollout-steps", "10", "--train-steps", "5"], timeout=900)
    if ref is not None and ref.get("rollout"):
        out["cpu_reference"] = ref["rollout"]
    try:
        out["training"] = training_bench(FlagModel, dev, ref.get("training") if ref else None)
    except Exception as exc:
        out["training"] = {"error": f"{type(exc).__name__}: {exc}"[:300]}
    return out


TRAIN_STEPS = 100


def flag_training_loop(model, frame, optimizer, steps):
    """The reference's inner training loop on one frame (MeshSimulator.py:131-139)."""
    for _ in range(steps):
        graph = model.build_graph(frame, True)
        loss = model.training_step(graph, frame)
        loss.backward()
        optimizer.step()
        optimizer.zero_grad()
    return loss


def training_bench(FlagModel, dev, cpu_reference):
    """Training iterations/s of the flag_simple-shaped model (BASELINE.json configs[1]: 1 600 nodes, GraphNet pna, 15 layers; one
    frame per iteration): the reference's own loop (build_graph, FlagModel.training_step, backward, Adam) on the installed hgn_b200
    modules in bf16, the same iteration captured in one CUDA graph (hgn_b200.graphed.FlagTrainingGraph), and the unmodified
    reference on the host cores."""
    import copy
    import hgn_b200
    from hgn_b200.graphed import FlagTrainingGraph
    prev_precision = hgn_b200.precision()
    hgn_b200.set_precision("bf16")
    try:
        model, traj = rollout_model_and_trajectory(FlagModel, dev, 2)
        frame = {k: v[0] for k, v in traj.items()}
        model.train()
        twin = copy.deepcopy(model)
        opt = torch.optim.Adam(model.parameters(), lr=1e-4)
        flag_training_loop(model, frame, opt, 5)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        loss = flag_training_loop(model, frame, opt, TRAIN_STEPS)
        torch.cuda.synchronize()
        out = {"unit": "training iterations/s", "steps": TRAIN_STEPS, "value": TRAIN_STEPS / (time.perf_counter() - t0), "via": "FlagModel.training_step + Adam",
               "finite": bool(torch.isfinite(loss))}
        runner = FlagTrainingGraph(twin, frame, torch.optim.Adam(twin.parameters(), lr=1e-4, capturable=True))
        for _ in range(5):
            runner.step(frame)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(TRAIN_STEPS):
            loss = runner.step(frame)
        torch.cuda.synchronize()
        out["cuda_graph"] = {"value": TRAIN_STEPS / (time.perf_counter() - t0), "finite": bool(torch.isfinite(loss)),
                             "what": "the same iteration (normalisers, encoder, 15 layers, decoder, masked loss, backward, Adam) as one CUDA graph"}
    finally:
        hgn_b200.set_precision(prev_precision)
    if cpu_reference:
        out["cpu_reference"] = cpu_reference
    return out


# ------------------------------------------------------------------------------------------------------
# CPU baseline / reference arm: the oracle port of the reference's torch path on the host cores
# ------------------------------------------------------------------------------------------------------
CPU_SAMPLE_W, CPU_SAMPLE_H, CPU_SAMPLE_LAYERS = 1000, 125, 1


def _reference_shim():
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import reference_shim
    return reference_shim


def cpu_state(sample=None, aggregator="sum", prefer_reference=True):
    """(step function, directed edges, kind).  kind 'reference': the reference's OWN ``Processor`` / ``GraphNet`` modules
    (src/migration/processor.py:27-28, graphnet.py:22-84; torch_scatter restated by oracle/reference_shim.py) from /root/reference or
    the staged oracle/_ref, with device = cpu -- only possible in a process that sees no GPU (src/util.py:9).  kind 'port':
    oracle/hgn_oracle.py, used when the reference tree is absent or a GPU is visible."""
    torch.set_num_threads(os.cpu_count() or 1)
    w_, h_, batch, layers = sample or (CPU_SAMPLE_W, CPU_SAMPLE_H, 1, CPU_SAMPLE_LAYERS)
    data = build_inputs(w_, h_, layers, aggregator=aggregator, batch=batch)
    v0, e0, s, r, coef = data["v0"], data["e0"], data["senders"], data["receivers"], data["coef_v"]
    shim = _reference_shim()
    if prefer_reference and shim.available() and not torch.cuda.is_available():
        shim.load()
        from src.migration.meshgraphnet import MeshGraphNet as RefMeshGraphNet
        from src.util import EdgeSet as RefEdgeSet, MultiGraph as RefMultiGraph
        proc = RefMeshGraphNet(output_size=3, latent_size=LATENT, num_layers=2, message_passing_aggregator=aggregator,
                               message_passing_steps=layers, architecture="none", edge_sets=["mesh_edges"]).processor
        with torch.no_grad():                   # materialise the LazyLinear parameters on a one-edge graph
            proc(RefMultiGraph([torch.zeros(2, LATENT)], [RefEdgeSet("mesh_edges", torch.zeros(1, LATENT), torch.zeros(1, dtype=torch.long),
                                                                     torch.ones(1, dtype=torch.long))]))
        proc.load_state_dict({k[len("processor."):]: t for k, t in data["weights"].items()})
        params = list(proc.parameters())

        def step():
            for p in params:
                p.grad = None
            v = v0.clone().requires_grad_(True)
            ed = e0.clone().requires_grad_(True)
            out = proc(RefMultiGraph([v], [RefEdgeSet("mesh_edges", ed, s, r)]))
            loss = (out.node_features[0] * coef).sum() + out.edge_sets[0].features.sum() * 1e-3
            loss.backward()
            return float(loss)
        return step, data["e"], "reference"
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import hgn_oracle as orc
    w = {k: t.clone().requires_grad_(True) for k, t in data["weights"].items()}

    def step():
        for t in w.values():
            t.grad = None
        v = v0.clone().requires_grad_(True)
        ed = e0.clone().requires_grad_(True)
        out = orc.processor(w, aggregator, "none", orc.MultiGraph([v], [orc.EdgeSet("mesh_edges", ed, s, r)]))
        loss = (out.node_features[0] * coef).sum() + out.edge_sets[0].features.sum() * 1e-3
        loss.backward()
        return float(loss)
    return step, data["e"], "port"


def _cpu_sample_text(sample, e, aggregator, kind):
    w_, h_, batch, layers = sample
    what = ("the reference's own src/migration Processor (unmodified; torch_scatter restated by oracle/reference_shim.py)" if kind == "reference"
            else "oracle/hgn_oracle.py (torch CPU ops = the reference's own arithmetic)")
    return (f"{w_}x{h_}" + (f" x {batch}" if batch > 1 else "") + f" mesh of the workload ({e} directed edges), {layers} layer(s), {aggregator}, "
            f"fwd+bwd, fp32, {what}, all host threads")


def cpu_baseline_inprocess(steps=1, sample=None, aggregator="sum"):
    sample = sample or _sample_override((CPU_SAMPLE_W, CPU_SAMPLE_H, 1, CPU_SAMPLE_LAYERS))
    step, e, kind = cpu_state(sample, aggregator)
    step()                               # untimed: first touch / thread pool start
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    dt = (time.perf_counter() - t0) / steps
    return {"value": e * sample[3] / dt, "unit": UNIT, "cores": torch.get_num_threads(), "kind": kind, "seconds_per_pass": dt,
            "sample": _cpu_sample_text(sample, e, aggregator, kind)}


def _reference_subprocess(extra, timeout=900):
    """`bench.py --impl reference ...` in a child that sees no GPU; returns its JSON line (or None)."""
    try:
        run = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference"] + extra, capture_output=True, text=True,
                             timeout=timeout, env=dict(os.environ, CUDA_VISIBLE_DEVICES="", WANDB_MODE="disabled"))
        lines = [ln for ln in run.stdout.splitlines() if ln.startswith("{")]
        return json.loads(lines[-1]) if run.returncode == 0 and lines else None
    except (subprocess.TimeoutExpired, OSError, ValueError):
        return None


def cpu_baseline(steps=1, sample=None, aggregator="sum", workload="cfg5"):
    """The CPU arm beside the number: the live reference in a GPU-less child process (kind 'reference'); the oracle port in this
    process only if that child could not run."""
    line = _reference_subprocess(["--workload", workload, "--aggregator", aggregator, "--steps", str(steps), "--warmup", "1"])
    if line is not None and line.get("cpu_baseline"):
        return line["cpu_baseline"]
    return cpu_baseline_inprocess(steps, _sample_override(sample) if sample else None, aggregator)


def torch_cuda_reference(dev, data, aggregator, layers):
    """Same-box torch path (SURVEY.md s8d): the reference's arithmetic (the oracle port: index_select / cat / addmm / relu /
    layer_norm / scatter_add through autograd, fp32 features, int64 indices) on the B200 through torch's own CUDA kernels, on the
    workload's full mesh.  A baseline beside the number, like `cpu_baseline`; none of hgn_b200's kernels run here."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import hgn_oracle as orc
    keep = tuple(f"processor.graphnet_blocks.{i}." for i in range(layers))
    w = {k: t.to(dev).requires_grad_(True) for k, t in data["weights"].items() if k.startswith(keep)}
    v0, e0, coef = data["v0"].to(dev), data["e0"].to(dev), data["coef_v"].to(dev)
    s, r = data["senders"].to(dev), data["receivers"].to(dev)

    def one():
        for t in w.values():
            t.grad = None
        v = v0.clone().requires_grad_(True)
        ed = e0.clone().requires_grad_(True)
        out = orc.processor(w, aggregator, "none", orc.MultiGraph([v], [orc.EdgeSet("mesh_edges", ed, s, r)]))
        ((out.node_features[0] * coef).sum() + out.edge_sets[0].features.sum() * 1e-3).backward()

    try:
        for _ in range(2):
            one()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        reps = 3
        a.record()
        for _ in range(reps):
            one()
        b.record()
        torch.cuda.synchronize()
        ms = a.elapsed_time(b) / reps
        return {"value": data["e"] * layers / (ms * 1e-3), "unit": UNIT, "ms_per_pass": ms, "kind": "port on torch CUDA ops",
                "sample": f"the workload's full mesh ({data['e']} directed edges), {layers} layer(s), {aggregator}, fwd+bwd, fp32, "
                          "oracle/hgn_oracle.py on cuda:0 (torch eager kernels: cuBLAS addmm, scatter_add atomics)"}
    except Exception as exc:                    # e.g. out of memory: a baseline, never fatal to the bench line
        return {"value": None, "error": f"{type(exc).__name__}: {exc}"[:200]}


def reference_rollout(steps):
    """The metric's second half on the reference arm: the reference's own ``FlagModel.rollout`` (src/model/flag.py:194-246) on the
    CPU -- 40x40 cloth, GraphNet pna, 15 layers (BASELINE.json configs[1]) -- for `steps` closed-loop steps."""
    shim = _reference_shim()
    shim.load()
    os.chdir(shim.REFERENCE_ROOT)
    from src.model.flag import FlagModel
    model, traj = rollout_model_and_trajectory(FlagModel, torch.device("cpu"), steps)
    model.rollout({k: v[:2] for k, v in traj.items()}, 2)        # lazy linears
    t0 = time.perf_counter()
    model.rollout(traj, steps)
    return steps / (time.perf_counter() - t0)


def _sample_override(sample):
    """HGN_BENCH_CPU_SAMPLE=WxH[xBATCH[xLAYERS]] shrinks the CPU sample (tests)."""
    env = os.environ.get("HGN_BENCH_CPU_SAMPLE")
    if not env:
        return sample
    parts = [int(x) for x in env.split("x")]
    return tuple(parts + list(sample[len(parts):]))


def run_reference(args):
    if int(os.environ.get("RANK", "0")) != 0:
        return
    _, _, _, _, default_agg, sample, wl_text = WORKLOADS.get(getattr(args, "workload", "cfg5"), WORKLOADS["cfg5"])
    sample = _sample_override(sample)
    aggregator = args.aggregator or default_agg
    step, e, kind = cpu_state(sample, aggregator)
    layers = sample[3]
    warm = max(1, min(args.warmup, 8))                         # W warm-up passes as asked (a pass is ~1.7 s on 16 cores; capped at 8)
    for _ in range(warm):
        step()
    steps = max(1, args.steps)
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    dt = (time.perf_counter() - t0) / steps
    value = e * layers / dt
    cores = torch.get_num_threads()
    sample_text = "each step = " + _cpu_sample_text(sample, e, aggregator, kind)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": int(os.environ.get("WORLD_SIZE", "1")),
        "steps": steps, "warmup": warm, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic (same seeded grid mesh family)",
        "config": {"workload": f"{wl_text}, {WORKLOADS.get(getattr(args, 'workload', 'cfg5'), WORKLOADS['cfg5'])[3]} GraphNet layers, {aggregator} aggregator, processor fwd+bwd",
                   "sample": sample_text},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample_text, "seconds_per_pass": dt},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    if getattr(args, "rollout_steps", 0) > 0 and kind == "reference":
        line["rollout"] = {"value": reference_rollout(args.rollout_steps), "unit": "rollout steps/s", "steps": args.rollout_steps, "cores": cores,
                           "via": "FlagModel.rollout (unmodified reference, CPU)"}
    if getattr(args, "train_steps", 0) > 0 and kind == "reference":
        shim = _reference_shim()
        shim.load()
        os.chdir(shim.REFERENCE_ROOT)
        from src.model.flag import FlagModel
        model, traj = rollout_model_and_trajectory(FlagModel, torch.device("cpu"), 2)
        frame = {k: v[0] for k, v in traj.items()}
        model.train()
        opt = torch.optim.Adam(model.parameters(), lr=1e-4)
        flag_training_loop(model, frame, opt, 1)
        t0 = time.perf_counter()
        flag_training_loop(model, frame, opt, args.train_steps)
        line["training"] = {"value": args.train_steps / (time.perf_counter() - t0), "unit": "training iterations/s", "steps": args.train_steps,
                            "cores": cores, "via": "FlagModel.training_step + Adam (unmodified reference, CPU)"}
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--aggregator", default=None, choices=["sum", "pna"],
                    help="message-passing aggregator (default: the workload's; the headline metric is quoted on 'sum'; 'pna' is the "
                         "reference configs' default)")
    ap.add_argument("--rollout-steps", type=int, default=0, help="reference arm only: also time FlagModel.rollout for this many steps")
    ap.add_argument("--train-steps", type=int, default=0, help="reference arm only: also time this many FlagModel training iterations")
    ap.add_argument("--workload", default="cfg5", choices=sorted(WORKLOADS) + ["cfg3"],
                    help="cfg5 = the headline 1M/6M mesh (the bench line); cfg2 / cfg4 = small-mesh batched training shapes; "
                         "cfg3 = HeteroGraphNet on a plateCluster-shaped batch (single GPU)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed (loss, sampled output latents and input-latent "
                         "gradients, parameter gradients) as float32 DIR/<name>.npy, at most 64 MB; single GPU, cfg2 / cfg4 / cfg5")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl == "reference" or args.workload == "cfg3"):
        ap.error("--dump-outputs covers the single-GPU path of --impl ours on cfg2 / cfg4 / cfg5")
    if args.impl == "reference":
        run_reference(args)
    elif args.workload == "cfg3":
        run_cfg3(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
