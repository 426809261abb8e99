"""Long-segment reductions (HyperGraphNet cluster pooling and broadcast at mesh scale): the existing segment entry points against the
split ones, alternated in one process.  Writes profiles/hyper_scale_b200.json (or --out) with the card's name and power limit.

1. Kernel sweep: one segment of L rows (L = 256 .. 10^6) and the up-pooling shape (10^6 rows into 16 clusters, behind 10^6 empty mesh
   segments), 'sum' and 'pna' (sum, mean, max, min + winners) forward, and the four-term backward of the up-pooling shape; the split
   path at piece sizes P = 128 .. 1024.  The library's split (threshold T, piece P) is what the bindings use; the other piece sizes, and
   lengths <= T, run the same split entry points on a split built here (every non-empty segment long), which is how T and P were chosen.
   Achieved GB/s counts the compulsory bytes only: forward E x 256 B of rows read plus, per long segment, 256 B per bf16 output and 512 B
   per int32 winner row; backward E x 256 B of gradient rows written plus four 256 B gradient rows read per long segment.
2. Processors: HyperGraphNet and HeteroGraphNet at 1000 x 1000 nodes in 16 clusters, 'sum' and 'pna', 5 layers, forward + backward in bf16,
   with the split and with every plan's split bypassed (the existing kernels), alternated: ms per step, peak allocation, per-kernel table.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "hyper-graph-nets_b200"))
from hgn_b200 import _cabi, ops, synthetic  # noqa: E402
from hgn_b200.migration.meshgraphnet import MeshGraphNet  # noqa: E402
from hgn_b200.plan import SegmentPlan  # noqa: E402
from hgn_b200.util import EdgeSet, MultiGraph  # noqa: E402

BF = _cabi.HGN_BF16


def _card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else "unknown"


def _time(fn, iters):
    fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / iters


class _Split:
    """A split of ``plan`` in which every non-empty segment is long, cut into pieces of ``P`` perm positions."""

    def __init__(self, plan, P):
        rowptr = plan.rowptr.cpu().long()
        counts = rowptr[1:] - rowptr[:-1]
        long_ids = torch.nonzero(counts > 0).flatten()
        pieces = [(int(s), b, min(b + P, int(rowptr[s + 1]))) for s in long_ids for b in range(int(rowptr[s]), int(rowptr[s + 1]), P)]
        n_per = (counts[long_ids] + P - 1) // P
        i32 = lambda t: torch.as_tensor(t, dtype=torch.int32).reshape(-1).cuda()
        self.long_ids, self.pieces = i32(long_ids), i32(pieces)
        self.piece_ptr = i32(torch.cat([torch.zeros(1, dtype=torch.int64), n_per.cumsum(0)]))
        self.perm_short, self.rowptr_short = torch.zeros(1, dtype=torch.int32, device="cuda"), torch.zeros(plan.num_segments + 1, dtype=torch.int32, device="cuda")
        self.n_long, self.n_pieces = len(long_ids), len(pieces)
        self.c = _cabi.SegmentSplit(plan.num_segments, plan.num_elements, self.n_long, self.n_pieces, 0, self.long_ids.data_ptr(),
                                    self.piece_ptr.data_ptr(), self.pieces.data_ptr(), self.perm_short.data_ptr(), self.rowptr_short.data_ptr())


def _case(ids, S, pna, iters, backward=False, P=None):
    lib = _cabi.load()
    plan = SegmentPlan(ids, S)
    E = ids.numel()
    x = torch.randn(E, 128, device="cuda").to(torch.bfloat16)
    sp = plan.split if P is None else _Split(plan, P)
    outs = [torch.empty(S, 128, dtype=torch.bfloat16, device="cuda") for _ in range(4 if pna else 1)] + [None] * (0 if pna else 3)
    am = torch.empty(S, 128, dtype=torch.int32, device="cuda") if pna else None
    an = torch.empty(S, 128, dtype=torch.int32, device="cuda") if pna else None
    ws = torch.empty(max(lib.hgn_segment_split_reduce_workspace_bytes(ctypes.byref(sp.c)), 1), dtype=torch.uint8, device="cuda")
    st = _cabi.stream_ptr()
    ptrs = [_cabi.ptr(o) for o in outs]
    old = lambda: lib.hgn_segment_reduce(BF, x.data_ptr(), E, 128, plan.perm.data_ptr(), plan.rowptr.data_ptr(), S, *ptrs, _cabi.ptr(am),
                                         _cabi.ptr(an), 0, st)
    new = lambda: lib.hgn_segment_reduce_split(BF, x.data_ptr(), E, 128, plan.perm.data_ptr(), plan.rowptr.data_ptr(), S, ctypes.byref(sp.c),
                                               *ptrs, _cabi.ptr(am), _cabi.ptr(an), 0, ws.data_ptr(), ws.numel(), st)
    n_out_bytes = sp.n_long * (256 * (4 if pna else 1) + (1024 if pna else 0))
    if backward:
        old()                                                # the winners the backward reads
        g = [torch.randn(S, 128, device="cuda").to(torch.bfloat16) for _ in range(4)]
        grad = torch.empty(E, 128, dtype=torch.bfloat16, device="cuda")
        old = lambda: lib.hgn_segment_reduce_bwd(BF, E, 128, plan.ids32.data_ptr(), plan.perm.data_ptr(), plan.rowptr.data_ptr(), S,
                                                 *[t.data_ptr() for t in g], am.data_ptr(), an.data_ptr(), grad.data_ptr(), 0, st)
        new = lambda: lib.hgn_segment_reduce_bwd_split(BF, E, 128, plan.ids32.data_ptr(), plan.perm.data_ptr(), plan.rowptr.data_ptr(), S,
                                                       ctypes.byref(sp.c), *[t.data_ptr() for t in g], am.data_ptr(), an.data_ptr(),
                                                       grad.data_ptr(), st)
    bytes_ = E * 256 + n_out_bytes
    if backward:
        bytes_ = E * 256 + sp.n_long * 4 * 256
    t_old, t_new = [], []
    for _ in range(3):                                      # alternated
        t_old.append(_time(old, iters))
        t_new.append(_time(new, iters))
    to, tn = min(t_old), min(t_new)
    return {"E": E, "S": S, "P": P or lib.hgn_segment_split_piece(), "n_long": sp.n_long, "n_pieces": sp.n_pieces, "pna": pna,
            "backward": backward,
            "old_ms": to, "split_ms": tn, "old_GBps": bytes_ / to / 1e6, "split_GBps": bytes_ / tn / 1e6, "speedup": to / tn}


def _processor(arch, agg, layers, steps, width=1000, height=1000, clusters=16):
    """ms per forward + backward step of a bf16 processor, with the split and with every plan's split bypassed, alternated."""
    torch.manual_seed(0)
    edges = {nm: (s.cuda(), r.cuda()) for nm, (s, r) in synthetic.hyper_grid_edges(width, height, clusters).items()}
    n = width * height
    w = synthetic.seeded_state_dict(synthetic.hyper_processor_shapes(arch, agg, layers), 5)
    proc = MeshGraphNet(3, 128, 2, agg, layers, arch, list(synthetic.HYPER_EDGE_SETS)).processor
    proc.load_state_dict({k[len("processor."):]: t for k, t in w.items()})
    proc = proc.cuda()
    proc.precision = "bf16"
    nodes = [torch.randn(n, 128, device="cuda").requires_grad_(True), torch.randn(clusters, 128, device="cuda").requires_grad_(True)]
    feats = {nm: torch.randn(s.numel(), 128, device="cuda").requires_grad_(True) for nm, (s, _) in edges.items()}

    def step():
        proc.zero_grad(set_to_none=True)
        out = proc(MultiGraph(list(nodes), [EdgeSet(nm, feats[nm], s, r) for nm, (s, r) in edges.items()]))
        loss = sum(v.float().square().mean() for v in out.node_features) + sum(x.features.float().square().mean() for x in out.edge_sets)
        loss.backward()

    split_of = ops._split_of
    modes = {"old": lambda plan, S, E: None, "split": split_of}
    res = {"architecture": arch, "aggregator": agg, "layers": layers, "nodes": n, "clusters": clusters,
           "edges": {nm: s.numel() for nm, (s, _) in edges.items()}, "kernels": {}}
    try:
        for mode, fn in modes.items():                      # warm-up: plans, splits, packed weights
            ops._split_of = fn
            step()
        times = {m: [] for m in modes}
        for _ in range(2):
            for mode, fn in modes.items():
                ops._split_of = fn
                torch.cuda.synchronize()
                torch.cuda.reset_peak_memory_stats()
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                for _ in range(steps):
                    step()
                b.record()
                torch.cuda.synchronize()
                times[mode].append(a.elapsed_time(b) / steps)
                res[f"{mode}_peak_GB"] = torch.cuda.max_memory_allocated() / 1e9
        for mode, fn in modes.items():                      # per-kernel table: one step each, in a run of its own
            ops._split_of = fn
            _cabi.profile(True)
            step()
            res["kernels"][mode] = _cabi.profile_report()
            _cabi.profile(False)
    finally:
        ops._split_of = split_of
    for mode in modes:
        res[f"{mode}_ms"] = min(times[mode])
    res["speedup"] = res["old_ms"] / res["split_ms"]
    seg = lambda m: sum(k["ms"] for k in res["kernels"][m] if "segment" in k["name"])
    res["segment_kernels_ms"] = {m: seg(m) for m in modes}
    return res


def _write(path, res):
    os.makedirs(os.path.dirname(os.path.abspath(path)), exist_ok=True)
    with open(path, "w") as f:
        json.dump(res, f, indent=1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "hyper_scale_b200.json"))
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--steps", type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_hyper_scale needs a GPU")
    res = {"card": _card(), "T": _cabi.load().hgn_segment_split_threshold(), "P": _cabi.load().hgn_segment_split_piece(), "sweep": []}
    T = res["T"]
    for L in [256, 1024, 2048, T + 1, 4096, 16384, 65536, 262144, 1_000_000]:
        for pna in (False, True):
            r = _case(torch.zeros(L, dtype=torch.int64, device="cuda"), 1, pna, args.iters, P=None if L > T else res["P"])
            r["shape"] = f"one segment of {L}"
            res["sweep"].append(r)
            print(json.dumps(r), flush=True)
    up = torch.arange(16, device="cuda").repeat_interleave(62_500) + 1_000_000
    up = up[torch.randperm(up.numel(), device="cuda")]
    for pna, bwd in ((False, False), (True, False), (True, True)):
        for P in (128, 256, 512, 1024):
            r = _case(up, 1_000_016, pna, args.iters, backward=bwd, P=None if P == res["P"] else P)
            r["shape"] = "up-pooling: 10^6 rows into 16 clusters + 10^6 empty segments"
            res["sweep"].append(r)
            print(json.dumps(r), flush=True)
    _write(args.out, res)
    res["processors"] = []
    for arch in ("hyper", "hetero"):
        for agg in ("sum", "pna"):
            r = _processor(arch, agg, 5, args.steps)
            res["processors"].append(r)
            print(json.dumps({k: v for k, v in r.items() if k != "kernels"}), flush=True)
            _write(args.out, res)
    print("card:", res["card"])


if __name__ == "__main__":
    main()
