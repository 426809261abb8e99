"""TEST INFRASTRUCTURE -- one process of tests/test_aggregator_layer_gpu.py::test_route_and_launch_count (the aggregator is the first
argument).

A one-block bf16 processor on the 40 x 32 grid of tests/test_layer_schedule_gpu.py: one fwd+bwd step after a warm-up step under
``torch.profiler`` (CUDA activities).  Prints one JSON line: the change in ``ops.launch_count`` and the names of the ``hgn::`` kernels the
profiler recorded.  A process of its own, so that the profiler sessions of this check leave the test process's profiler state as it was:
``tests/test_layer_schedule_gpu.py`` makes the same comparison there."""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (os.path.join(ROOT, "hyper-graph-nets_b200"), os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests")):
    sys.path.insert(0, p)

import torch  # noqa: E402

from hgn_b200 import ops, synthetic  # noqa: E402
from test_layer_schedule_gpu import _processor, _step, _whole  # noqa: E402

aggregator = sys.argv[1]
W, H = 40, 32
s, r = synthetic.grid_edges_two_way(W, H)
gen = torch.Generator().manual_seed(3)
n, e = W * H, s.numel()
v0, e0, coef = (torch.randn(rows, 128, generator=gen).cuda() for rows in (n, e, n))
proc = _processor(aggregator, 1)
run, params = _whole(proc, s, r), list(proc.parameters())
_step(run, params, v0, e0, coef)                  # warm-up: the packed weights are cached after it
torch.cuda.synchronize()
before = ops.launch_count
with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
    _step(run, params, v0, e0, coef)
    torch.cuda.synchronize()
counted = ops.launch_count - before
print(json.dumps({"counted": counted, "kernels": [ev.name for ev in prof.events() if "hgn::" in ev.name]}), flush=True)
