"""bench.py on the GPU: `--steps` sets the number of steps of every timed leg, and `--dump-outputs` writes the last timed step's
results -- the same arrays from two runs with the same arguments (seeded inputs, deterministic kernels)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
pytestmark = pytest.mark.gpu


def _bench(out_dir):
    env = dict(os.environ, HGN_BENCH_NO_CPU="1", HGN_BENCH_NO_TORCH_REFERENCE="1")
    run = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "cfg2", "--steps", "2", "--warmup", "1",
                          "--dump-outputs", str(out_dir)], capture_output=True, text=True, timeout=600, env=env)
    assert run.returncode == 0, run.stdout[-2000:] + run.stderr[-4000:]
    line = json.loads(run.stdout.strip().splitlines()[-1])
    return line, {f.name[:-4]: np.load(f) for f in out_dir.iterdir()}


def test_steps_and_dump_outputs(tmp_path):
    line, first = _bench(tmp_path / "a")
    assert line["steps"] == 2 and line["e2e"]["steps"] == 2 and line["cuda_graph"]["steps"] == 2
    assert {"loss", "node_latents", "edge_latents", "node_latents_grad", "edge_latents_grad"} <= set(first)
    assert sum(k.startswith("grad.graphnet_blocks.") for k in first) == 16 * 15          # every parameter of the 15 layers
    assert all(a.dtype == np.float32 and np.isfinite(a).all() for a in first.values())
    assert sum(a.nbytes for a in first.values()) <= 64 << 20
    assert first["node_latents"].shape == (16384, 128) and first["edge_latents_grad"].shape == (16384, 128)
    _, second = _bench(tmp_path / "b")
    assert set(second) == set(first)
    for name, a in first.items():
        assert np.array_equal(a, second[name]), name
