"""TEST INFRASTRUCTURE -- worker of tests/test_io_mlp_gpu.py (a subprocess: it installs hgn_b200 as the reference's ``src.migration``).
The reference's own ``FlagModel.rollout`` eagerly, against the same closed loop captured in one CUDA graph per step
(``hgn_b200.graphed.FlagRolloutGraph``), in bf16 with the encoder and decoder kernels (HGN_B200_IO_KERNELS=1 in the environment):
the positions must be bit-identical."""
import os
import sys

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, os.path.join(ROOT, "oracle"))
sys.path.insert(0, os.path.join(ROOT, "hyper-graph-nets_b200"))
sys.path.insert(0, HERE)
os.environ.setdefault("WANDB_MODE", "disabled")

import reference_shim  # noqa: E402
import dropin_runner  # noqa: E402

if not reference_shim.available():
    raise SystemExit("SKIP: no reference tree")
reference_shim._install_stub_modules()
sys.path.insert(0, reference_shim.REFERENCE_ROOT)
os.chdir(reference_shim.REFERENCE_ROOT)
import hgn_b200  # noqa: E402
from hgn_b200 import ops, synthetic  # noqa: E402
from hgn_b200.graphed import FlagRolloutGraph  # noqa: E402

hgn_b200.set_precision("bf16")
assert hgn_b200.io_kernels(), "run with HGN_B200_IO_KERNELS=1"
hgn_b200.install_as_reference_modules()
from src.model.flag import FlagModel  # noqa: E402
import src.util  # noqa: E402

dev = src.util.device
frames = [{k: v.to(dev) for k, v in f.items()} for f in dropin_runner.make_frames("flag", 12)]
torch.manual_seed(0)
model = FlagModel(dropin_runner.model_params("flag"))
model.eval()
with torch.no_grad():
    model(model.build_graph(frames[0], False))
net = model.learned_model
shapes = {k: tuple(v.shape) for k, v in net.state_dict().items()}
net.load_state_dict({k: v.to(dev) for k, v in synthetic.seeded_state_dict(shapes, 3).items()})
traj = {k: torch.stack([f[k] for f in frames]).unsqueeze(0) for k in frames[0]}
steps = len(frames)
before = ops.launch_count
with torch.no_grad():
    eager, _ = model.rollout({k: v[:steps] for k, v in traj.items()}, steps)
assert ops.launch_count > before
initial_state = {k: torch.squeeze(v, 0)[0] for k, v in traj.items()}
runner = FlagRolloutGraph(model, initial_state)
got = runner.rollout(steps)
ref = eager["pred_pos"]
assert got.shape == ref.shape, (got.shape, ref.shape)
diff = float((got - ref).abs().max())
assert torch.equal(got, ref), f"graphed rollout differs from the eager one by {diff:.3e}"
print("IO-ROLLOUT-OK", steps, "steps, bit-identical")
