"""The bf16 tcgen05 encoder and decoder MLPs (``ops.encoder_mlp`` / ``ops.decoder_mlp``, csrc/io_mlp_tc.cu) against torch fp32
arithmetic on bf16-rounded operands at the kernels' rounding points, their C ABI refusals, and the models with the switch
(``hgn_b200.set_io_kernels``) on: the golden cases in bf16, fp32 parity mode untouched, an empty edge set, off by default, the
reference's system models and the captured rollout / training iteration."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import GoldenCase, MODEL_CASES, ROOT, rel_err, rel_l2
from test_gpu_parity import GRAD_TOL, TOL, _MLP_NAMES, _param_errs, _report, _row_errs
from hgn_b200 import _cabi, config, ops, synthetic
from hgn_b200 import util as hutil
from hgn_b200.migration.encoder import Encoder
from hgn_b200.migration.meshgraphnet import MeshGraphNet

pytestmark = pytest.mark.gpu


def _sms():
    return torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count


ROWS = [0, 1, 127, 128, 129, "SMs x 128 + 1", 200000]
_rd = lambda t: t.to(torch.bfloat16).float()


def _rows(rows):
    return _sms() * 128 + 1 if rows == "SMs x 128 + 1" else rows


def _leaf(t):
    return t.cuda().requires_grad_(True)


def _encoder_params(k, seed):
    g = torch.Generator().manual_seed(seed)
    n = lambda *s: torch.randn(*s, generator=g)
    return [_leaf(n(128, k) / k ** 0.5), _leaf(0.1 * n(128)), _leaf(n(128, 128) / 128 ** 0.5), _leaf(0.1 * n(128)),
            _leaf(n(128, 128) / 128 ** 0.5), _leaf(0.1 * n(128)), _leaf(1 + 0.1 * n(128)), _leaf(0.1 * n(128))]


def _decoder_params(n_out, seed):
    g = torch.Generator().manual_seed(seed)
    n = lambda *s: torch.randn(*s, generator=g)
    return [_leaf(n(128, 128) / 128 ** 0.5), _leaf(0.1 * n(128)), _leaf(n(128, 128) / 128 ** 0.5), _leaf(0.1 * n(128)),
            _leaf(n(n_out, 128) / 128 ** 0.5), _leaf(0.1 * n(n_out))]


def _st(t):
    """bf16 rounding in the forward, the gradient passed through unrounded: the kernels keep the fp32 weight gradients and the
    encoder's fp32 raw-feature gradient."""
    return t + (_rd(t) - t).detach()


class _RoundGrad(torch.autograd.Function):
    """Identity whose gradient is rounded to bf16: the encoder's LayerNorm backward output dY, an MMA operand of the dgrad chain."""

    @staticmethod
    def forward(ctx, t):
        return t.view_as(t)

    @staticmethod
    def backward(ctx, g):
        return _rd(g)


def _hidden(x, w, taps=None):
    """Both ReLU layers at the kernels' rounding points: bf16 operands, fp32 sum + bias + ReLU, rounded to bf16 (and in the backward
    dH' = bf16(acc * [H > 0]), which is what the gradient of the rounding cast gives).  ``taps`` receives the first pre-activation."""
    W0, b0, W1, b1 = w[:4]
    pre0 = x @ _st(W0).t() + b0
    if taps is not None:
        pre0.retain_grad()
        taps.append(pre0)
    h = _rd(torch.relu(pre0))
    return _rd(torch.relu(h @ _st(W1).t() + b1))


def _encoder_emulation(x, w, taps=None):
    pre = _RoundGrad.apply(_hidden(_st(x), w, taps) @ _st(w[4]).t() + w[5])
    return torch.nn.functional.layer_norm(pre, (128,), w[6], w[7], 1e-5)


def _decoder_emulation(x, w):
    return _hidden(_rd(x), w) @ _st(w[4]).t() + w[5]         # the kernel rounds its input gradient to bf16


def _relu_edge_rows(x, w, rel=3e-4):
    """Rows whose hidden pre-activations (either layer) include one within ``rel`` x that layer's std of zero: kernel and emulation
    sum in different orders, so such a unit may switch on one side only; these rows get no upstream gradient (every gradient is
    linear in it, so both sides give exact zeros there), and the forward is still compared on every row."""
    W0, b0, W1, b1 = (p.detach() for p in w[:4])
    with torch.no_grad():
        pre1 = _rd(x) @ _rd(W0).t() + b0
        edge = (pre1.abs() < rel * pre1.std()).any(1)
        pre2 = _rd(torch.relu(pre1)) @ _rd(W1).t() + b1
        return edge | (pre2.abs() < rel * pre2.std()).any(1)


def _cancelled_rows(x, w, gup, rel=3e-3):
    """Rows whose raw-feature gradient dX = dH0' W0 cancels to below ``rel`` x the norm of its terms (sum_j |dH0'_j| |W0_jk|).  A bf16
    rounding of a dgrad value that falls the other way in the kernel than in the emulation (fp32 sums in another order) moves such a
    row by up to 2^-8 of one term, which is a large share of a nearly cancelled result -- a single-element window (K = 1, one row in the
    last tile) measures only that.  Like the rows on a ReLU edge these get no upstream gradient, so both sides give exact zeros there."""
    wr = [p.detach().clone().requires_grad_(True) for p in w]
    xf = x.detach().clone().requires_grad_(True)
    taps = []
    _encoder_emulation(xf, wr, taps).backward(gup.float())
    with torch.no_grad():
        scale = (taps[0].grad.abs() @ _rd(wr[0]).abs()).norm(dim=1)
        return (scale > 0) & (xf.grad.norm(dim=1) < rel * scale)


def _run_encoder(x, params, gup):
    out = ops.encoder_mlp(params, {}, x)
    out.backward(gup)
    grads = [p.grad.clone() for p in params]
    gx = x.grad.clone() if x.requires_grad else None
    for p in params:
        p.grad = None
    if x.requires_grad:
        x.grad = None
    return out.detach(), gx, grads


def _encoder_case(rows, k, want_grad_x=True, seed=0):
    torch.manual_seed(seed + 1000 * k + rows % 997)
    params = _encoder_params(k, seed + k)
    x = torch.randn(rows, k, device="cuda").requires_grad_(want_grad_x)
    gup = torch.randn(rows, 128, device="cuda").to(torch.bfloat16)
    edge = _relu_edge_rows(x.detach(), params) if rows else torch.zeros(0, dtype=torch.bool, device="cuda")
    gup[edge] = 0
    cancelled = _cancelled_rows(x, params, gup) if rows and want_grad_x else torch.zeros_like(edge)
    gup[cancelled] = 0
    edge = edge | cancelled
    out, gx, grads = _run_encoder(x, params, gup)
    out2, gx2, grads2 = _run_encoder(x, params, gup)                # two runs: bitwise identical
    assert torch.equal(out, out2) and all(torch.equal(a, b) for a, b in zip(grads, grads2))
    assert gx is None or torch.equal(gx, gx2)
    assert out.shape == (rows, 128) and out.dtype == torch.bfloat16
    assert [tuple(g.shape) for g in grads] == [tuple(p.shape) for p in params]
    if rows == 0:
        assert all(int(torch.count_nonzero(g)) == 0 for g in grads)
        return
    wr = [p.detach().clone().requires_grad_(True) for p in params]
    xf = x.detach().clone().requires_grad_(want_grad_x)
    ref = _encoder_emulation(xf, wr)
    ref.backward(gup.float())
    checks = {"out": (*_row_errs(out.float(), ref.detach(), rel_err), 1e-2)}
    if want_grad_x:
        assert int(torch.count_nonzero(gx[edge])) == 0
        checks["grad x"] = (*_row_errs(gx, xf.grad, rel_l2), 1e-2)
    for p, g in zip(params, grads):
        p.grad = g
    err, name = _param_errs(params, wr, _MLP_NAMES)
    checks[f"weights (worst {name})"] = (err, 0.0, 1.5e-2)
    _report(f"encoder kernel, K={k}, {rows} rows ({int(edge.sum())} rows on a ReLU edge or with a cancelled dX: {int(cancelled.sum())})", checks)


@pytest.mark.parametrize("rows", ROWS)
@pytest.mark.parametrize("k", [1, 3, 5, 7, 8, 9, 16, 17, 128])
def test_encoder_kernel_vs_bf16_emulation(k, rows):
    _encoder_case(_rows(rows), k)


def test_encoder_kernel_cfg5_edges_vs_bf16_emulation():
    """The cfg5 mesh-edge encoder: 5 992 002 rows of K = 7 (three backward passes of 2 M rows), raw-feature gradient not requested."""
    _encoder_case(5992002, 7, want_grad_x=False)


def _run_decoder(x, params, gup):
    out = ops.decoder_mlp(params, {}, x)
    out.backward(gup)
    grads = [p.grad.clone() for p in params]
    gx = x.grad.clone()
    for p in params:
        p.grad = None
    x.grad = None
    return out.detach(), gx, grads


@pytest.mark.parametrize("rows", ROWS)
@pytest.mark.parametrize("n_out", [1, 2, 3, 16])
def test_decoder_kernel_vs_bf16_emulation(n_out, rows):
    rows = _rows(rows)
    torch.manual_seed(n_out + rows % 991)
    params = _decoder_params(n_out, n_out)
    x = torch.randn(rows, 128, device="cuda").to(torch.bfloat16).requires_grad_(True)
    gup = torch.randn(rows, n_out, device="cuda")
    edge = _relu_edge_rows(x.detach().float(), params) if rows else torch.zeros(0, dtype=torch.bool, device="cuda")
    gup[edge] = 0
    out, gx, grads = _run_decoder(x, params, gup)
    out2, gx2, grads2 = _run_decoder(x, params, gup)
    assert torch.equal(out, out2) and torch.equal(gx, gx2) and all(torch.equal(a, b) for a, b in zip(grads, grads2))
    assert out.shape == (rows, n_out) and out.dtype == torch.float32 and gx.dtype == torch.bfloat16
    assert [tuple(g.shape) for g in grads] == [tuple(p.shape) for p in params]
    if rows == 0:
        assert all(int(torch.count_nonzero(g)) == 0 for g in grads)
        return
    wr = [p.detach().clone().requires_grad_(True) for p in params]
    xf = x.detach().float().requires_grad_(True)
    ref = _decoder_emulation(xf, wr)
    ref.backward(_rd(gup))                                        # the kernel rounds the upstream gradient to bf16
    assert int(torch.count_nonzero(gx[edge])) == 0
    checks = {"out": (*_row_errs(out, ref.detach(), rel_err), 1e-2),
              "grad x": (*_row_errs(gx.float(), xf.grad, rel_l2), 1e-2)}
    for p, g in zip(params, grads):
        p.grad = g
    err, name = _param_errs(params, wr, _MLP_NAMES[:6])
    checks[f"weights (worst {name})"] = (err, 0.0, 1.5e-2)
    _report(f"decoder kernel, n_out={n_out}, {rows} rows ({int(edge.sum())} rows on a ReLU edge)", checks)


def test_io_kernels_refuse_out_of_range_arguments():
    lib = _cabi.load()
    st = _cabi.stream_ptr()
    rows = 300
    enc = [p.detach() for p in _encoder_params(5, 1)]
    dec = [p.detach() for p in _decoder_params(3, 1)]
    blob = torch.empty(lib.hgn_io_mlp_packed_bytes(), dtype=torch.uint8, device="cuda")
    p = lambda t: t.data_ptr()
    for kind, width in ((_cabi.HGN_IO_ENCODER, 0), (_cabi.HGN_IO_ENCODER, 129), (_cabi.HGN_IO_DECODER, 0), (_cabi.HGN_IO_DECODER, 17), (2, 3)):
        assert lib.hgn_io_mlp_pack(kind, width, *map(p, enc), p(blob), st) == -1
    assert lib.hgn_io_mlp_pack(_cabi.HGN_IO_DECODER, 3, *map(p, dec), None, None, p(blob), st) == 0
    assert lib.hgn_io_mlp_pack(_cabi.HGN_IO_ENCODER, 5, *map(p, enc[:6]), None, None, p(blob), st) == -1    # encoder needs gamma / beta
    assert lib.hgn_io_mlp_pack(_cabi.HGN_IO_ENCODER, 5, *map(p, enc), p(blob), st) == 0
    x = torch.randn(rows, 5, device="cuda")
    xb = torch.randn(rows, 128, device="cuda").to(torch.bfloat16)
    out_b = torch.empty(rows, 128, dtype=torch.bfloat16, device="cuda")
    out_f = torch.empty(rows, 17, device="cuda")
    for k in (0, 129):
        assert lib.hgn_encoder_forward(rows, k, p(x), p(blob), p(out_b), st) == -1
        assert lib.hgn_encoder_backward_workspace_bytes(rows, k) == 0
    for n in (0, 17):
        assert lib.hgn_decoder_forward(rows, n, p(xb), p(blob), p(out_f), st) == -1
        assert lib.hgn_decoder_backward_workspace_bytes(rows, n) == 0
    gW = [torch.empty(128, 128, device="cuda") for _ in range(3)]
    gv = [torch.empty(128, device="cuda") for _ in range(5)]
    gparams = [p(gW[0]), p(gv[0]), p(gW[1]), p(gv[1]), p(gW[2]), p(gv[2])]
    ws_e = lib.hgn_encoder_backward_workspace_bytes(rows, 5)
    ws_d = lib.hgn_decoder_backward_workspace_bytes(rows, 3)
    ws = torch.empty(max(ws_e, ws_d), dtype=torch.uint8, device="cuda")
    go_b = torch.randn(rows, 128, device="cuda").to(torch.bfloat16)
    go_f = torch.randn(rows, 3, device="cuda")
    gx_b = torch.empty_like(xb)
    assert lib.hgn_encoder_backward(rows, 5, p(x), p(blob), p(go_b), None, *gparams, p(gv[3]), p(gv[4]), p(ws), ws_e - 1, st) == -4
    assert lib.hgn_encoder_backward(rows, 5, p(x), p(blob), None, None, *gparams, p(gv[3]), p(gv[4]), p(ws), ws_e, st) == -1
    assert lib.hgn_encoder_backward(rows, 5, p(x), p(blob), p(go_b), None, *gparams, None, p(gv[4]), p(ws), ws_e, st) == -1
    assert lib.hgn_decoder_backward(rows, 3, p(xb), p(blob), p(go_f), p(gx_b), *gparams, p(ws), ws_d - 1, st) == -4
    assert lib.hgn_decoder_backward(rows, 3, p(xb), p(blob), p(go_f), None, *gparams, p(ws), ws_d, st) == -1
    assert lib.hgn_decoder_backward(rows, 3, p(xb), p(blob), p(go_f), p(gx_b), *gparams[:5], None, p(ws), ws_d, st) == -1
    assert "decoder_backward" in lib.hgn_last_error().decode()
    torch.cuda.synchronize()


# ---- models ---------------------------------------------------------------------------------------------------------------
def _golden_model(case, precision, kernels):
    m = MeshGraphNet(3, 128, 2, case.meta["aggregation"], case.meta["steps"], case.meta["architecture"], case.meta["edge_sets"])
    m.load_state_dict(case.weights())
    m = m.cuda()
    m.processor.precision = m.encoder.precision = m.decoder.precision = precision
    m.encoder.kernels = m.decoder.kernels = kernels
    return m


def _golden_run(case, m):
    g = case.graph(hutil.MultiGraph, hutil.EdgeSet, device="cuda", requires_grad=True)
    out = m(g)
    coef = synthetic.seeded_tensor("loss_coef", out.shape, 3).cuda()
    (out * coef).sum().backward()
    grads = [nf.grad for nf in g.node_features] + [es.features.grad for es in g.edge_sets]
    return out.detach(), grads, {k: (p.grad.clone() if p.grad is not None else None) for k, p in m.named_parameters()}


# Raw-feature gradients against the fp32 reference.  With the torch encoder the bf16 golden test measures up to 0.279 (GRAD_TOL's
# derivation: ReLU units that switch within bf16 rounding of zero); the encoder kernel also rounds X, W0 and H0 to bf16 and returns the
# gradient through one more bf16 dgrad, so more units switch: measured on one B200 (1000 W) up to 0.305 (hgn_multiscale_sum_L1).
# The kernels' own arithmetic is pinned at 1e-2 by the emulation tests above; parameter gradients keep GRAD_TOL.
INPUT_GRAD_TOL = 4e-1


@pytest.mark.parametrize("name", MODEL_CASES)
def test_golden_models_bf16_with_io_kernels(name):
    """The golden cases in bf16 with the encoder and decoder kernels: output within the bf16 golden bound, input and parameter gradients
    at the bounds of the bf16 golden test (test_gpu_parity.test_model_matches_reference_golden)."""
    case = GoldenCase(name)
    m = _golden_model(case, "bf16", True)
    before = ops.launch_count
    g = case.graph(hutil.MultiGraph, hutil.EdgeSet, device="cuda", requires_grad=True)
    latent = m.encoder(g)
    assert all(t.dtype == torch.bfloat16 for t in latent.node_features) and all(es.features.dtype == torch.bfloat16 for es in latent.edge_sets)
    assert [es.name for es in latent.edge_sets] == [es.name for es in g.edge_sets if es.name in m.encoder.edge_models]
    latent = m.processor(latent)
    out = m.decoder(latent._replace(node_features=latent.node_features[0]))
    assert out.dtype == torch.float32 and ops.launch_count > before
    err = rel_err(out, case.arr("output"))
    coef = synthetic.seeded_tensor("loss_coef", out.shape, 3).cuda()
    (out * coef).sum().backward()
    worst = 0.0
    for i, nf in enumerate(g.node_features):
        worst = max(worst, rel_l2(nf.grad, case.arr(f"grad_node_features_{i}")))
    for es in g.edge_sets:
        key = f"grad_edge_{es.name}_features"
        if key in case.z:
            worst = max(worst, rel_l2(es.features.grad, case.arr(key)))
    print(f"\nio kernels [{name}]: output {err:.3e} (bound {TOL['bf16']:.0e}), input gradients relative L2 {worst:.3e} (bound {INPUT_GRAD_TOL:.0e})")
    assert err < TOL["bf16"] and worst < INPUT_GRAD_TOL
    gtol = GRAD_TOL["bf16"]
    params = dict(m.named_parameters())
    for key, ref in case.meta["grad_proj"].items():
        gflat = params[key].grad.double().reshape(-1).cpu()
        norm = ref[-1]
        assert abs(float(gflat.norm()) - norm) <= gtol * max(norm, 1e-6), key
        for i, val in enumerate(ref[:-1]):
            proj = float(torch.dot(gflat, synthetic.seeded_tensor(f"proj{i}:{key}", gflat.shape, 11).double()))
            assert abs(proj - val) <= gtol * max(norm * np.sqrt(gflat.numel()), 1e-6), (key, i)


@pytest.mark.parametrize("name", MODEL_CASES)
def test_fp32_parity_mode_ignores_the_switch(name):
    case = GoldenCase(name)
    out_a, grads_a, params_a = _golden_run(case, _golden_model(case, "fp32", True))
    out_b, grads_b, params_b = _golden_run(case, _golden_model(case, "fp32", False))
    same = lambda a, b: (a is None and b is None) or (a is not None and b is not None and torch.equal(a, b))
    assert torch.equal(out_a, out_b)
    assert all(same(a, b) for a, b in zip(grads_a, grads_b))
    assert all(same(params_a[k], params_b[k]) for k in params_b)


def test_empty_world_edges_with_io_kernels():
    """A frame without contact: the world-edge set has no rows; its latents are empty and its MLP's gradients exactly zero."""
    enc = Encoder(MeshGraphNet(3, 128, 2, "sum", 1, "none", ["mesh_edges"])._make_mlp, 128, ["mesh_edges", "world_edges"], hierarchical=False)
    enc = enc.cuda()
    enc.precision, enc.kernels = "bf16", True
    s, r = synthetic.grid_edges_two_way(6, 5)
    g = hutil.MultiGraph([torch.randn(30, 9, device="cuda")],
                         [hutil.EdgeSet("mesh_edges", torch.randn(s.shape[0], 7, device="cuda"), s.cuda(), r.cuda()),
                          hutil.EdgeSet("world_edges", torch.zeros(0, 4, device="cuda"), s[:0].cuda(), r[:0].cuda())])
    out = enc(g)
    world = out.edge_sets[1].features
    assert world.shape == (0, 128) and world.dtype == torch.bfloat16
    (out.node_features[0].float().sum() + out.edge_sets[0].features.float().sum() + world.float().sum()).backward()
    for name, p in enc.edge_models["world_edges"].named_parameters():
        assert p.grad is not None and int(torch.count_nonzero(p.grad)) == 0, name
    assert all(int(torch.count_nonzero(p.grad)) > 0 for p in enc.edge_models["mesh_edges"].parameters())


def test_io_kernels_are_off_by_default():
    """With the switch unset a bf16 MeshGraphNet step runs none of the encoder / decoder kernels; switched on, it runs both."""
    from torch.profiler import ProfilerActivity, profile
    assert config.io_kernels() is False or os.environ.get("HGN_B200_IO_KERNELS")
    case = GoldenCase("mgn_sum_L2")

    def kernel_names(kernels):
        m = _golden_model(case, "bf16", kernels)
        g = case.graph(hutil.MultiGraph, hutil.EdgeSet, device="cuda", requires_grad=True)
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            m(g).sum().backward()
            torch.cuda.synchronize()
        return [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]

    saved = config._io_kernels
    try:
        config.set_io_kernels(False)
        assert not any("io_mlp_tc_kernel" in n for n in kernel_names(None))
        config.set_io_kernels(True)
        on = {n.split("(")[0] for n in kernel_names(None) if "io_mlp_tc_kernel" in n}
        assert len(on) == 4, on                                                     # encoder + decoder, forward + backward
    finally:
        config._io_kernels = saved


# ---- the reference's system models (need the reference tree) --------------------------------------------------------------
def _needs_reference():
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import reference_shim
    if not reference_shim.available():
        pytest.skip("no reference tree: neither /root/reference nor oracle/_ref (run oracle/make_ref.sh in the build container)")


def test_graphed_training_iteration_with_io_kernels(tmp_path):
    """FlagTrainingGraph follows the eager loop over ten Adam steps with the encoder / decoder kernels, as it does without them."""
    _needs_reference()
    out = str(tmp_path / "tg.npz")
    run = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "training_graph_worker.py"), "bf16", out], capture_output=True, text=True,
                         timeout=900, env=dict(os.environ, WANDB_MODE="disabled", HGN_B200_IO_KERNELS="1"))
    assert run.returncode == 0 and "TRAINING-GRAPH-OK" in run.stdout, run.stdout[-3000:] + run.stderr[-5000:]
    z = np.load(out)
    eager, graphed, frozen = z["eager"], z["graphed"], z["frozen"]
    assert abs(graphed[0] - eager[0]) <= 2e-3 * abs(eager[0])
    for k in range(1, len(eager)):
        moved = abs(eager[k] - frozen[k])
        assert abs(graphed[k] - eager[k]) <= max(0.1 * moved, 5e-3 * abs(eager[k])), (k, graphed[k], eager[k], frozen[k])
    assert float(z["weight_gap"]) <= 0.1 * float(z["weight_move"])


def test_graphed_rollout_with_io_kernels_is_bit_identical_to_eager():
    _needs_reference()
    run = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "io_rollout_worker.py")], capture_output=True, text=True, timeout=900,
                         env=dict(os.environ, WANDB_MODE="disabled", HGN_B200_IO_KERNELS="1"))
    assert run.returncode == 0 and "IO-ROLLOUT-OK" in run.stdout, run.stdout[-3000:] + run.stderr[-5000:]


@pytest.mark.parametrize("case", ("flag", "plate", "cylinder", "flag_hyper"))
def test_reference_system_model_with_io_kernels(case, tmp_path):
    """training_step + rollout of the reference's own models on the installed modules with HGN_B200_IO_KERNELS=1 against the reference
    on the CPU, within the bf16 bounds of test_dropin_gpu."""
    _needs_reference()
    from test_dropin_gpu import RUNNER, TOL as DROPIN_TOL
    env = dict(os.environ, WANDB_MODE="disabled", PYTHONHASHSEED="0")
    ref_path = str(tmp_path / f"reference_{case}.npz")
    ref_env = dict(env, CUDA_VISIBLE_DEVICES="", OMP_NUM_THREADS="4")
    run = subprocess.run([sys.executable, RUNNER, "reference", case, ref_path], env=ref_env, capture_output=True, text=True, timeout=1500)
    assert run.returncode == 0 and "DROPIN-RUNNER-OK" in run.stdout, run.stdout[-4000:]
    ours_path = str(tmp_path / f"ours_{case}.npz")
    run = subprocess.run([sys.executable, RUNNER, "ours", case, ours_path, "bf16", ref_path], env=dict(env, HGN_B200_IO_KERNELS="1"),
                         capture_output=True, text=True, timeout=1500)
    assert run.returncode == 0 and "DROPIN-RUNNER-OK" in run.stdout, run.stdout[-3000:] + run.stderr[-5000:]
    ref, ours = dict(np.load(ref_path)), dict(np.load(ours_path))
    tol = DROPIN_TOL["bf16"]
    loss_err = abs(ours["losses"][0] - ref["losses"][0]) / abs(ref["losses"][0])
    total = float(np.sqrt((ref["grad_norms"] ** 2).sum()))
    total_err = float(np.abs((ours["grad_projs"] - ref["grad_projs"]).sum(0)).max() / total)
    loss2_err = abs(ours["losses"][1] - ref["losses"][1]) / abs(ref["losses"][1])
    travelled = np.abs(ref["rollout_pred"] - ref["rollout_pred"][:1]).max()
    roll_err = float(np.abs(ours["rollout_pred"] - ref["rollout_pred"]).max() / max(travelled, 1e-12))
    print(f"\ndropin io kernels [{case}]: loss {loss_err:.2e} grad(total) {total_err:.2e} loss_after_adam {loss2_err:.2e} rollout {roll_err:.2e}")
    assert loss_err < tol["loss"] and total_err < tol["grad_total"] and loss2_err < tol["loss2"] and roll_err < tol["rollout"]
