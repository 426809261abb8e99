"""The fp32 parity mode of the fused MLP tile (``csrc/mlp_f32.cu``: FFMA register tiles of 64 rows, a separate weight-gradient kernel,
the backward in slabs of 2^19 rows) against float64, through ``ops.fused_mlp`` and through the C ABI (``-m gpu``).

Reference: the oracle's own functions (``orc.edge_update``, ``orc.mlp``) on float64 copies of the same fp32 inputs, fp32 weights and fp32
upstream gradient, on the GPU.  Every bound is in the max metric max|a - b| / max|b| against float64: outputs 1e-5 (the fp32 parity bar
of include/hgn_b200.h), data gradients and every parameter gradient 5e-5 (``GRAD_TOL["fp32"]`` of tests/test_gpu_parity.py).  Held
in the max metric at every size, a defect confined to one row cannot hide in a norm.

A hidden unit whose pre-activation lies within fp32 noise of zero may take the other ReLU branch in the kernel than in float64, which
moves that row's gradient by O(10 %) (tests/test_scale_gpu.py: GRAD_L2).  Rows with a unit within ``RELU_EDGE`` x that layer's std of
zero, the pre-activations taken in float64, get no upstream gradient: every gradient is linear in it, so both sides are exactly zero
there (checked).  The forward is continuous and is compared on every row.
"""
import ctypes

import pytest
import torch
import torch.nn.functional as F

import hgn_oracle as orc
from hgn_b200 import _cabi, ops, synthetic
from hgn_b200.plan import segment_plan
from test_gpu_parity import _MLP_NAMES, _mlp_params, _random_mlp_weights, _report

pytestmark = pytest.mark.gpu

# Measured on one B200 (1000 W power limit), worst over all cases: outputs 1.1e-6, data gradients 1.4e-6, parameter gradients 2.1e-6
# (2^19 + 1 edges; 2.05e-6 at 1.5 M edges, where each of the 64 parts of a slab sums 8 192 rows in sequence).
OUT_TOL, GRAD_TOL = 1e-5, 5e-5
# About 100 x the fp32 error of a K <= 3072 dot product relative to its std (an estimate); masks about 2 % of the rows
# (256 hidden units x a window of 2e-4 sigma x a density of 0.4 at zero; measured 1.9 - 2.1 % on every case of 16 384 rows or more).
RELU_EDGE = 1e-4
SLAB = 1 << 19                      # rows per backward pass of csrc/mlp_f32.cu (bwd_layout_f32)
HGN_ERR_INVALID_ARGUMENT, HGN_ERR_WORKSPACE = -1, -4


def _max_rel(got, want):
    """conftest.rel_err, computed on the device: the tensors here reach 1.5 M x 128."""
    g, w = got.detach().double(), want.detach().double()
    return float((g - w).abs().max() / w.abs().max().clamp_min(1e-30))


def _f64_weights(w, prefix):
    """float64 leaves on the GPU of the weights ``w`` of ``_random_mlp_weights`` (keys ``m.*``) under the oracle key ``prefix``, and the same
    tensors in the kernels' parameter order."""
    w64 = {prefix + k[1:]: t.cuda().double().requires_grad_(True) for k, t in w.items()}
    order = [f"{prefix}.0.layers.linear_{k}.{p}" for k in range(3) for p in ("weight", "bias")] + [f"{prefix}.1.weight", f"{prefix}.1.bias"]
    return w64, [w64[k] for k in order]


def _relu_edge_rows(x64, p64):
    """(rows with a float64 hidden pre-activation, of either layer, within RELU_EDGE x that layer's std of zero; for every row the distance
    of its closest unit from zero in those units)."""
    W0, b0, W1, b1 = (p.detach() for p in p64[:4])
    with torch.no_grad():
        pre1 = F.linear(x64, W0, b0)
        pre2 = F.linear(torch.relu(pre1), W1, b1)
        closest = torch.minimum(pre1.abs().min(1).values / pre1.std(), pre2.abs().min(1).values / pre2.std())
    return closest < RELU_EDGE, closest


def _row_checks(checks, name, got, want, bound, closest):
    """Add a row-indexed tensor to ``checks``; beyond the bound, print its worst row and that row's unit closest to a ReLU edge."""
    err = _max_rel(got, want)
    checks[name] = (err, 0.0, bound)
    if not err < bound:
        diff = (got.detach().double() - want.detach().double()).abs().amax(1)
        row = int(diff.argmax())
        print(f"\n{name}: worst row {row}, {float(diff[row]) / float(want.detach().abs().max()):.3e} of the tensor's max; its hidden unit "
              f"closest to zero lies {float(closest[row]):.3e} sigma from it (masked below {RELU_EDGE:g})")


def _param_checks(checks, grads, p64):
    """Add the worst of the eight parameter gradients ``grads`` to ``checks``."""
    err, name = max((_max_rel(g, p.grad), n) for g, p, n in zip(grads, p64, _MLP_NAMES))
    checks[f"weights (worst {name})"] = (err, 0.0, GRAD_TOL)


def _assert_bitwise(a, b, what):
    assert torch.equal(a.view(torch.int32), b.view(torch.int32)), what


# ------------------------------------------------------------------------------------------------------------------------------------
# edge update: [v[s] | v[r] | e], residual e (GraphNet._update_edge_features in fp32)
# ------------------------------------------------------------------------------------------------------------------------------------
GRID = (1000, 250)                  # bench.py's fp32 leg: 1 495 002 edges, three backward slabs, the last one partial

# rows straddle the 64-row tile (1, 63, 64, 65), the 32-row staging of the weight-gradient kernel (33, 257: two parts of 160 rows), the
# change from ceil(slab / 256) parts to 64 (16383 .. 16385), and the 2^19 slab (the second slab of 2^19 + 1 has one row); more nodes
# than edges below the slab size, so that some nodes have no incident edge (at n = rows about 13 % still have none)
_EDGE_CASES = [(1, 5), (33, 100), (63, 100), (64, 100), (65, 100), (257, 400), (16383, 20000), (16384, 20000), (16385, 20000),
               (SLAB - 1, SLAB), (SLAB, SLAB), (SLAB + 1, SLAB), ("grid", GRID[0] * GRID[1])]


@pytest.mark.parametrize("rows,n_nodes", _EDGE_CASES)
def test_fp32_edge_update_vs_float64(rows, n_nodes):
    """ops.fused_mlp called as GraphNet._update_edge_features calls it in fp32, against orc.edge_update in float64: e', the gradients of
    v and e and of every parameter.  Masked rows have an exactly zero gradient of e, nodes without an incident edge an exactly zero
    gradient of v.  The grid (the largest case) runs twice and must be bit-identical."""
    grid = rows == "grid"
    if grid:
        s, r = (t.cuda() for t in synthetic.grid_edges_two_way(*GRID))
        rows = s.numel()
        assert rows == 1_495_002
    torch.manual_seed(rows)
    if not grid:
        s, r = (torch.randint(0, n_nodes, (rows,), device="cuda") for _ in range(2))
    w = _random_mlp_weights(3, 5)
    v0, e0 = torch.randn(n_nodes, 128, device="cuda"), torch.randn(rows, 128, device="cuda")
    gup = torch.randn(rows, 128, device="cuda")

    w64, p64 = _f64_weights(w, "blk.edge_models.mesh_edges")
    v64, e64 = v0.double().requires_grad_(True), e0.double().requires_grad_(True)
    edge, closest = _relu_edge_rows(torch.cat([v64.detach()[s], v64.detach()[r], e64.detach()], -1), p64)
    gup[edge] = 0
    ref = orc.edge_update(w64, "blk", [v64], orc.EdgeSet("mesh_edges", e64, s, r))
    ref.backward(gup.double())
    ref = ref.detach()

    sp, rp = segment_plan(s, n_nodes), segment_plan(r, n_nodes)
    runs = []
    for _ in range(2 if grid else 1):
        params = _mlp_params(w)
        v, e = v0.clone().requires_grad_(True), e0.clone().requires_grad_(True)
        out = ops.fused_mlp(params, {}, [v, e], [ops.ChunkSpec(0, sp), ops.ChunkSpec(0, rp), ops.ChunkSpec(1)], rows, resid_source=1)
        out.backward(gup)
        runs.append([out.detach(), v.grad, e.grad] + [p.grad for p in params])
    if grid:                            # fp32 mode is bit-for-bit reproducible (DESIGN.md), here over three slabs
        for a, b, name in zip(*runs, ["e'", "grad v", "grad e"] + _MLP_NAMES):
            _assert_bitwise(a, b, f"two runs differ: {name}")
    out, v_grad, e_grad = runs[-1][:3]

    assert int(torch.count_nonzero(e_grad[edge])) == 0, "masked rows of grad e"
    isolated = (torch.bincount(s, minlength=n_nodes) + torch.bincount(r, minlength=n_nodes)) == 0
    assert grid or bool(isolated.any())
    assert int(torch.count_nonzero(v_grad[isolated])) == 0, "grad v of nodes without an incident edge"
    checks = {}
    _row_checks(checks, "e'", out, ref, OUT_TOL, closest)
    _row_checks(checks, "grad e", e_grad, e64.grad, GRAD_TOL, closest)
    checks["grad v"] = (_max_rel(v_grad, v64.grad), 0.0, GRAD_TOL)
    _param_checks(checks, [p.grad for p in params], p64)
    _report(f"fp32 edge update, {rows} edges / {n_nodes} nodes ({float(edge.double().mean()):.2%} of the rows on a ReLU edge, "
            f"{int(isolated.sum())} nodes without an edge)", checks)
    del runs, ref, v64, e64, w64, p64
    torch.cuda.empty_cache()


# ------------------------------------------------------------------------------------------------------------------------------------
# node updates: [v_stacked] + aggregates, dense at the target's row offset, residual from v_stacked (GraphNet._fused_node_update in fp32)
# ------------------------------------------------------------------------------------------------------------------------------------
def _node_update_vs_float64(n_chunks, target, n_mesh, n_hyper, agg_grad):
    """Sources [v_stacked] + aggregates, each of n_mesh + n_hyper rows; the target's rows are the mesh rows (offset 0) or the hyper rows
    (offset n_mesh).  Against v + orc.mlp([v | agg_1 | ...]) in float64 on the target's rows; the source gradients are exactly zero
    outside them and on the masked rows, an aggregate without requires_grad leaves its grad_chunk entry NULL."""
    torch.manual_seed(1000 * n_chunks + n_mesh + n_hyper + (target == "hyper"))
    offset, rows = (0, n_mesh) if target == "mesh" else (n_mesh, n_hyper)
    w = _random_mlp_weights(n_chunks, 9)
    params = _mlp_params(w)
    srcs = [torch.randn(n_mesh + n_hyper, 128, device="cuda").requires_grad_(c == 0 or agg_grad) for c in range(n_chunks)]
    gup = torch.randn(rows, 128, device="cuda")

    w64, p64 = _f64_weights(w, "m")
    sf = [t.detach()[offset: offset + rows].double().requires_grad_(True) for t in srcs]
    x64 = torch.cat(sf, -1)
    edge, closest = _relu_edge_rows(x64.detach(), p64)
    gup[edge] = 0
    ref = sf[0] + orc.mlp(w64, "m", x64)
    ref.backward(gup.double())
    ref = ref.detach()
    del x64

    out = ops.fused_mlp(params, {}, srcs, [ops.ChunkSpec(c, None, offset) for c in range(n_chunks)], rows, resid_source=0,
                        resid_offset=offset)
    out.backward(gup)
    checks = {}
    _row_checks(checks, "out", out, ref, OUT_TOL, closest)
    for c, (t, f) in enumerate(zip(srcs, sf)):
        if not (c == 0 or agg_grad):
            assert t.grad is None
            continue
        g = t.grad
        outside = int(torch.count_nonzero(g[:offset])) + int(torch.count_nonzero(g[offset + rows:]))
        assert outside == 0, f"source {c}: {outside} gradient entries written outside the target's rows"
        g = g[offset: offset + rows]
        assert int(torch.count_nonzero(g[edge])) == 0, f"masked rows of source {c}"
        _row_checks(checks, f"grad src{c}", g, f.grad, GRAD_TOL, closest)
    _param_checks(checks, [p.grad for p in params], p64)
    _report(f"fp32 node update, {n_chunks} chunks, {target} rows {rows} at offset {offset}"
            f"{'' if agg_grad else ', aggregates without gradient'} ({float(edge.double().mean()):.2%} of the rows on a ReLU edge)", checks)


# chunk counts: 2 / 5 = 'sum' / 'pna' over one set (in fp32 these go through the tile kernels too), 3 = 'sum' over two sets, 6 = 'sum' over
# five, 9 = hyper 'pna' over two inter sets, 13 = 'pna' over three, 21 = hetero 'pna' over five sets, 24 = HGN_MAX_CHUNKS
_NODE_LAYOUTS = [(k, t, n, c, True) for k in (2, 3, 5, 6, 9, 13, 21, 24) for t in ("mesh", "hyper") for n, c in ((1600, 16), (40000, 200))]
_NODE_LAYOUTS += [(2, "mesh", 1600, 16, False), (9, "hyper", 1600, 16, False), (21, "mesh", 40000, 200, False)]


@pytest.mark.parametrize("n_chunks,target,n_mesh,n_hyper,agg_grad", _NODE_LAYOUTS)
def test_fp32_node_update_layouts_vs_float64(n_chunks, target, n_mesh, n_hyper, agg_grad):
    _node_update_vs_float64(n_chunks, target, n_mesh, n_hyper, agg_grad)


@pytest.mark.parametrize("n_chunks,target,n_mesh,n_hyper", [(5, "mesh", SLAB + 401, 16), (3, "hyper", 33_333, SLAB + 97)])
def test_fp32_node_update_multi_slab_vs_float64(n_chunks, target, n_mesh, n_hyper):
    """Two backward slabs, the second partial: the weight-gradient partials and the LayerNorm partials accumulated over slabs.  The hyper
    target of more than 2^19 rows at an odd row offset meets the slab offset in the backward kernel and in the weight-gradient gather."""
    _node_update_vs_float64(n_chunks, target, n_mesh, n_hyper, True)
    torch.cuda.empty_cache()


# ------------------------------------------------------------------------------------------------------------------------------------
# the C ABI: hgn_mlp_forward / hgn_mlp_backward with HGN_F32
# ------------------------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("rows", [1, 1000, SLAB + 1])
def test_fp32_mlp_cabi_contract(rows):
    """hgn_mlp_forward / hgn_mlp_backward called directly on [v[s] | v[r] | e[7 + row]], the residual e at row offset 7:
    * output and gradients against float64;
    * resid_chunk = 2 against -1: chunk 2 is the fp32 sum of the first run's chunk 2 and grad_out bit for bit (the kernel adds grad_out
      once to the same GEMM result), every other output bit-identical;
    * grad_chunk NULL as a whole array, or NULL for chunks 0 and 2: what is still written is bit-identical;
    * a workspace one byte short returns HGN_ERR_WORKSPACE and writes nothing;
    * n_chunks 0 and 25 are refused by every entry point, which write nothing."""
    lib, f32, st = _cabi.load(), _cabi.HGN_F32, _cabi.stream_ptr()
    torch.manual_seed(rows)
    n_nodes, off = rows + 3, 7
    w = _random_mlp_weights(3, 5)
    params = _mlp_params(w)
    packed = ops._pack_weights({}, torch.float32, 3, params)
    s, r = (torch.randint(0, n_nodes, (rows,), device="cuda", dtype=torch.int32) for _ in range(2))
    v = torch.randn(n_nodes, 128, device="cuda")
    e = torch.randn(off + rows + 5, 128, device="cuda")
    gup = torch.randn(rows, 128, device="cuda")

    w64, p64 = _f64_weights(w, "m")
    x64 = torch.cat([v[s.long()], v[r.long()], e[off: off + rows]], -1).double().requires_grad_(True)
    edge, closest = _relu_edge_rows(x64.detach(), p64)
    gup[edge] = 0
    ref = x64.detach()[:, 256:] + orc.mlp(w64, "m", x64)
    ref.backward(gup.double())

    ch = _cabi.Chunks()
    ch.n_chunks = 3
    for c, (src, idx, ro) in enumerate(((v, s, 0), (v, r, 0), (e, None, off))):
        ch.src[c], ch.idx[c], ch.row_offset[c] = src.data_ptr(), _cabi.ptr(idx), ro
    nan = lambda *shape: torch.full(shape, float("nan"), device="cuda")
    out = nan(rows, 128)
    _cabi.check(lib.hgn_mlp_forward(f32, rows, ctypes.byref(ch), packed.data_ptr(), e.data_ptr(), off, out.data_ptr(), st),
                "hgn_mlp_forward")
    ws_bytes = lib.hgn_mlp_backward_workspace_bytes(f32, rows, 3)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device="cuda")

    def backward(resid_chunk, which=(0, 1, 2), nbytes=ws_bytes, chunks=ch):
        """(grad_chunk buffers, None where NULL; the eight parameter gradients, return code); every buffer NaN-filled before the call."""
        bufs = [nan(rows, 128) if which is not None and c in which else None for c in range(3)]
        gparams = [nan(*p.shape) for p in params]
        gptrs = None if which is None else (ctypes.c_void_p * 3)(*[_cabi.ptr(b) for b in bufs])
        rc = lib.hgn_mlp_backward(f32, rows, ctypes.byref(chunks), packed.data_ptr(), gup.data_ptr(), resid_chunk, gptrs,
                                  *[g.data_ptr() for g in gparams], ws.data_ptr(), nbytes, st)
        return bufs, gparams, rc

    first, gp_first, rc = backward(-1)
    assert rc == _cabi.HGN_OK
    second, gp_second, rc = backward(2)
    assert rc == _cabi.HGN_OK
    checks = {}
    _row_checks(checks, "out", out, ref, OUT_TOL, closest)
    for c in range(3):
        want = x64.grad[:, 128 * c: 128 * (c + 1)] + (gup.double() if c == 2 else 0.0)
        _row_checks(checks, f"grad chunk {c}", second[c], want, GRAD_TOL, closest)
        masked = int(torch.count_nonzero(second[c][edge])) + int(torch.count_nonzero(first[c][edge]))
        assert masked == 0, f"masked rows of chunk {c}"
    _param_checks(checks, gp_second, p64)
    _report(f"fp32 C ABI, {rows} rows ({float(edge.double().mean()):.2%} of the rows on a ReLU edge)", checks)

    _assert_bitwise(second[2], first[2] + gup, "resid_chunk = 2: chunk 2 != first + grad_out")
    for c in (0, 1):
        _assert_bitwise(second[c], first[c], f"resid_chunk = 2 changed chunk {c}")
    for which in (None, (1,)):
        bufs, gps, rc = backward(2, which=which)
        assert rc == _cabi.HGN_OK
        for a, b, name in zip(gps, gp_first, _MLP_NAMES):
            _assert_bitwise(a, b, f"grad_chunk {which or 'NULL'}: grad {name} differs")
    _assert_bitwise(bufs[1], first[1], "grad_chunk NULL for chunks 0 and 2: chunk 1 differs")

    bufs, gps, rc = backward(2, nbytes=ws_bytes - 1)
    assert rc == HGN_ERR_WORKSPACE, rc
    for t in [b for b in bufs if b is not None] + gps:
        assert bool(torch.isnan(t).all()), "a refused call wrote an output"

    assert lib.hgn_mlp_packed_bytes(f32, 3) == packed.numel()
    for n in (0, _cabi.HGN_MAX_CHUNKS + 1):
        bad = _cabi.Chunks.from_buffer_copy(ch)
        bad.n_chunks = n
        assert lib.hgn_mlp_packed_bytes(f32, n) == 0 and lib.hgn_mlp_backward_workspace_bytes(f32, rows, n) == 0
        blob = torch.full((packed.numel(),), 0xA5, dtype=torch.uint8, device="cuda")
        assert lib.hgn_mlp_pack(f32, n, *[p.data_ptr() for p in params], blob.data_ptr(), st) == HGN_ERR_INVALID_ARGUMENT
        assert bool((blob == 0xA5).all()), f"hgn_mlp_pack wrote with n_chunks = {n}"
        o = nan(rows, 128)
        rc = lib.hgn_mlp_forward(f32, rows, ctypes.byref(bad), packed.data_ptr(), e.data_ptr(), off, o.data_ptr(), st)
        assert rc == HGN_ERR_INVALID_ARGUMENT, rc
        assert bool(torch.isnan(o).all()), f"hgn_mlp_forward wrote with n_chunks = {n}"
        bufs, gps, rc = backward(-1, chunks=bad)
        assert rc == HGN_ERR_INVALID_ARGUMENT, rc
        for t in bufs + gps:
            assert bool(torch.isnan(t).all()), f"hgn_mlp_backward wrote with n_chunks = {n}"
    torch.cuda.empty_cache()

