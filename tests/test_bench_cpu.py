"""bench.py's CPU legs (the `cpu_baseline` object and the `--impl reference` arm) on a reduced sample: the JSON contract of
the reference arm must hold without a GPU."""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402
import bench  # noqa: E402


def test_cpu_baseline_and_reference_arm_contract(monkeypatch, capsys):
    """The reference arm runs the LIVE reference's Processor (kind 'reference') when a reference tree is present and no GPU is visible,
    the oracle port (kind 'port') otherwise; `cpu_baseline` of the GPU arm gets the same object from a GPU-less child process."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import reference_shim
    want_kind = "reference" if reference_shim.available() and not torch.cuda.is_available() else "port"
    monkeypatch.setenv("HGN_BENCH_CPU_SAMPLE", "60x20")
    cpu = bench.cpu_baseline(steps=1)                    # child process: python bench.py --impl reference
    assert cpu["kind"] in ("reference", "port") and cpu["unit"] == bench.UNIT and cpu["value"] > 0 and cpu["cores"] >= 1
    assert "60x20" in cpu["sample"]
    if reference_shim.available():
        assert cpu["kind"] == "reference"
    port = bench.cpu_baseline_inprocess(steps=1)
    assert port["kind"] == want_kind and port["value"] > 0
    monkeypatch.delenv("RANK", raising=False)
    bench.run_reference(argparse.Namespace(steps=1, warmup=1, gpus=1, impl="reference", aggregator="sum", workload="cfg5", rollout_steps=0))
    line = json.loads(capsys.readouterr().out.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["metric"] == bench.METRIC and line["unit"] == bench.UNIT
    assert line["higher_is_better"] is True and line["value"] > 0 and line["steps"] == 1
    assert line["cpu_baseline"]["kind"] == want_kind and line["cpu_baseline"]["value"] == line["value"]
    assert line["e2e"] == {"value": line["value"], "unit": bench.UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    # ranks other than 0 print nothing
    monkeypatch.setenv("RANK", "1")
    bench.run_reference(argparse.Namespace(steps=1, warmup=1, gpus=2, impl="reference", aggregator="sum", workload="cfg5", rollout_steps=0))
    assert capsys.readouterr().out.strip() == ""


def test_reference_processor_equals_oracle_port_on_the_bench_sample(monkeypatch):
    """The two CPU arms compute the same thing: one step's loss of the live reference Processor == the oracle port's."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import reference_shim
    if not reference_shim.available() or torch.cuda.is_available():
        import pytest
        pytest.skip("needs the reference tree and no visible GPU")
    ref_step, e1, kind = bench.cpu_state((30, 20, 1, 2), "pna")
    port_step, e2, kind2 = bench.cpu_state((30, 20, 1, 2), "pna", prefer_reference=False)
    assert (kind, kind2) == ("reference", "port") and e1 == e2
    a, b = ref_step(), port_step()
    assert abs(a - b) <= 1e-5 * abs(b)


def test_roofline_accounting_of_the_projected_kernels():
    peaks = {"hbm_gbs": 6448.1, "bf16_tflops": 1625.3, "bf16_tflops_sustained": 1378.8, "source": "test"}
    e, n = 5992002, 1000000
    kernels = [{"name": "edge_bwd_tc", "launches": 15, "ms": 15 * 3.5}, {"name": "edge_fwd_tc", "launches": 15, "ms": 15 * 1.1}]
    r = bench.dominant_kernel_roofline(kernels, 1, e, n, peaks)
    assert r["kernel"] == "edge_bwd_tc" and r["bound"] == "tensor" and r["unit"] == "TFLOP/s"
    assert abs(r["achieved"] - e * 20 * 128 * 128 / 3.5e-3 / 1e12) < 1e-6           # SURVEY s8d: backward = 2 x 10 D^2 per edge
    assert abs(r["frac"] - r["achieved"] / 1378.8) < 1e-12 and r["executed_tflops"] < r["achieved"]
    assert r["traffic"] == bench.ncu_traffic("edge_bwd_tc")                          # profiles/ncu_traffic.json (ncu capture), cfg5 launch size only
    assert r["traffic"] is None or 4e9 < r["traffic"] < 2e10
    assert bench.dominant_kernel_roofline(kernels, 1, 1000, 100, peaks)["traffic"] is None
    seg = bench.dominant_kernel_roofline([{"name": "segment_reduce", "launches": 3, "ms": 0.93}], 1, e, n, peaks)
    assert seg["bound"] == "hbm" and abs(seg["achieved"] - ((e + n) * 256 + e * 4) / 0.31e-3 / 1e9) < 1e-6


def test_batched_workload_is_disjoint_copies_of_the_mesh():
    # MeshSimulator._get_batched (src/algorithms/MeshSimulator.py:196-217): graph i's indices are offset by i * N
    one = bench.build_inputs(5, 4, 1)
    three = bench.build_inputs(5, 4, 1, batch=3, aggregator="pna")
    n, e = one["n"], one["e"]
    assert three["n"] == 3 * n and three["e"] == 3 * e and three["v0"].shape == (3 * n, 128)
    for i in range(3):
        assert torch.equal(three["senders"][i * e:(i + 1) * e], one["senders"] + i * n)
        assert torch.equal(three["receivers"][i * e:(i + 1) * e], one["receivers"] + i * n)
    assert set(bench.WORKLOADS) == {"cfg2", "cfg4", "cfg5"} and bench.WORKLOADS["cfg5"][:5] == (1000, 1000, 1, 15, "sum")


def test_cfg3_plate_clustering_and_batched_graph(monkeypatch):
    # block clustering: a disjoint cover of the plate body, 30 clusters (plateCluster.yaml asks for 31), face-adjacent neighbour pairs
    clusters, neighbors = bench.plate_block_clusters(bench.CFG3_PLATE)
    n_plate = bench.CFG3_PLATE[0] * bench.CFG3_PLATE[1] * bench.CFG3_PLATE[2]
    members = torch.cat(clusters)
    assert len(clusters) == 30 and members.numel() == n_plate and torch.equal(members.sort().values, torch.arange(n_plate))
    assert all(0 <= int(p[0]) < int(p[1]) < len(clusters) for p in neighbors) and len({tuple(p.tolist()) for p in neighbors}) == len(neighbors)
    # the batched graph, with the world-edge kernel replaced by the dense oracle (no GPU here)
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "oracle"))
    import hgn_oracle as orc
    import hgn_b200.world_edges as we
    monkeypatch.setattr(we, "world_edges", lambda pos, types, ms, mr, **kw: orc.world_edges(pos.cpu(), types.cpu(), ms.cpu(), mr.cpu()))
    graph, sizes = bench.build_plate_batch(torch.device("cpu"))
    n = (n_plate + 64) * bench.CFG3_BATCH
    assert sizes["nodes"] == n and sizes["hyper_nodes"] == 30 * bench.CFG3_BATCH and sizes["edges"]["world_edges"] > 0
    assert [es.name for es in graph.edge_sets] == ["mesh_edges", "world_edges", "intra_cluster_to_cluster", "intra_cluster_to_mesh", "inter_cluster"]
    assert set(bench.CFG3_SETS) == {es.name for es in graph.edge_sets}
    for es in graph.edge_sets:
        assert es.features.shape == (es.senders.numel(), 128) and int(es.senders.min()) >= 0
        assert int(max(es.senders.max(), es.receivers.max())) < n + sizes["hyper_nodes"]


def test_dump_outputs_writes_float32_arrays_on_a_fixed_row_sample(tmp_path):
    """--dump-outputs: loss, sampled latents and latent gradients, full parameter gradients, all float32, within 64 MB; the row
    sample is a fixed, sorted, duplicate-free function of the row count."""
    import numpy as np
    from hgn_b200.util import EdgeSet, MultiGraph
    n, e = 300, bench.DUMP_ROWS + 500
    g = torch.Generator().manual_seed(3)
    v = torch.randn(n, 128, generator=g).to(torch.bfloat16)
    ed = torch.randn(e, 128, generator=g)
    v.grad, ed.grad = torch.randn(n, 128, generator=g).to(torch.bfloat16), torch.randn(e, 128, generator=g)
    out = MultiGraph([v * 2], [EdgeSet("mesh_edges", ed * 3, None, None)])
    w = torch.nn.Parameter(torch.randn(128, 384, generator=g))
    w.grad = torch.randn(128, 384, generator=g)
    unused = torch.nn.Parameter(torch.zeros(4))
    bench.dump_outputs(str(tmp_path / "d"), torch.tensor(1.5), out, v, ed, [("blk.w", w), ("blk.unused", unused)])
    files = {f.name[:-4]: np.load(f) for f in (tmp_path / "d").iterdir()}
    assert set(files) == {"loss", "node_latents", "edge_latents", "node_latents_grad", "edge_latents_grad", "grad.blk.w"}
    assert all(a.dtype == np.float32 for a in files.values()) and sum(a.nbytes for a in files.values()) <= bench.DUMP_BYTES_MAX
    rows = bench.dump_rows(e)
    assert torch.equal(rows, bench.dump_rows(e)) and rows.numel() == bench.DUMP_ROWS
    assert bool((rows[1:] > rows[:-1]).all()) and int(rows[-1]) < e
    assert torch.equal(bench.dump_rows(n), torch.arange(n))
    assert float(files["loss"]) == 1.5 and files["node_latents"].shape == (n, 128) and files["edge_latents"].shape == (bench.DUMP_ROWS, 128)
    assert np.array_equal(files["node_latents"], (v * 2).float().numpy())
    assert np.array_equal(files["edge_latents_grad"], ed.grad[rows].numpy())
    assert np.array_equal(files["grad.blk.w"], w.grad.numpy())


def test_clock_sampler_summary_from_nvml_and_nvidia_smi_rows():
    """The `clocks` object of the bench line: median SM clock, max clock and the set of active clock-event reasons, from NVML samples
    (numbers + 'Active' / 'Not Active') and from `nvidia-smi --format=csv` rows (strings); 'unavailable' without samples or a GPU."""
    s = bench.ClockSampler(0)
    assert s.summary() == {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
    s.rows = [[1965.0, 1965.0, "Not Active", "Not Active", "Not Active", "Not Active"],
              [1890.0, 1965.0, "Not Active", "Not Active", "Not Active", "Active"],
              [1875.0, 1965.0, "Not Active", "Not Active", "Not Active", "Active"]]
    out = s.summary()
    assert out["sm_mhz"] == 1890.0 and out["sm_max_mhz"] == 1965.0 and out["reasons"] == ["sw_power_cap"] and out["samples"] == 3
    s.rows = [["1965", "1965", "Not Active", "Active", "Not Active", "Not Active"], ["[N/A]", "x"], ["1200", "1965", "Active", "Not Active", "Not Active", "Not Active"]]
    out = s.summary()
    assert out["samples"] == 2 and out["reasons"] == ["hw_slowdown", "hw_thermal_slowdown"]
    with bench.ClockSampler(0) as live:                  # no GPU here: both back ends are absent, the bench line still gets an object
        pass
    assert live.summary()["reasons"] == ["unavailable"] or live.summary()["sm_mhz"] is not None
