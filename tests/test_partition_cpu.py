"""Host-side logic of the edge-cut partitioning (SURVEY.md s8e), on CPU:
* the partition bookkeeping is bit-exact (every edge owned once, ghosts = remote senders, send/recv lists agree);
* a world_size-2 gloo run of the halo exchange + weight-gradient all-reduce, with the CPU oracle doing the
  arithmetic, reproduces the single-process result (forward latents and all gradients)."""
import os
import sys

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import hgn_oracle as orc
from conftest import ROOT
from hgn_b200 import partition, synthetic


@pytest.mark.parametrize("world", [2, 3, 4, 8])
def test_partition_bookkeeping_bit_exact(world):
    w, h = 13, 11
    s, r = synthetic.grid_edges_two_way(w, h)
    n = w * h
    part = partition.block_partition(n, world)
    lgs = [partition.build_local_graph(s, r, part, p, world) for p in range(world)]
    all_edges = torch.cat([lg.edge_ids for lg in lgs])
    assert torch.equal(torch.sort(all_edges).values, torch.arange(s.numel()))          # each edge owned exactly once
    assert torch.equal(torch.sort(torch.cat([lg.owned for lg in lgs])).values, torch.arange(n))
    for lg in lgs:
        glob = torch.cat([lg.owned, lg.ghosts])
        assert torch.equal(glob[lg.senders], s[lg.edge_ids]) and torch.equal(glob[lg.receivers], r[lg.edge_ids])
        assert int(lg.receivers.max()) < lg.n_own                                     # receivers are always owned
        assert (part[lg.ghosts] != lg.rank).all() and sum(lg.ghost_splits) == lg.n_ghost
        assert torch.equal(lg.edge_ids, torch.sort(lg.edge_ids).values)               # original edge order kept
    for p in range(world):
        for q in range(world):
            if p == q:
                continue
            lo = sum(lgs[p].send_splits[:q])
            sent_global = lgs[p].owned[lgs[p].send_index[lo:lo + lgs[p].send_splits[q]]]
            glo = sum(lgs[q].ghost_splits[:p])
            assert torch.equal(sent_global, lgs[q].ghosts[glo:glo + lgs[q].ghost_splits[p]])   # same rows, same order


@pytest.mark.parametrize("world", [2, 4, 8])
def test_interior_first_edge_order(world):
    """interior_first lists the edges with an owned sender before the cut edges, each group in original order, and changes
    nothing else (same edge set, same ghosts, same exchange lists)."""
    w, h = 13, 11
    s, r = synthetic.grid_edges_two_way(w, h)
    part = partition.block_partition(w * h, world)
    for p in range(world):
        base = partition.build_local_graph(s, r, part, p, world)
        lg = partition.build_local_graph(s, r, part, p, world, interior_first=True)
        k = lg.n_interior
        assert base.n_interior is None and 0 < k < lg.edge_ids.numel()
        assert (lg.senders[:k] < lg.n_own).all() and (lg.senders[k:] >= lg.n_own).all()
        assert torch.equal(lg.edge_ids[:k], torch.sort(lg.edge_ids[:k]).values)
        assert torch.equal(lg.edge_ids[k:], torch.sort(lg.edge_ids[k:]).values)
        assert torch.equal(torch.sort(lg.edge_ids).values, base.edge_ids)
        assert torch.equal(lg.ghosts, base.ghosts) and torch.equal(lg.send_index, base.send_index)
        glob = torch.cat([lg.owned, lg.ghosts])
        assert torch.equal(glob[lg.senders], s[lg.edge_ids]) and torch.equal(glob[lg.receivers], r[lg.edge_ids])


def test_coordinate_bisection_balanced():
    pos = synthetic.cloth_frame(16, 12, 0)["mesh_pos"]
    part = partition.coordinate_bisection(pos, 4)
    counts = torch.bincount(part, minlength=4)
    assert int(counts.max() - counts.min()) <= 1


def _oracle_block(weights, prefix, nodes, ghosts, es):
    g = orc.block_graphnet(weights, prefix, "sum", orc.MultiGraph([nodes, ghosts], [es]))
    return g.node_features[0], g.edge_sets[0]


def _cpu_row_kernels():
    """CPU stand-ins (torch indexing) for the two row kernels of the halo exchange: the product's ``_gather_rows`` /
    ``_scatter_add_rows`` are CUDA only, these let the gloo runs exercise the exchange BOOKKEEPING without a GPU."""
    partition._gather_rows = lambda src, index, index32: src.index_select(0, index)

    def scatter_add(dst, rows, index, index32):
        if rows.numel():
            dst.index_add_(0, index, rows)
    partition._scatter_add_rows = scatter_add


def _mesh_edges(w, h, directed):
    """The two-way grid mesh, or only its ascending edges (sender < receiver): with a block partition the lower rank then sends boundary
    rows but owns no ghost, and in the backward receives ghost gradients but returns none -- the asymmetric case of ADVICE r1."""
    s, r = synthetic.grid_edges_two_way(w, h)
    if directed:
        keep = s < r
        s, r = s[keep], r[keep]
    return s, r


def _worker(rank, world, port, tmpdir, directed=False):
    _cpu_row_kernels()
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        w, h, layers = 9, 8, 2
        s, r = _mesh_edges(w, h, directed)
        n, e = w * h, s.numel()
        weights = {k: t.clone().requires_grad_(True) for k, t in
                   synthetic.seeded_state_dict(synthetic.processor_shapes(layers, ["mesh_edges"], "sum"), 3).items()}
        v0 = synthetic.seeded_tensor("pv", (n, 128), 2)
        e0 = synthetic.seeded_tensor("pe", (e, 128), 2)
        coef = synthetic.seeded_tensor("pc", (n, 128), 2)
        lg = partition.build_local_graph(s, r, partition.block_partition(n, world), rank, world)
        plan = partition.HaloPlan(lg, "cpu")
        owned = v0[lg.owned].clone().requires_grad_(True)
        edges = e0[lg.edge_ids].clone().requires_grad_(True)
        es = orc.EdgeSet("mesh_edges", edges, lg.senders, lg.receivers)
        nodes = owned
        for b in range(layers):
            ghosts = partition.halo_exchange(nodes, plan)
            nodes, es = _oracle_block(weights, f"processor.graphnet_blocks.{b}", nodes, ghosts, es)
        loss = (nodes * coef[lg.owned]).sum() + es.features.sum() * 1e-3
        loss.backward()

        class _Holder(torch.nn.Module):
            def __init__(self, ws):
                super().__init__()
                self.ps = torch.nn.ParameterList([torch.nn.Parameter(t.detach()) for t in ws.values()])
                for p, t in zip(self.ps, ws.values()):
                    p.grad = t.grad
        holder = _Holder(weights)
        partition.allreduce_gradients(holder)
        torch.save({"owned_ids": lg.owned, "edge_ids": lg.edge_ids, "nodes": nodes.detach(), "edges": es.features.detach(),
                    "grad_v": owned.grad, "grad_e": edges.grad, "grad_w": [p.grad for p in holder.ps]},
                   os.path.join(tmpdir, f"rank{rank}.pt"))
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("directed", [False, True])
def test_two_rank_halo_exchange_matches_single_process(tmp_path, directed):
    world = 2
    port = 29500 + (os.getpid() % 2000) + (7 if directed else 0)
    mp.spawn(_worker, args=(world, port, str(tmp_path), directed), nprocs=world, join=True)
    w, h, layers = 9, 8, 2
    s, r = _mesh_edges(w, h, directed)
    n, e = w * h, s.numel()
    weights = {k: t.clone().requires_grad_(True) for k, t in
               synthetic.seeded_state_dict(synthetic.processor_shapes(layers, ["mesh_edges"], "sum"), 3).items()}
    v = synthetic.seeded_tensor("pv", (n, 128), 2).requires_grad_(True)
    ed = synthetic.seeded_tensor("pe", (e, 128), 2).requires_grad_(True)
    coef = synthetic.seeded_tensor("pc", (n, 128), 2)
    out = orc.processor(weights, "sum", "none", orc.MultiGraph([v], [orc.EdgeSet("mesh_edges", ed, s, r)]))
    ((out.node_features[0] * coef).sum() + out.edge_sets[0].features.sum() * 1e-3).backward()
    parts = [torch.load(os.path.join(tmp_path, f"rank{k}.pt")) for k in range(world)]
    for p in parts:
        assert torch.allclose(p["nodes"], out.node_features[0].detach()[p["owned_ids"]], rtol=1e-5, atol=1e-5)
        assert torch.allclose(p["edges"], out.edge_sets[0].features.detach()[p["edge_ids"]], rtol=1e-5, atol=1e-5)
        assert torch.allclose(p["grad_v"], v.grad[p["owned_ids"]], rtol=1e-4, atol=1e-5)     # includes ghost gradients returned
        assert torch.allclose(p["grad_e"], ed.grad[p["edge_ids"]], rtol=1e-4, atol=1e-5)
        for g, ref in zip(p["grad_w"], weights.values()):
            assert torch.allclose(g, ref.grad, rtol=1e-4, atol=1e-4)                          # identical on both ranks after all-reduce


# ---- trajectory data parallelism (cfg 4: replicas + gradient all-reduce, SURVEY.md s8e) -------------------------------------
def _dp_batch(seed):
    w, h = 7, 6
    s, r = synthetic.grid_edges_two_way(w, h)
    v = synthetic.seeded_tensor(f"dp_v{seed}", (w * h, 128), seed)
    e = synthetic.seeded_tensor(f"dp_e{seed}", (s.numel(), 128), seed)
    return s, r, v, e


def _dp_loss(weights, batch):
    s, r, v, e = batch
    out = orc.processor(weights, "sum", "none", orc.MultiGraph([v], [orc.EdgeSet("mesh_edges", e, s, r)]))
    return out.node_features[0].square().mean() + out.edge_sets[0].features.square().mean()


def _dp_weights():
    return {k: t.clone().requires_grad_(True) for k, t in
            synthetic.seeded_state_dict(synthetic.processor_shapes(2, ["mesh_edges"], "sum"), 5).items()}


def _dp_worker(rank, world, port, tmpdir):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        weights = _dp_weights()
        _dp_loss(weights, _dp_batch(10 + rank)).backward()          # rank i takes trajectory batch i

        class _Holder(torch.nn.Module):
            def __init__(self, ws):
                super().__init__()
                self.ps = torch.nn.ParameterList([torch.nn.Parameter(t.detach()) for t in ws.values()])
                for p, t in zip(self.ps, ws.values()):
                    p.grad = t.grad
        holder = _Holder(weights)
        partition.allreduce_gradients(holder)
        torch.save([p.grad for p in holder.ps], os.path.join(tmpdir, f"dp_rank{rank}.pt"))
    finally:
        dist.destroy_process_group()


def test_two_rank_data_parallel_gradients_match_summed_batches(tmp_path):
    """Replicas on different trajectory batches + `allreduce_gradients` == one process summing the batches' gradients."""
    world = 2
    port = 31500 + (os.getpid() % 2000)
    mp.spawn(_dp_worker, args=(world, port, str(tmp_path)), nprocs=world, join=True)
    weights = _dp_weights()
    sum(_dp_loss(weights, _dp_batch(10 + k)) for k in range(world)).backward()
    per_rank = [torch.load(os.path.join(tmp_path, f"dp_rank{k}.pt")) for k in range(world)]
    for g0, g1, ref in zip(per_rank[0], per_rank[1], weights.values()):
        assert torch.equal(g0, g1)                                   # replicas stay identical
        assert torch.allclose(g0, ref.grad, rtol=1e-5, atol=1e-6)


def _norm_batch(step, rank):
    g = torch.Generator().manual_seed(100 + 10 * step + rank)
    return torch.randn(13 + rank, 5, generator=g) * (1.0 + rank) + step


def _norm_worker(rank, world, port, tmpdir):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from hgn_b200 import util
        from hgn_b200.migration.normalizer import Normalizer
        util.device = torch.device("cpu")                                # host statistics, also where a GPU is visible
        nzs = [Normalizer(5, "a"), Normalizer(5, "b")]
        outs = []
        for step in range(3):
            nzs[0](_norm_batch(step, rank), True)
            if step != 1:
                nzs[1](_norm_batch(step, rank) * 2.0, True)           # the second normaliser skips a step: zero increment there
            partition.allreduce_normalizers(nzs)
            outs.append(nzs[0](_norm_batch(7, 0), False))              # evaluation with the synchronised statistics
        torch.save({"state": [[getattr(nz, f) for f in partition._NORMALIZER_FIELDS] for nz in nzs], "outs": outs},
                   os.path.join(tmpdir, f"norm_rank{rank}.pt"))
    finally:
        dist.destroy_process_group()


def test_two_rank_normalizer_statistics_match_one_process_seeing_all_batches(tmp_path, monkeypatch):
    """Replicas accumulate their own batches; `allreduce_normalizers` leaves every rank with the totals of a single process that
    accumulated all ranks' batches (rank order within a step), so normalised features agree across replicas and with that process."""
    from hgn_b200 import util
    from hgn_b200.migration.normalizer import Normalizer
    monkeypatch.setattr(util, "device", torch.device("cpu"))            # the workers keep their statistics on the host too
    world = 2
    port = 33500 + (os.getpid() % 2000)
    mp.spawn(_norm_worker, args=(world, port, str(tmp_path)), nprocs=world, join=True)
    ref = [Normalizer(5, "a"), Normalizer(5, "b")]
    ref_outs = []
    for step in range(3):
        for rank in range(world):
            ref[0](_norm_batch(step, rank), True)
            if step != 1:
                ref[1](_norm_batch(step, rank) * 2.0, True)
        ref_outs.append(ref[0](_norm_batch(7, 0), False))
    per_rank = [torch.load(os.path.join(tmp_path, f"norm_rank{k}.pt")) for k in range(world)]
    for k in range(len(ref)):
        for j, f in enumerate(partition._NORMALIZER_FIELDS):
            a, b = per_rank[0]["state"][k][j], per_rank[1]["state"][k][j]
            assert torch.equal(a, b), f                                            # replicas identical
            assert torch.allclose(a, getattr(ref[k], f), rtol=1e-6, atol=1e-6), f
    assert float(per_rank[0]["state"][0][3]) == 6.0 and float(per_rank[0]["state"][1][3]) == 4.0      # _num_accumulations
    for o0, o1, r in zip(per_rank[0]["outs"], per_rank[1]["outs"], ref_outs):
        assert torch.equal(o0, o1) and torch.allclose(o0, r, rtol=1e-4, atol=1e-5)
