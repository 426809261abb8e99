"""Host-side bookkeeping of the partitioned HyperGraphNet processor, on CPU: ``partition.build_local_hyper_graph`` is bit-exact (every
mesh, up and down edge on exactly one rank, ``inter_cluster`` on every rank, local indices that map back to the global lists, ascending
global edge order, hyper node c at local row n_own + c, the mesh part equal to ``build_local_graph``), and the processors the partitioned
processor does not support raise ``HgnError`` instead of taking the generic route."""
import pytest
import torch

from hgn_b200 import partition, synthetic
from hgn_b200._cabi import HgnError
from hgn_b200.migration.meshgraphnet import MeshGraphNet
from hgn_b200.rmp.hierarchical_connector import connector_indices

W, H, C = 13, 11, 6
N = W * H


def _clusters(kind):
    ids = torch.arange(N)
    if kind == "band":          # consecutive node ids: row bands of the grid
        return list(ids.tensor_split(C))
    if kind == "column":        # column bands: every cluster crosses every row-slab part
        col = ids % W
        return [ids[(col * C) // W == c] for c in range(C)]
    return [ids[ids % C == c] for c in range(C)]      # round robin


def _index_lists(kind):
    return {"mesh_edges": synthetic.grid_edges_two_way(W, H), **connector_indices(_clusters(kind), [], N, fully_connect=True)}


@pytest.mark.parametrize("kind", ["band", "column", "round_robin"])
@pytest.mark.parametrize("world", [1, 2, 3, 4, 8])
def test_local_hyper_graph_bit_exact(world, kind):
    sets = _index_lists(kind)
    part = partition.block_partition(N, world)
    lhs = [partition.build_local_hyper_graph(sets, N, C, part, p, world) for p in range(world)]
    for p, lh in enumerate(lhs):
        ref = partition.build_local_graph(*sets["mesh_edges"], part, p, world)
        for field in ("owned", "ghosts", "send_index", "edge_ids", "senders", "receivers"):
            assert torch.equal(getattr(lh.mesh, field), getattr(ref, field)), field
        assert lh.mesh.ghost_splits == ref.ghost_splits and lh.mesh.send_splits == ref.send_splits
        assert lh.num_clusters == C and lh.n_own == ref.n_own
        glob = torch.cat([lh.mesh.owned, N + torch.arange(C)])          # [owned | hyper]: hyper node c at local row n_own + c
        for name, loc in lh.remote.items():
            s, r = sets[name]
            assert torch.equal(glob[loc.senders], s[loc.edge_ids]) and torch.equal(glob[loc.receivers], r[loc.edge_ids]), name
            assert torch.equal(loc.edge_ids, torch.sort(loc.edge_ids).values), name
            assert loc.edge_ids.dtype == loc.senders.dtype == loc.receivers.dtype == torch.int64
        up, down = lh.remote["intra_cluster_to_cluster"], lh.remote["intra_cluster_to_mesh"]
        assert (up.senders < lh.n_own).all() and (up.receivers >= lh.n_own).all()
        assert (down.receivers < lh.n_own).all() and (down.senders >= lh.n_own).all()
        assert torch.equal(lh.remote["inter_cluster"].edge_ids, torch.arange(sets["inter_cluster"][0].numel()))
    for name in ("intra_cluster_to_cluster", "intra_cluster_to_mesh"):
        every = torch.cat([lh.remote[name].edge_ids for lh in lhs])
        assert torch.equal(torch.sort(every).values, torch.arange(sets[name][0].numel())), name     # each edge on exactly one rank
    every = torch.cat([lh.mesh.edge_ids for lh in lhs])
    assert torch.equal(torch.sort(every).values, torch.arange(sets["mesh_edges"][0].numel()))


def test_local_hyper_graph_refuses_other_sets():
    sets = _index_lists("band")
    part = partition.block_partition(N, 2)
    with pytest.raises(HgnError, match="exactly"):
        partition.build_local_hyper_graph({**sets, "world_edges": sets["mesh_edges"]}, N, C, part, 0, 2)
    bad = dict(sets)
    bad["intra_cluster_to_cluster"] = (sets["intra_cluster_to_cluster"][1], sets["intra_cluster_to_cluster"][0])
    with pytest.raises(HgnError, match="outside"):
        partition.build_local_hyper_graph(bad, N, C, part, 0, 2)


def _processor(arch, agg="sum", sets=synthetic.HYPER_EDGE_SETS):
    return MeshGraphNet(3, 128, 2, agg, 2, arch, list(sets)).processor


@pytest.mark.parametrize("arch", ["hetero", "multiscale", "hyper"])
def test_out_of_scope_processors_raise(arch):
    """HeteroGraphNet and MultiScaleGraphNet blocks, and HyperGraphNet blocks without a PeerHalo and a LocalHyperGraph, are refused
    with the supported scope named (the generic route would read the hyper rows as ghosts)."""
    with pytest.raises(HgnError, match="HyperGraphNet blocks with edge sets exactly"):
        partition.PartitionedProcessor(_processor(arch), None, None)


def test_hyper_with_world_edges_or_plain_graph_sets_raises():
    sets = _index_lists("band")
    lh = partition.build_local_hyper_graph(sets, N, C, partition.block_partition(N, 1), 0, 1)
    with pytest.raises(HgnError, match="world_edges"):
        partition.PartitionedProcessor(_processor("hyper", sets=list(synthetic.HYPER_EDGE_SETS) + ["world_edges"]), None, None, hyper=lh)
    with pytest.raises(HgnError, match="not supported"):     # a LocalHyperGraph given to a processor of plain GraphNet blocks
        partition.PartitionedProcessor(MeshGraphNet(3, 128, 2, "sum", 2, "none", ["mesh_edges"]).processor, None, None, hyper=lh)


def test_allreduce_gradients_exclude_keyword_defaults_to_everything(monkeypatch):
    """``exclude`` leaves the named parameters out of the all-reduce; without it every gradient is reduced, as before."""
    lin = torch.nn.Linear(3, 2)
    for p in lin.parameters():
        p.grad = torch.ones_like(p)
    seen = []
    monkeypatch.setattr(partition.dist, "all_reduce", lambda flat, op=None, group=None: seen.append(flat.numel()))
    partition.allreduce_gradients(lin)
    partition.allreduce_gradients(lin, exclude=[lin.bias])
    assert seen == [8, 6]
