"""``GraphNet`` block on the fused B200 kernels -- mirror of src/migration/graphnet.py.

Same constructor, method names and mutation conventions as the reference (new ``EdgeSet``s via
``_replace``; the ``node_features`` *list* is mutated in place), so the reference's subclasses, system
models and pickled checkpoints keep working.  What differs is the arithmetic: one fused kernel per edge
update (gather sender/receiver rows + 3-layer MLP + LayerNorm + residual, graphnet.py:22-32), one CSR
pass per edge set for every requested aggregate (graphnet.py:50-70) and one fused kernel per node
update (graphnet.py:34-48) -- no ``[E,384]`` / ``[N,128(1+kS)]`` concatenations, no float atomics.
"""
from typing import Callable, List, Sequence

import torch
from torch import nn, Tensor

from .. import ops
from .._cabi import HgnError
from ..plan import segment_plan, to_device_index
from ..util import EdgeSet, MultiGraph

PNA_OPS = ('sum', 'mean', 'max', 'min')     # order fixed by graphnet.py:53-64


def _stack_rows(node_features: Sequence[Tensor]) -> Tensor:
    """Row-concatenation of the node list (mesh rows first, hyper rows after)."""
    if len(node_features) == 1:
        return node_features[0]
    return torch.cat(tuple(node_features), dim=0)


def _mlp_parameters(model: nn.Module, in_features: int, like: Tensor):
    """The eight tensors of a reference MLP ``Sequential(LazyMLP, LayerNorm)`` (meshgraphnet.py:53-60).
    Lazy linears are materialised exactly like the reference does it -- by the module's own first
    forward -- on a zero-row input, so the Parameter objects an optimizer already holds stay valid."""
    try:
        lazy_mlp, norm = model[0], model[1]
        linears = [getattr(lazy_mlp.layers, f'linear_{k}') for k in range(3)]
    except (TypeError, IndexError, AttributeError, KeyError) as err:
        raise HgnError('the fused kernels need the reference MLP: Sequential(LazyMLP(3 linears), LayerNorm)') from err
    if not isinstance(norm, nn.LayerNorm) or hasattr(lazy_mlp.layers, 'linear_3'):
        raise HgnError('the fused kernels need the reference MLP: Sequential(LazyMLP(3 linears), LayerNorm)')
    if any(isinstance(lin.weight, nn.parameter.UninitializedParameter) for lin in linears):
        with torch.no_grad():
            model(torch.zeros((0, in_features), dtype=torch.float32, device=like.device))
    if abs(norm.eps - 1e-5) > 1e-12:
        raise HgnError('LayerNorm eps other than 1e-5 is not supported by the fused kernels')
    return (linears[0].weight, linears[0].bias, linears[1].weight, linears[1].bias,
            linears[2].weight, linears[2].bias, norm.weight, norm.bias)


def _packed_cache(model: nn.Module) -> dict:
    cache = model.__dict__.get('_hgn_packed')
    if cache is None:
        cache = {}
        model.__dict__['_hgn_packed'] = cache
    return cache


class GraphNet(nn.Module):
    """Multi-Edge Interaction Network with residual connections."""

    def __init__(self, model_fn: Callable, output_size: int, message_passing_aggregator: str, edge_sets: List[str]):
        super().__init__()
        self.node_model_cross = model_fn(output_size)
        self.edge_models = nn.ModuleDict({name: model_fn(output_size) for name in edge_sets})
        self.message_passing_aggregator = message_passing_aggregator

    # checkpoints are whole-object pickles (MeshSimulator.py:483-493): drop device-side caches
    def __getstate__(self):
        state = self.__dict__.copy()
        state.pop('_hgn_packed', None)
        return state

    # ---- edge update (graphnet.py:22-32) -----------------------------------------------------
    def _update_edge_features(self, node_features: List[Tensor], edge_set: EdgeSet) -> Tensor:
        """``e' = e + LN(MLP([v[senders] | v[receivers] | e]))`` in one kernel."""
        model = self.edge_models[edge_set.name]          # KeyError for a set without a model, like the reference
        v = _stack_rows(node_features)
        if not v.is_cuda:
            raise HgnError('hgn_b200 blocks run on CUDA tensors only (no CPU fallback)')
        e = edge_set.features.to(v.device)
        num_nodes = v.shape[0]
        senders = segment_plan(to_device_index(edge_set.senders, v.device), num_nodes)
        receivers = segment_plan(to_device_index(edge_set.receivers, v.device), num_nodes)
        params = _mlp_parameters(model, 3 * v.shape[1], v)
        if v.dtype == torch.bfloat16 and e.dtype == torch.bfloat16:
            # throughput mode: node-side pre-projection + projected edge kernels; with the 'sum' aggregator the
            # receiver-keyed aggregate is produced by the same autograd node (see ops._EdgeUpdate) and handed to
            # _aggregates through the tensor it belongs to
            want_agg = self.message_passing_aggregator == 'sum'
            out, agg = ops.edge_update(params, _packed_cache(model), v, e, senders, receivers, want_agg)
            if agg is not None:
                out._hgn_sum_agg = (receivers, agg)
            return out
        chunks = [ops.ChunkSpec(0, senders), ops.ChunkSpec(0, receivers), ops.ChunkSpec(1)]
        return ops.fused_mlp(params, _packed_cache(model), [v, e], chunks, rows=e.shape[0], resid_source=1)

    # ---- aggregation (graphnet.py:50-70) -----------------------------------------------------
    def _aggregates(self, edge_sets: List[EdgeSet], num_nodes: int, device) -> List[Tensor]:
        names = self.edge_models.keys()
        reducers = PNA_OPS if self.message_passing_aggregator == 'pna' else (self.message_passing_aggregator,)
        if any(op not in PNA_OPS for op in reducers):
            raise Exception('Invalid operation type!')
        out: List[Tensor] = []
        for edge_set in edge_sets:
            if edge_set.name not in names:      # graphnet.py:43
                continue
            plan = segment_plan(to_device_index(edge_set.receivers, device), num_nodes)
            ready = getattr(edge_set.features, '_hgn_sum_agg', None)
            if ready is not None and reducers == ('sum',) and ready[0] is plan:
                out.append(ready[1])
                continue
            out.extend(ops.segment_aggregate(edge_set.features, plan, reducers))
        return out

    def aggregation(self, edge_sets: List[EdgeSet], features: List[Tensor], num_nodes: int) -> Tensor:
        """API-compatible form: ``cat([*features, aggregates...], -1)``.  The block itself never calls
        this -- the node kernels consume the aggregates chunk by chunk without a concatenation."""
        aggregates = self._aggregates(edge_sets, num_nodes, features[0].device)
        return torch.cat(list(features) + aggregates, dim=-1)

    # ---- node updates (graphnet.py:34-48, 94-108, 110-124) -------------------------------------
    def _fused_node_update(self, graph: MultiGraph, edge_sets: List[EdgeSet], model: nn.Module, target: int,
                           aggregates: List[Tensor] = None) -> Tensor:
        """``rows' = rows + LN(MLP([rows | agg_1 | ...]))`` for the mesh rows (target 0) or the hyper rows
        (target 1); aggregates are taken over all ``N + C`` rows like the reference does (``aggregates``: already computed
        by the caller, when two updates consume the same ones)."""
        node_features = graph.node_features
        offset = 0 if target == 0 else node_features[0].shape[0]
        v = _stack_rows(node_features)
        rows = node_features[target].shape[0]
        if aggregates is None:
            aggregates = self._aggregates(edge_sets, v.shape[0], v.device)
        sources = [v] + aggregates
        params = _mlp_parameters(model, v.shape[1] * len(sources), v)
        if (1 <= len(aggregates) <= 4 and rows > 0 and v.dtype == torch.bfloat16
                and all(a.dtype == torch.bfloat16 for a in aggregates) and v.shape[1] == ops.D_LATENT):
            # throughput mode, one edge set ('sum' ... or the four 'pna' aggregates): the aggregates' blocks of the first linear
            # are applied per node row and the projected edge kernels do the rest (ops._NodeUpdate).  With hyper / ghost rows in
            # the list only the target's slice of each aggregate is consumed, like the reference's agg_features[:N] / [N:]
            # (graphnet.py:45,105); a full-range slice is skipped (it would still cost a zero-fill + copy in backward).
            full = offset == 0 and rows == aggregates[0].shape[0]
            aggs = aggregates if full else [a[offset: offset + rows] for a in aggregates]
            return ops.node_update(params, _packed_cache(model), node_features[target], aggs)
        chunks = [ops.ChunkSpec(i, None, offset) for i in range(len(sources))]
        return ops.fused_mlp(params, _packed_cache(model), sources, chunks, rows=rows, resid_source=0, resid_offset=offset)

    def _update_node_features(self, graph: MultiGraph, edge_sets: List[EdgeSet]):
        graph.node_features[0] = self._fused_node_update(graph, edge_sets, self.node_model_cross, 0)

    def _update_hyper_node_features(self, graph: MultiGraph, edge_sets: List[EdgeSet], model: nn.Module):
        graph.node_features[1] = self._fused_node_update(graph, edge_sets, model, 1)

    def _update_down(self, graph: MultiGraph, edge_sets: List[EdgeSet]):
        graph.node_features[0] = self._fused_node_update(graph, edge_sets, self.node_model_down, 0)

    # ---- schedules ---------------------------------------------------------------------------
    def _whole_layer(self, graph: MultiGraph):
        """A block that ``takes_whole_layer`` on its one node list runs as a single autograd node (ops.graphnet_layer)."""
        if len(graph.node_features) != 1 or not takes_whole_layer(self, graph.node_features[0], graph.edge_sets):
            return None
        v, es = graph.node_features[0], graph.edge_sets[0]
        num_nodes = v.shape[0]
        senders = segment_plan(to_device_index(es.senders, v.device), num_nodes)
        receivers = segment_plan(to_device_index(es.receivers, v.device), num_nodes)
        v_new, e_new = self._layer(v, es.features.to(v.device), es.name, senders, receivers)
        graph = graph._replace(edge_sets=[es._replace(features=e_new)])
        graph.node_features[0] = v_new
        return graph

    def _layer(self, v: Tensor, e: Tensor, edge_set_name: str, senders, receivers, halo=None):
        """``(v', e')`` of ``ops.graphnet_layer`` with this block's weights and aggregator."""
        edge_model = self.edge_models[edge_set_name]
        k = 4 if self.message_passing_aggregator == 'pna' else 1
        ep = _mlp_parameters(edge_model, 3 * v.shape[1], v)
        np_ = _mlp_parameters(self.node_model_cross, (1 + k) * v.shape[1], v)
        return ops.graphnet_layer(ep, _packed_cache(edge_model), np_, _packed_cache(self.node_model_cross), v, e, senders, receivers,
                                  self.message_passing_aggregator, halo)

    def forward(self, graph: MultiGraph, mask=None) -> MultiGraph:
        """graphnet.py:72-84: every edge set from the OLD node latents, then one mesh-node update."""
        fused = self._whole_layer(graph)
        if fused is not None:
            return fused
        updated = [edge_set._replace(features=self._update_edge_features(graph.node_features, edge_set))
                   for edge_set in graph.edge_sets]
        graph = graph._replace(edge_sets=updated)
        self._update_node_features(graph, updated)
        return graph

    def perform_edge_updates(self, graph, edge_set_name, new_edge_sets):
        """graphnet.py:86-92: silently nothing for a name without a model."""
        if edge_set_name not in self.edge_models.keys():
            return
        edge_set = next(es for es in graph.edge_sets if es.name == edge_set_name)
        new_edge_sets[edge_set_name] = edge_set._replace(features=self._update_edge_features(graph.node_features, edge_set))

    def _present(self, *names) -> List[str]:
        """Iteration order of the reference's ``{...}.intersection(self.edge_models.keys())``
        (hypergraphnet.py:31,44): evaluated the same way so it is the same order in the same process."""
        return list(set(names).intersection(self.edge_models.keys()))


def takes_whole_layer(block: nn.Module, v: Tensor, edge_sets: Sequence[EdgeSet]) -> bool:
    """Whether ``block`` runs on node latents ``v`` and ``edge_sets`` as one ``ops.graphnet_layer``: plain GraphNet with the 'sum',
    'mean', 'max', 'min' or 'pna' aggregator, one edge set with a model, bf16 latents of width 128 on the GPU, at least one edge and one
    node.  The one-GPU block (``GraphNet._whole_layer``) and the partitioned processor (``partition.PartitionedProcessor``) both
    decide with it."""
    if (type(block) is not GraphNet or block.message_passing_aggregator not in PNA_OPS + ('pna',) or len(edge_sets) != 1
            or edge_sets[0].name not in block.edge_models.keys()):
        return False
    e = edge_sets[0].features
    return (v.is_cuda and v.dtype == torch.bfloat16 and e.dtype == torch.bfloat16 and v.shape[-1] == ops.D_LATENT
            and e.shape[-1] == ops.D_LATENT and v.shape[0] > 0 and e.shape[0] > 0)
