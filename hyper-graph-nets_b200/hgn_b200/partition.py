"""Edge-cut graph partitioning with a one-ring halo of sender latents (SURVEY.md s8e).

The reference is single-device (no ``torch.distributed`` anywhere), so this is new functionality whose
parity contract is "P-rank result == 1-rank result".  Scheme:

* nodes are split into P parts; every directed edge belongs to the OWNER OF ITS RECEIVER, so the
  edge->node aggregation and the node update are rank-local and edge latents never move;
* the only remote data are sender latents of cut edges: each rank keeps them as GHOST rows.  A rank's
  node list is ``[owned | ghosts]`` -- exactly the reference's ``node_features = [mesh, hyper]`` row
  concatenation (util.py:11-12, hierarchical_connector.py:37), so the unmodified ``GraphNet`` block
  updates the owned rows (list slot 0) and leaves the ghosts (slot 1) alone;
* before every block the owners send their boundary rows to the ranks that hold them as ghosts
  (``HaloExchange``: pack kernel -> grouped NCCL send/recv over NVLink -> ghosts land contiguously, ordered by
  owner, so no unpack is needed); in the backward pass ghost gradients travel back and are added at the
  owner peer by peer in rank order (deterministic);
* weight gradients are summed with one all-reduce after the backward pass.

Nothing here does arithmetic on latents besides the pack / scatter-add row kernels of ``libhgn_b200.so``
(CPU tensors use torch indexing instead, which is how the world_size-2 gloo tests exercise this logic).
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import List, NamedTuple, Optional, Sequence

import torch
import torch.distributed as dist

from . import _cabi, ops


# ------------------------------------------------------------------------------------------------------
# partition plan (pure index bookkeeping, bit-exact, CPU)
# ------------------------------------------------------------------------------------------------------
@dataclass
class LocalGraph:
    rank: int
    world: int
    owned: torch.Tensor            # [n_own]   global ids of the owned nodes (ascending)
    ghosts: torch.Tensor           # [n_ghost] global ids of the ghost nodes, sorted by (owner, id)
    ghost_splits: List[int]        # ghosts received from each rank (sums to n_ghost)
    send_index: torch.Tensor       # [n_send]  LOCAL owned indices to send, grouped by destination rank
    send_splits: List[int]         # rows sent to each rank
    edge_ids: torch.Tensor         # [e_loc]   global ids of the local edges (ascending -> original order kept)
    senders: torch.Tensor          # [e_loc]   local sender index into [owned | ghosts]
    receivers: torch.Tensor        # [e_loc]   local receiver index (always < n_own)
    n_interior: Optional[int] = None   # with interior_first: edges [0, n_interior) have an owned sender, the rest a ghost sender

    @property
    def n_own(self) -> int:
        return int(self.owned.numel())

    @property
    def n_ghost(self) -> int:
        return int(self.ghosts.numel())


def block_partition(num_nodes: int, world: int) -> torch.Tensor:
    """Contiguous id ranges (row slabs of a row-major grid mesh): part id per node."""
    bounds = [(num_nodes * p) // world for p in range(world + 1)]
    part = torch.empty(num_nodes, dtype=torch.int64)
    for p in range(world):
        part[bounds[p]:bounds[p + 1]] = p
    return part


def coordinate_bisection(pos: torch.Tensor, world: int) -> torch.Tensor:
    """Recursive coordinate bisection of node positions into ``world`` (power of two) parts."""
    n = pos.shape[0]
    part = torch.zeros(n, dtype=torch.int64)
    groups = [torch.arange(n)]
    while len(groups) < world:
        nxt = []
        for ids in groups:
            p = pos[ids]
            axis = int(torch.argmax(p.max(0).values - p.min(0).values))
            order = torch.argsort(p[:, axis], stable=True)
            half = ids.numel() // 2
            nxt += [ids[order[:half]], ids[order[half:]]]
        groups = nxt
    for k, ids in enumerate(groups):
        part[ids] = k
    return part


def build_local_graph(senders: torch.Tensor, receivers: torch.Tensor, part: torch.Tensor, rank: int, world: int,
                      interior_first: bool = False) -> LocalGraph:
    """Rank ``rank``'s share of a directed edge list under the receiver-owner rule.  ``interior_first`` lists the edges whose
    sender is owned before the cut edges (each group in original order), which is what lets the halo exchange overlap the
    interior edge tiles (``PartitionedProcessor``)."""
    senders, receivers, part = senders.cpu(), receivers.cpu(), part.cpu()
    owned = torch.nonzero(part == rank).flatten()
    edge_ids = torch.nonzero(part[receivers] == rank).flatten()
    n_interior = None
    if interior_first:
        cut = part[senders[edge_ids]] != rank
        edge_ids = torch.cat([edge_ids[~cut], edge_ids[cut]])
        n_interior = int((~cut).sum())
    s_glob, r_glob = senders[edge_ids], receivers[edge_ids]
    # ghosts: senders of local edges owned elsewhere, ordered by (owner, global id)
    remote = torch.unique(s_glob[part[s_glob] != rank])
    order = torch.argsort(part[remote] * (part.numel() + 1) + remote)
    ghosts = remote[order]
    ghost_splits = torch.bincount(part[ghosts], minlength=world).tolist()
    # global -> local id
    local_of = torch.full((part.numel(),), -1, dtype=torch.int64)
    local_of[owned] = torch.arange(owned.numel())
    local_of[ghosts] = owned.numel() + torch.arange(ghosts.numel())
    # what do the other ranks need from me?  (their ghost lists restricted to my nodes, same ordering rule)
    send_lists = []
    for q in range(world):
        if q == rank:
            send_lists.append(torch.empty(0, dtype=torch.int64))
            continue
        q_edges = part[receivers] == q
        need = torch.unique(senders[q_edges & (part[senders] == rank)])   # ascending global id == q's ghost order
        send_lists.append(local_of[need])
    return LocalGraph(rank=rank, world=world, owned=owned, ghosts=ghosts, ghost_splits=ghost_splits,
                      send_index=torch.cat(send_lists), send_splits=[int(t.numel()) for t in send_lists],
                      edge_ids=edge_ids, senders=local_of[s_glob], receivers=local_of[r_glob], n_interior=n_interior)


# ------------------------------------------------------------------------------------------------------
# halo exchange
# ------------------------------------------------------------------------------------------------------
def _gather_rows(src: torch.Tensor, index: torch.Tensor, index32: Optional[torch.Tensor]) -> torch.Tensor:
    """``src[index]`` through the pack kernel.  CUDA only: the world_size-2 gloo tests install their own CPU stand-ins for this
    function and ``_scatter_add_rows`` (tests/test_partition_cpu.py) -- the product has no CPU path."""
    _cabi.require_cuda(src)
    lib = _cabi.load()
    out = torch.empty((index.numel(), src.shape[1]), dtype=src.dtype, device=src.device)
    if index.numel():
        _cabi.check(lib.hgn_rows_gather(_cabi.dtype_code(src.dtype), src.data_ptr(), index32.data_ptr(), index.numel(), src.shape[1],
                                        out.data_ptr(), _cabi.stream_ptr()), "hgn_rows_gather")
    return out


def _scatter_add_rows(dst: torch.Tensor, rows: torch.Tensor, index: torch.Tensor, index32: Optional[torch.Tensor]) -> None:
    """dst[index[i]] += rows[i]; ``index`` has no duplicates (one peer at a time)."""
    if not rows.numel():
        return
    _cabi.require_cuda(dst, rows)
    lib = _cabi.load()
    _cabi.check(lib.hgn_rows_scatter(_cabi.dtype_code(dst.dtype), rows.data_ptr(), index32.data_ptr(), index.numel(), dst.shape[1],
                                     dst.data_ptr(), 1, _cabi.stream_ptr()), "hgn_rows_scatter")


def _exchange(send: torch.Tensor, send_splits: Sequence[int], recv_splits: Sequence[int], group) -> torch.Tensor:
    """All-to-all-v of row blocks with grouped point-to-point operations (NCCL: one fused launch over NVLink)."""
    world = dist.get_world_size(group)
    rank = dist.get_rank(group)
    recv = torch.empty((sum(recv_splits), send.shape[1]), dtype=send.dtype, device=send.device)
    ops, so, ro = [], 0, 0
    for q in range(world):
        if q != rank and recv_splits[q]:
            ops.append(dist.P2POp(dist.irecv, recv[ro:ro + recv_splits[q]], q, group))
        ro += recv_splits[q]
    for q in range(world):
        if q != rank and send_splits[q]:
            ops.append(dist.P2POp(dist.isend, send[so:so + send_splits[q]].contiguous(), q, group))
        so += send_splits[q]
    if ops:
        for work in dist.batch_isend_irecv(ops):
            work.wait()
    return recv


class HaloPlan:
    """Device-side copy of a ``LocalGraph``'s exchange lists."""

    def __init__(self, lg: LocalGraph, device, group=None):
        self.lg = lg
        self.group = group
        self.send_index = lg.send_index.to(device)
        self.send_index32 = self.send_index.to(torch.int32)
        self.send_splits = list(lg.send_splits)
        self.ghost_splits = list(lg.ghost_splits)
        self.peer_offsets = [0]
        for n in self.send_splits:
            self.peer_offsets.append(self.peer_offsets[-1] + n)


class _HaloExchange(torch.autograd.Function):
    @staticmethod
    def forward(ctx, owned: torch.Tensor, plan: HaloPlan):
        ctx.plan = plan
        ctx.n_own = owned.shape[0]
        packed = _gather_rows(owned.contiguous(), plan.send_index, plan.send_index32)
        return _exchange(packed, plan.send_splits, plan.ghost_splits, plan.group)

    @staticmethod
    def backward(ctx, grad_ghosts: torch.Tensor):
        plan: HaloPlan = ctx.plan
        back = _exchange(grad_ghosts.contiguous(), plan.ghost_splits, plan.send_splits, plan.group)
        grad_owned = torch.zeros((ctx.n_own, grad_ghosts.shape[1]), dtype=grad_ghosts.dtype, device=grad_ghosts.device)
        for q in range(len(plan.send_splits)):          # peers in rank order: fixed summation order
            lo, hi = plan.peer_offsets[q], plan.peer_offsets[q + 1]
            if hi > lo:
                idx32 = plan.send_index32[lo:hi] if plan.send_index32 is not None else None
                _scatter_add_rows(grad_owned, back[lo:hi], plan.send_index[lo:hi], idx32)
        return grad_owned, None


def halo_exchange(owned: torch.Tensor, plan: HaloPlan) -> torch.Tensor:
    """Ghost rows ``[n_ghost, D]`` (ordered by owner rank) holding the owners' current latents."""
    return _HaloExchange.apply(owned, plan)


class _DeviceBytes:
    """``__cuda_array_interface__`` view of a raw device allocation, for ``torch.as_tensor`` (no copy)."""

    def __init__(self, ptr: int, nbytes: int):
        self.__cuda_array_interface__ = {"shape": (nbytes,), "typestr": "|u1", "data": (ptr, False), "version": 2}


class PeerHalo:
    """One rank's exchange pool in NVLink peer memory and the mapped pools of its peers (csrc/peer.cu).

    Instead of exchanging the node latents ``v`` of the boundary nodes and projecting the ghosts again on every rank, the owners
    push the rows of their sender table ``Ps = v Ws^T`` (the only thing an edge kernel reads of a ghost) straight into the ghost
    part of their peers' tables; in the backward pass the ghost rows of ``segsum_senders(G0)`` go home the same way and are added at
    the owner in rank order.  A push is one small kernel of the SENDING rank plus a 4-byte flag per peer; the receiving stream
    waits for its flags with a one-warp kernel.  No NCCL kernel is involved, so nothing competes with the persistent compute
    kernels for SMs, and nothing returns to the host.

    Pool layout (bytes): ``[flags: 2 directions x world uint32 | push counter | tables: 2 parities x layers x (n_own + n_ghost) rows |
    inbox: layers x n_send rows]``.  The table of (step parity, layer) is also what the backward pass of that step reads again, so a
    peer that is one forward pass ahead (it cannot be further: its second layer needs this rank's rows) writes into the other parity."""

    def __init__(self, lg: LocalGraph, layers: int, device, group=None, width: int = 128):
        import ctypes
        lib = _cabi.load()
        self.lg, self.group, self.layers, self.width = lg, group, int(layers), int(width)
        self.device = torch.device(device)
        self.world, self.rank = dist.get_world_size(group), dist.get_rank(group)
        self.n_own, self.n_ghost, self.n_send = lg.n_own, lg.n_ghost, int(lg.send_index.numel())
        self.row_bytes = self.width * 2                      # bf16 rows
        self.rows = self.n_own + self.n_ghost
        self.off_counter = 2 * self.world * 4
        self.off_tables = 256 * ((self.off_counter + 4 + 255) // 256)
        self.off_inbox = self.off_tables + 2 * self.layers * self.rows * self.row_bytes
        self.nbytes = self.off_inbox + self.layers * max(self.n_send, 1) * self.row_bytes
        with torch.cuda.device(self.device):
            ptr = ctypes.c_void_p()
            handle = ctypes.create_string_buffer(64)
            _cabi.check(lib.hgn_peer_alloc(self.nbytes, ctypes.byref(ptr), handle), "hgn_peer_alloc")
        self.base = int(ptr.value)
        self.pool = torch.as_tensor(_DeviceBytes(self.base, self.nbytes), device=self.device)
        info = {"handle": bytes(handle.raw), "n_own": self.n_own, "off_tables": self.off_tables, "off_inbox": self.off_inbox, "rows": self.rows,
                "n_send": self.n_send, "ghost_splits": list(lg.ghost_splits), "send_splits": list(lg.send_splits)}
        infos = [None] * self.world
        dist.all_gather_object(infos, info, group=group)
        self.peer_base = [0] * self.world
        self.peer_info = infos
        with torch.cuda.device(self.device):
            for q in range(self.world):
                if q != self.rank and (lg.send_splits[q] or lg.ghost_splits[q]):
                    mapped = ctypes.c_void_p()
                    _cabi.check(lib.hgn_peer_open(infos[q]["handle"], ctypes.byref(mapped)), "hgn_peer_open")
                    self.peer_base[q] = int(mapped.value)
        self.send_index32 = lg.send_index.to(self.device, dtype=torch.int32)
        self.ghost_index32 = (self.n_own + torch.arange(self.n_ghost, dtype=torch.int32)).to(self.device)
        self.send_index = lg.send_index.to(self.device)
        self.steps_done = 0
        dist.barrier(group=group)                             # every pool exists and is mapped before anybody pushes

    def close(self) -> None:
        lib = _cabi.load()
        torch.cuda.synchronize(self.device)
        dist.barrier(group=self.group)
        for q, p in enumerate(self.peer_base):
            if p:
                lib.hgn_peer_close(p)
                self.peer_base[q] = 0
        if self.base:
            self.pool = None
            lib.hgn_peer_free(self.base)
            self.base = 0

    # ---- views into the own pool -----------------------------------------------------------------------------------
    def table(self, parity: int, layer: int) -> torch.Tensor:
        """``[n_own + n_ghost, width]`` bf16: Ps of the owned rows (written here) and of the ghosts (written by their owners)."""
        off = self.off_tables + (parity * self.layers + layer) * self.rows * self.row_bytes
        return self.pool[off: off + self.rows * self.row_bytes].view(torch.bfloat16).view(self.rows, self.width)

    def inbox(self, layer: int) -> torch.Tensor:
        """``[n_send, width]`` bf16: gradients of the rows this rank sent, grouped by the peer that returns them."""
        off = self.off_inbox + layer * max(self.n_send, 1) * self.row_bytes
        return self.pool[off: off + self.n_send * self.row_bytes].view(torch.bfloat16).view(self.n_send, self.width)

    # ---- the two exchanges ---------------------------------------------------------------------------------------------
    def _epoch(self, step: int, layer: int, backward: bool) -> int:
        return (1 + step * self.layers + (self.layers - 1 - layer if backward else layer)) & 0x7FFFFFFF

    def push_forward(self, step: int, layer: int) -> None:
        """Boundary rows of this rank's Ps table -> the ghost rows of its peers' tables of the same (parity, layer); then wait for
        the peers' pushes into this rank's table."""
        import ctypes
        lib = _cabi.load()
        parity, epoch = step & 1, self._epoch(step, layer, False)
        peers, flags = _cabi.HaloPeers(), _cabi.HaloFlags()
        n_push = n_wait = 0
        lo = 0
        for q in range(self.world):
            n = self.lg.send_splits[q]
            if q != self.rank and n:
                inf = self.peer_info[q]
                ghost_off = sum(inf["ghost_splits"][:self.rank])
                peers.dst[n_push] = (self.peer_base[q] + inf["off_tables"]
                                     + ((parity * self.layers + layer) * inf["rows"] + inf["n_own"] + ghost_off) * self.row_bytes)
                peers.flag[n_push] = self.peer_base[q] + (0 * self.world + self.rank) * 4
                peers.row_begin[n_push] = lo
                n_push += 1
            lo += n
            if q != self.rank and self.lg.ghost_splits[q]:
                flags.flag[n_wait] = self.base + (0 * self.world + q) * 4
                n_wait += 1
        peers.row_begin[n_push] = lo
        self._run(lib, self.table(parity, layer), self.send_index32, peers, n_push, flags, n_wait, epoch, compact=True)

    def push_backward(self, step: int, layer: int, gs: torch.Tensor) -> None:
        """Ghost rows of ``gs`` (sender-keyed sums of G0, ``[n_own + n_ghost, width]``) -> their owners' inboxes; then wait for the
        rows the peers return to this rank and add them into the owned rows of ``gs``, peer by peer in rank order (a fixed summation
        order)."""
        lib = _cabi.load()
        epoch = self._epoch(step, layer, True)
        peers, flags = _cabi.HaloPeers(), _cabi.HaloFlags()
        n_push = n_wait = 0
        lo = 0
        for q in range(self.world):
            n = self.lg.ghost_splits[q]
            if q != self.rank and n:
                inf = self.peer_info[q]
                send_off = sum(inf["send_splits"][:self.rank])
                peers.dst[n_push] = self.peer_base[q] + inf["off_inbox"] + (layer * max(inf["n_send"], 1) + send_off) * self.row_bytes
                peers.flag[n_push] = self.peer_base[q] + (1 * self.world + self.rank) * 4
                peers.row_begin[n_push] = lo
                n_push += 1
            lo += n
            if q != self.rank and self.lg.send_splits[q]:
                flags.flag[n_wait] = self.base + (1 * self.world + q) * 4
                n_wait += 1
        peers.row_begin[n_push] = lo
        self._run(lib, gs, self.ghost_index32, peers, n_push, flags, n_wait, epoch, compact=False)
        inbox = self.inbox(layer)
        lo = 0
        for q in range(self.world):
            n = self.lg.send_splits[q]
            if n and q != self.rank:
                ops._rows_add(inbox[lo:lo + n], self.send_index32[lo:lo + n], gs)
            lo += n

    def _run(self, lib, table, index32, peers, n_push, flags, n_wait, epoch, compact):
        import ctypes
        # row_begin was filled with offsets into the FULL per-rank ordering; peers without rows were skipped, so the offsets of the
        # kept ones are already right (rows of a skipped peer do not exist)
        with torch.cuda.device(self.device):
            st = _cabi.stream_ptr()
            _cabi.check(lib.hgn_halo_push(_cabi.HGN_BF16, table.data_ptr(), index32.data_ptr(), self.width, ctypes.byref(peers), n_push, epoch,
                                          self.base + self.off_counter, st), "hgn_halo_push")
            _cabi.check(lib.hgn_halo_wait(ctypes.byref(flags), n_wait, epoch, st), "hgn_halo_wait")
        ops._count(int(n_push > 0) + int(n_wait > 0))     # csrc/peer.cu: each entry point launches one kernel, none without peers


class PeerLayerHalo(NamedTuple):
    """The halo of one (step, layer) of a ``PeerHalo``, in the form ``ops.graphnet_sum_layer`` takes it."""
    peer: PeerHalo
    step: int
    layer: int

    def sender_table(self) -> torch.Tensor:
        return self.peer.table(self.step & 1, self.layer)

    def exchange_forward(self) -> None:
        self.peer.push_forward(self.step, self.layer)

    def exchange_backward(self, gs: torch.Tensor) -> None:
        self.peer.push_backward(self.step, self.layer, gs)


class PartitionedProcessor(torch.nn.Module):
    """Runs a (reference-API) ``Processor`` on one rank's share of the graph.

    Generic path (any block type, any aggregator, fp32 or bf16): ghosts are refreshed before every block with a grouped NCCL
    send/recv; the block itself is unchanged (it sees ``[owned | ghosts]`` as ``[mesh | hyper]`` rows).
    Fast path (``PeerHalo`` given, and every block takes the whole-layer route of ``GraphNet`` -- the cfg5 benchmark):
    ``ops.graphnet_sum_layer`` per block with the halo of that layer; halo rows travel as peer-memory stores issued by a kernel of
    the sending rank."""

    def __init__(self, processor: torch.nn.Module, plan: HaloPlan, peer: Optional[PeerHalo] = None):
        super().__init__()
        self.processor = processor
        self.plan = plan
        self.peer = peer
        if peer is not None:
            from .plan import segment_plan
            lg, dev = peer.lg, peer.device
            peer.senders, peer.receivers = lg.senders.to(dev), lg.receivers.to(dev)
            peer.s_plan = segment_plan(peer.senders, lg.n_own + lg.n_ghost)
            peer.r_plan = segment_plan(peer.receivers, lg.n_own)

    def _fast_path(self, owned, edge_sets) -> bool:
        from .migration.graphnet import takes_whole_layer
        blocks = self.processor.graphnet_blocks
        return (self.peer is not None and len(blocks) == self.peer.layers
                and all(takes_whole_layer(b, owned, edge_sets) for b in blocks))

    def forward(self, owned: torch.Tensor, edge_sets):
        from . import config
        from .util import MultiGraph
        precision = getattr(self.processor, "precision", None) or config.precision()
        in_dtype = owned.dtype
        if precision == "bf16":
            owned = owned.to(torch.bfloat16)
            edge_sets = [es._replace(features=es.features.to(torch.bfloat16)) for es in edge_sets]
        if precision == "bf16" and self._fast_path(owned, edge_sets):
            es = edge_sets[0]
            e = es.features
            step = self.peer.steps_done
            self.peer.steps_done += 1
            for layer, block in enumerate(self.processor.graphnet_blocks):
                owned, e = block._sum_layer(owned, e, es.name, self.peer.s_plan, self.peer.r_plan, PeerLayerHalo(self.peer, step, layer))
            return owned.to(in_dtype), [es._replace(features=e)]
        graph = MultiGraph([owned, None], list(edge_sets))
        for block in self.processor.graphnet_blocks:
            graph.node_features[1] = halo_exchange(graph.node_features[0], self.plan)
            graph = block(graph)
        out_nodes = graph.node_features[0].to(in_dtype)
        return out_nodes, list(graph.edge_sets)      # edge latents stay in the compute dtype (see Processor.forward)


def allreduce_gradients(module: torch.nn.Module, group=None) -> None:
    """Sum the per-rank partial weight gradients (one flat fp32 all-reduce)."""
    grads = [p.grad for p in module.parameters() if p.grad is not None]
    if not grads:
        return
    flat = torch.cat([g.reshape(-1) for g in grads])
    dist.all_reduce(flat, op=dist.ReduceOp.SUM, group=group)
    off = 0
    for g in grads:
        g.copy_(flat[off:off + g.numel()].view_as(g))
        off += g.numel()


_NORMALIZER_FIELDS = ("_acc_sum", "_acc_sum_squared", "_acc_count", "_num_accumulations")


def allreduce_normalizers(normalizers, group=None) -> None:
    """Keep the replicas' online feature statistics identical (SURVEY.md s8e): every ``Normalizer``
    (src/migration/normalizer.py:53-63) accumulates its own rank's batches; this sums, over the ranks, what each accumulated since
    the previous call and adds it to the common state -- the totals a single process that had seen every rank's batches would hold
    (``_num_accumulations`` advances by the world size per step, like that process's counter).  One flat all-reduce for all of them."""
    normalizers = list(normalizers)
    if not normalizers:
        return
    bases, deltas = [], []
    for nz in normalizers:
        base = getattr(nz, "_synced_state", None)
        if base is None:
            base = {f: torch.zeros_like(getattr(nz, f)) for f in _NORMALIZER_FIELDS}
        bases.append(base)
        deltas.extend((getattr(nz, f) - base[f]).reshape(-1).float() for f in _NORMALIZER_FIELDS)
    flat = torch.cat(deltas)
    dist.all_reduce(flat, op=dist.ReduceOp.SUM, group=group)
    off = 0
    for nz, base in zip(normalizers, bases):
        state = {}
        for f in _NORMALIZER_FIELDS:
            cur = getattr(nz, f)
            state[f] = base[f] + flat[off:off + cur.numel()].view_as(cur).to(cur.dtype)
            off += cur.numel()
            setattr(nz, f, state[f])
        nz._synced_state = {f: t.clone() for f, t in state.items()}


# ------------------------------------------------------------------------------------------------------
# multi-GPU benchmark (bench.py --gpus N under torchrun)
# ------------------------------------------------------------------------------------------------------
def bench_partitioned(args, world, rank, dev, width, height, layers, metric, unit, peaks, clock_sampler_cls, roofline_fn=None, extra_leg=None):
    import json
    import os
    from . import ops, synthetic
    from .migration.meshgraphnet import MeshGraphNet
    from .util import EdgeSet

    n = width * height
    senders, receivers = synthetic.grid_edges_two_way(width, height)
    e_total = senders.numel()
    part = block_partition(n, world)
    lg = build_local_graph(senders, receivers, part, rank, world, interior_first=True)
    gen = torch.Generator().manual_seed(0)
    v0 = torch.randn(n, 128, generator=gen)[lg.owned]
    e0 = torch.randn(e_total, 128, generator=gen)[lg.edge_ids]
    coef = torch.randn(n, 128, generator=gen)[lg.owned].to(dev)
    weights = synthetic.seeded_state_dict(synthetic.processor_shapes(layers, ["mesh_edges"], "sum"), seed=17)
    shell = MeshGraphNet(3, 128, 2, "sum", layers, "none", ["mesh_edges"])
    proc = shell.processor
    proc.load_state_dict({k[len("processor."):]: t for k, t in weights.items()})
    proc = proc.to(dev)
    proc.precision = "bf16"
    plan = HaloPlan(lg, dev)
    use_peer = os.environ.get("HGN_HALO", "peer") == "peer"          # "nccl": the generic path (grouped send/recv before every block)
    peer = PeerHalo(lg, layers, dev) if use_peer else None
    model = PartitionedProcessor(proc, plan, peer)
    params = list(proc.parameters())
    v_dev, e_dev = v0.to(dev).to(torch.bfloat16), e0.to(dev).to(torch.bfloat16)     # resident: the dtype the path computes in
    v_host, e_host = v0.pin_memory(), e0.pin_memory()                                # e2e: fp32 host buffers
    s_loc, r_loc = lg.senders.to(dev), lg.receivers.to(dev)
    loss_host = torch.empty(1).pin_memory()

    kept = {}

    def step(v_in, e_in, keep=False):
        for p in params:
            p.grad = None
        v = v_in.requires_grad_(True)
        ed = e_in.requires_grad_(True)
        out_v, out_sets = model(v, [EdgeSet("mesh_edges", ed, s_loc, r_loc)])
        loss = (out_v * coef).sum() + out_sets[0].features.sum() * 1e-3
        loss.backward()
        allreduce_gradients(proc)
        if keep:
            kept.update(out_v=out_v.detach(), grad_v=v.grad.detach())
        return loss

    def timed(fn, steps):
        dist.barrier()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(steps):
            fn()
        b.record()
        dist.barrier()
        torch.cuda.synchronize()
        ms = torch.tensor([a.elapsed_time(b) / steps], device=dev)
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms)

    for _ in range(max(args.warmup, 3)):
        step(v_dev.detach(), e_dev.detach())
    from . import _cabi
    launches0 = ops.launch_count
    with clock_sampler_cls(dev.index) as clocks:
        ms_per_step = timed(lambda: step(v_dev.detach(), e_dev.detach()), args.steps)
    launches = ops.launch_count - launches0
    # per-kernel times from a second pass of the same steps: at several ranks the kernels are short and the two CUDA events the
    # library records around every launch would make the timed region host-bound
    _cabi.profile(True)
    timed(lambda: step(v_dev.detach(), e_dev.detach()), args.steps)
    kernels = _cabi.profile_report()
    _cabi.profile(False)
    roofline = roofline_fn(kernels, args.steps, int(lg.edge_ids.numel()), int(lg.owned.numel()), peaks) if roofline_fn else None

    copy_stream = torch.cuda.Stream(device=dev)

    def upload():
        with torch.cuda.stream(copy_stream):
            v, ed = v_host.to(dev, non_blocking=True), e_host.to(dev, non_blocking=True)
            ready = torch.cuda.Event()
            ready.record(copy_stream)
        return v, ed, ready

    e2e_steps = max(2, min(args.steps, 8))

    def run_e2e(steps=e2e_steps):
        """Every step's inputs cross PCIe inside the region (step i+1's copy overlaps step i) and every loss is read back."""
        nxt = upload()
        for i in range(steps):
            v, ed, ready = nxt
            if i + 1 < steps:
                nxt = upload()
            torch.cuda.current_stream().wait_event(ready)
            v.record_stream(torch.cuda.current_stream()); ed.record_stream(torch.cuda.current_stream())
            loss = step(v, ed)
            loss_host.copy_(loss.detach().reshape(1), non_blocking=True)
            torch.cuda.current_stream().synchronize()

    run_e2e(3)                                  # warm-up: two input sets are alive at a time, let the allocator cache both
    e2e_ms = timed(run_e2e, 1) / e2e_steps
    halo_rows = torch.tensor([float(lg.n_ghost)], device=dev)
    dist.all_reduce(halo_rows, op=dist.ReduceOp.MAX)
    # partition_check: one more (untimed) partitioned step; rank 0 then runs the SAME step on the whole mesh on its one GPU and
    # compares its owned rows (latents and their gradients) and the all-reduced weight gradients
    step(v_dev.detach(), e_dev.detach(), keep=True)
    part_grads = [p.grad.detach().clone() for p in params]
    torch.cuda.synchronize()
    dist.barrier()
    check = None
    if rank == 0:
        gen = torch.Generator().manual_seed(0)
        v_full = torch.randn(n, 128, generator=gen)
        e_full = torch.randn(e_total, 128, generator=gen)
        coef_full = torch.randn(n, 128, generator=gen).to(dev)
        for p in params:
            p.grad = None
        vf = v_full.to(dev).requires_grad_(True)
        ef = e_full.to(dev).requires_grad_(True)
        from .util import MultiGraph
        out = proc(MultiGraph([vf], [EdgeSet("mesh_edges", ef, senders.to(dev), receivers.to(dev))]))
        ((out.node_features[0] * coef_full).sum() + out.edge_sets[0].features.sum() * 1e-3).backward()
        own = lg.owned.to(dev)

        def rel(a, b):
            return float((a.float() - b.float()).norm() / b.float().norm().clamp_min(1e-30))
        check = {"latents_owned_rows": rel(kept["out_v"], out.node_features[0].detach()[own]),
                 "latent_gradients_owned_rows": rel(kept["grad_v"], vf.grad[own]),
                 "weight_gradients_worst": max(rel(a, p.grad) for a, p in zip(part_grads, params)),
                 "metric": "relative L2, partitioned vs the same bf16 step on one GPU (rank 0's owned rows; all-reduced weight gradients)"}
        check["value"] = max(check["latents_owned_rows"], check["latent_gradients_owned_rows"], check["weight_gradients_worst"])
        del vf, ef, out
        torch.cuda.empty_cache()
    dist.barrier()
    extra = extra_leg(world, rank, dev) if extra_leg is not None else None      # e.g. the data-parallel cfg4 leg (all ranks take part)
    if rank == 0:
        value = e_total * layers / (ms_per_step * 1e-3)
        print(json.dumps({
            "metric": metric, "value": value, "unit": unit, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "bf16",
            "data": "synthetic (seeded 1000x1000 triangulated grid, seeded weights)",
            "config": {"workload": "cfg5: 1M-node / 5 992 002-edge triangulated mesh, 15 GraphNet layers, sum aggregator, processor fwd+bwd",
                       "nodes": n, "edges": e_total, "layers": layers, "latent": 128,
                       "partitioning": f"edge-cut, {world} row slabs, receiver-owner rule, one-ring halo per layer (max {int(halo_rows)} ghost "
                                       f"rows per rank): " + ("rows of the sender table Ps pushed into the peers' tables over NVLink peer memory by a "
                                       "kernel of the sending rank + flags (csrc/peer.cu), ghost gradients return the same way" if use_peer else
                                       "node latents by NCCL grouped send/recv before each block") + ", weight-gradient all-reduce (NCCL)",
                       "l2_policy": "inputs larger than L2"},
            "e2e": {"value": e_total * layers / (e2e_ms * 1e-3), "unit": unit, "ms_per_step": e2e_ms,
                    "h2d_bytes_per_step": int((v_host.numel() + e_host.numel()) * 4), "d2h_bytes_per_step": 4},
            "gpu_launches": launches, "clocks": clocks.summary(),
            "roofline": roofline, "cpu_baseline": None, "partition_check": check, "data_parallel_cfg4": extra,
            "kernels": [{"name": k["name"], "launches": k["launches"], "ms_per_step": k["ms"] / args.steps} for k in kernels],
            "kernel_times": "second pass of the same steps with the library's per-launch CUDA events enabled",
        }))
    if peer is not None:
        peer.close()
    dist.destroy_process_group()
