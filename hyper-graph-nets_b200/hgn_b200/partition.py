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

import ctypes
from dataclasses import dataclass
from typing import Dict, List, NamedTuple, Optional, Sequence

import torch
import torch.distributed as dist

from . import _cabi, ops
from ._cabi import HgnError


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


HYPER_REMOTE_SETS = ("intra_cluster_to_cluster", "inter_cluster", "intra_cluster_to_mesh")


class LocalEdges(NamedTuple):
    edge_ids: torch.Tensor         # [e_loc] global ids of the local edges (ascending)
    senders: torch.Tensor          # [e_loc] local sender index into [owned | hyper]
    receivers: torch.Tensor        # [e_loc] local receiver index into [owned | hyper]


@dataclass
class LocalHyperGraph:
    """One rank's share of a HyperGraphNet graph.  The mesh edges follow ``build_local_graph``; in the remote edge sets the local node
    list is ``[owned | hyper]`` (hyper node c is local row ``n_own + c``, the reference's ``[mesh, hyper]`` layout), and
    ``intra_cluster_to_cluster`` keeps the edges of an owned sender, ``intra_cluster_to_mesh`` those of an owned receiver and
    ``inter_cluster`` every edge."""
    mesh: LocalGraph
    num_clusters: int
    remote: Dict[str, LocalEdges]

    @property
    def n_own(self) -> int:
        return self.mesh.n_own


def build_local_hyper_graph(index_lists, num_nodes: int, num_clusters: int, part: torch.Tensor, rank: int, world: int) -> LocalHyperGraph:
    """Rank ``rank``'s share of the four edge sets of a HyperGraphNet graph.  ``index_lists``: set name -> global ``(senders,
    receivers)``, with hyper node c numbered ``num_nodes + c`` (``rmp.hierarchical_connector.connector_indices``)."""
    names = set(index_lists)
    if names != {"mesh_edges", *HYPER_REMOTE_SETS}:
        raise HgnError(f"build_local_hyper_graph: edge sets must be exactly mesh_edges and {', '.join(HYPER_REMOTE_SETS)}; got {sorted(names)}")
    part = part.cpu()
    mesh = build_local_graph(*index_lists["mesh_edges"], part, rank, world)
    n_own = mesh.n_own
    local_of = torch.full((num_nodes,), -1, dtype=torch.int64)
    local_of[mesh.owned] = torch.arange(n_own)
    mesh_side = {"intra_cluster_to_cluster": (True, False), "inter_cluster": (False, False), "intra_cluster_to_mesh": (False, True)}
    remote = {}
    for name in HYPER_REMOTE_SETS:
        s, r = (t.cpu().to(torch.int64) for t in index_lists[name])
        mesh_s, mesh_r = mesh_side[name]
        for ids, is_mesh in ((s, mesh_s), (r, mesh_r)):
            lo, hi = (0, num_nodes) if is_mesh else (num_nodes, num_nodes + num_clusters)
            if ids.numel() and (int(ids.min()) < lo or int(ids.max()) >= hi):
                raise HgnError(f"build_local_hyper_graph: {name} indices outside [{lo}, {hi})")
        owner_side = s if mesh_s else (r if mesh_r else None)
        edge_ids = torch.arange(s.numel()) if owner_side is None else torch.nonzero(part[owner_side] == rank).flatten()
        loc = lambda ids, is_mesh: local_of[ids] if is_mesh else n_own + (ids - num_nodes)
        remote[name] = LocalEdges(edge_ids, loc(s[edge_ids], mesh_s), loc(r[edge_ids], mesh_r))
    return LocalHyperGraph(mesh=mesh, num_clusters=int(num_clusters), remote=remote)


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
    """The halo of one (step, layer) of a ``PeerHalo``, in the form ``ops.graphnet_layer`` takes it."""
    peer: PeerHalo
    step: int
    layer: int

    def sender_table(self) -> torch.Tensor:
        return self.peer.table(self.step & 1, self.layer)

    def exchange_forward(self) -> None:
        self.peer.push_forward(self.step, self.layer)

    def exchange_backward(self, gs: torch.Tensor) -> None:
        self.peer.push_backward(self.step, self.layer, gs)


class PeerPool:
    """Every rank's ``[C, W]`` rows of one cross-rank cluster exchange, in NVLink peer memory (csrc/peer.cu).  A partitioned
    HyperGraphNet block has three such exchanges: the fp32 partials of its cluster pooling (forward, ``POOL``), and in the backward pass
    the gradients of the replicated hyper rows its down-edge senders (``DOWN``) and up-edge receivers (``UP``) read.  Each rank pushes
    its rows into slot ``rank`` of every rank's pool (its own included) with ``hgn_halo_push``, waits for the peers' flags with
    ``hgn_halo_wait``, and reduces slots ``0 .. world-1`` in rank order: every rank runs the same arithmetic on the same bytes.

    Pool layout (bytes): ``[flags: 3 directions x world uint32 | push counter | per (step parity, layer): POOL world x C x 388 fp32,
    DOWN and UP world x C x 128 bf16]``.  Slots are per (step parity, layer, direction), like ``PeerHalo``'s tables, and every rank
    waits for every other in each exchange, so no rank can be far enough ahead to overwrite rows that are still to be read.  Unlike
    ``PeerHalo``, every peer is mapped."""

    POOL, DOWN, UP = 0, 1, 2

    def __init__(self, num_clusters: int, layers: int, device, group=None):
        lib = _cabi.load()
        self.C, self.layers, self.group, self.device = int(num_clusters), int(layers), group, torch.device(device)
        self.world, self.rank = dist.get_world_size(group), dist.get_rank(group)
        if self.world > _cabi.HGN_MAX_PEERS:
            raise HgnError(f"PeerPool: {self.world} ranks, at most {_cabi.HGN_MAX_PEERS}")
        self.row_bytes = {self.POOL: _cabi.HGN_SEGMENT_PARTIAL_WIDTH * 4, self.DOWN: ops.D_LATENT * 2, self.UP: ops.D_LATENT * 2}
        self.dir_off, off = {}, 0
        for d in (self.POOL, self.DOWN, self.UP):
            self.dir_off[d] = off
            off += self.world * self.C * self.row_bytes[d]
        self.layer_bytes = 256 * ((off + 255) // 256)
        self.off_counter = 3 * self.world * 4
        self.off_slots = 256 * ((self.off_counter + 4 + 255) // 256)
        self.nbytes = self.off_slots + 2 * self.layers * self.layer_bytes
        with torch.cuda.device(self.device):
            ptr = ctypes.c_void_p()
            handle = ctypes.create_string_buffer(64)
            _cabi.check(lib.hgn_peer_alloc(self.nbytes, ctypes.byref(ptr), handle), "hgn_peer_alloc")
        self.base = int(ptr.value)
        self.pool = torch.as_tensor(_DeviceBytes(self.base, self.nbytes), device=self.device)
        handles = [None] * self.world
        dist.all_gather_object(handles, bytes(handle.raw), group=group)
        self.peer_base = [0] * self.world
        with torch.cuda.device(self.device):
            for q in range(self.world):
                if q != self.rank:
                    mapped = ctypes.c_void_p()
                    _cabi.check(lib.hgn_peer_open(handles[q], ctypes.byref(mapped)), "hgn_peer_open")
                    self.peer_base[q] = int(mapped.value)
        self.index32 = torch.arange(self.C, dtype=torch.int32).repeat(self.world).to(self.device)
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

    def _slot_offset(self, step: int, layer: int, direction: int) -> int:
        return self.off_slots + ((step & 1) * self.layers + layer) * self.layer_bytes + self.dir_off[direction]

    def exchange(self, rows: torch.Tensor, step: int, layer: int, direction: int) -> torch.Tensor:
        """Pushes ``rows`` ([C, W], contiguous: fp32 partials for ``POOL``, bf16 gradients otherwise) into slot ``rank`` of every rank's
        pool, waits for the other ranks' rows and returns this rank's ``[world, C, W]`` view of all of them, in rank order."""
        lib = _cabi.load()
        off, rb = self._slot_offset(step, layer, direction), self.row_bytes[direction]
        assert rows.is_contiguous() and rows.shape[0] == self.C and rows.shape[1] * rows.element_size() == rb
        # epochs rise within a direction: the forward visits the layers in ascending order, the backward in descending order
        epoch = (1 + step * self.layers + (layer if direction == self.POOL else self.layers - 1 - layer)) & 0x7FFFFFFF
        peers, flags = _cabi.HaloPeers(), _cabi.HaloFlags()
        n_wait = 0
        for q in range(self.world):
            base = self.base if q == self.rank else self.peer_base[q]
            peers.dst[q] = base + off + self.rank * self.C * rb
            peers.flag[q] = None if q == self.rank else base + (direction * self.world + self.rank) * 4
            peers.row_begin[q] = q * self.C
            if q != self.rank:
                flags.flag[n_wait] = self.base + (direction * self.world + q) * 4
                n_wait += 1
        peers.row_begin[self.world] = self.world * self.C
        with torch.cuda.device(self.device):
            st = _cabi.stream_ptr()
            _cabi.check(lib.hgn_halo_push(_cabi.dtype_code(rows.dtype), rows.data_ptr(), self.index32.data_ptr(), rows.shape[1], ctypes.byref(peers),
                                          self.world, epoch, self.base + self.off_counter, st), "hgn_halo_push")
            _cabi.check(lib.hgn_halo_wait(ctypes.byref(flags), n_wait, epoch, st), "hgn_halo_wait")
        ops._count(1 + int(n_wait > 0))               # csrc/peer.cu: one push kernel, one wait kernel when there are peers
        n = self.world * self.C * rb
        return self.pool[off: off + n].view(rows.dtype).view(self.world, self.C, rows.shape[1])


class _ClusterPool(torch.autograd.Function):
    """The cluster pooling of the up edges across ranks: this rank's fp32 partials (``hgn_segment_partials`` over its own up edges,
    keyed by cluster) -> every rank's pool -> ``hgn_cluster_combine`` in rank order -> the bf16 ``[C, 128]`` aggregates of ``reducers``,
    bit-identical on every rank.  Backward: each rank's partial receives the full gradient of the aggregates ('mean' divided by the
    global count; max / min only where this rank holds the winner, as the combine cleared the other winners), through the existing
    segment backward over the local elements."""

    @staticmethod
    def forward(ctx, e, plan, pool: PeerPool, step, layer, reducers):
        C, dev = plan.num_segments, e.device
        minmax = "max" in reducers or "min" in reducers
        winners = minmax and ctx.needs_input_grad[0]
        new_arg = lambda op: torch.empty((C, ops.D_LATENT), dtype=torch.int32, device=dev) if winners and op in reducers else None
        argmax, argmin = new_arg("max"), new_arg("min")
        partial = torch.empty((C, _cabi.HGN_SEGMENT_PARTIAL_WIDTH), dtype=torch.float32, device=dev)
        outs = {op: torch.empty((C, ops.D_LATENT), dtype=torch.bfloat16, device=dev) for op in reducers}
        count = torch.empty(C, dtype=torch.int32, device=dev)
        with torch.cuda.device(dev):
            ops._segment_partials(e, plan, partial, minmax, argmax, argmin)
            slots = pool.exchange(partial, step, layer, PeerPool.POOL)
            ops._cluster_combine(slots, pool.world, pool.rank, [outs.get(op) for op in ops.OP_BITS], argmax, argmin, count)
        ctx.save_for_backward(argmax, argmin, count)
        ctx.plan, ctx.reducers, ctx.E = plan, reducers, e.shape[0]
        return tuple(outs[op] for op in reducers)

    @staticmethod
    def backward(ctx, *grads):
        argmax, argmin, count = ctx.saved_tensors
        g = {op: gi.contiguous().to(torch.bfloat16) for op, gi in zip(ctx.reducers, grads) if gi is not None}
        ref = next(iter(g.values()))
        grad = torch.empty((ctx.E, ops.D_LATENT), dtype=torch.bfloat16, device=ref.device)
        with torch.cuda.device(ref.device):
            g_sum = g.get("sum")
            if "mean" in g:
                g_sum_mean = torch.empty_like(g["mean"])
                ops._cluster_mean_grad(g_sum, g["mean"], count, g_sum_mean)
                g_sum = g_sum_mean
            ops._segment_backward(ctx.plan, ctx.E, g_sum, g.get("max"), g.get("min"), argmax if "max" in g else None,
                                  argmin if "min" in g else None, grad)
        return grad, None, None, None, None, None


class _EnterLocal(torch.autograd.Function):
    """Where the replicated hyper rows feed rank-local edges: the identity forward; backward, the rank-ordered sum of every rank's
    gradient (``hgn_cluster_grad_sum``), so the gradient that reaches the replicated computation is complete and the same on every
    rank."""

    @staticmethod
    def forward(ctx, h, pool: PeerPool, step, layer, direction):
        ctx.pool, ctx.step, ctx.layer, ctx.direction = pool, step, layer, direction
        return h.view_as(h)

    @staticmethod
    def backward(ctx, g):
        g = g.contiguous().to(torch.bfloat16)
        out = torch.empty_like(g)
        with torch.cuda.device(g.device):
            slots = ctx.pool.exchange(g, ctx.step, ctx.layer, ctx.direction)
            ops._cluster_grad_sum(slots, out)
        return out, None, None, None, None


_HYPER_SCOPE = ("the partitioned processor takes plain GraphNet blocks, or HyperGraphNet blocks with edge sets exactly mesh_edges, "
                "intra_cluster_to_cluster, inter_cluster and intra_cluster_to_mesh, the 'sum', 'mean', 'max', 'min' or 'pna' aggregator, "
                "bf16 latents of width 128, a PeerHalo and the rank's LocalHyperGraph (build_local_hyper_graph); HeteroGraphNet, "
                "MultiScaleGraphNet, world_edges and fp32 parity mode are not supported")


class _HyperLocal:
    """Device-side index tensors and segment plans of a ``LocalHyperGraph`` (the tensors stay referenced: plans are cached by them)."""

    def __init__(self, hyper: LocalHyperGraph, device):
        from .plan import segment_plan
        n_own, C = hyper.n_own, hyper.num_clusters
        self.n_own, self.C = n_own, C

        def plans(s, r, n):
            s, r = s.to(device), r.to(device)
            return s, r, segment_plan(s, n), segment_plan(r, n)
        rem = hyper.remote
        self.up = plans(rem["intra_cluster_to_cluster"].senders, rem["intra_cluster_to_cluster"].receivers, n_own + C)
        self.down = plans(rem["intra_cluster_to_mesh"].senders, rem["intra_cluster_to_mesh"].receivers, n_own + C)
        # the across phase runs on the C hyper rows alone: every rank computes it from the same rows
        self.across = plans(rem["inter_cluster"].senders - n_own, rem["inter_cluster"].receivers - n_own, C)
        self.cluster_ids = (rem["intra_cluster_to_cluster"].receivers - n_own).to(device)
        self.cluster_plan = segment_plan(self.cluster_ids, C)


def _edge(block, name, v, e, s_plan, r_plan, want_agg):
    from .migration.graphnet import _mlp_parameters, _packed_cache
    model = block.edge_models[name]
    return ops.edge_update(_mlp_parameters(model, 3 * v.shape[1], v), _packed_cache(model), v, e, s_plan, r_plan, want_agg)


def _node(model, rows, aggs):
    from .migration.graphnet import _mlp_parameters, _packed_cache
    return ops.node_update(_mlp_parameters(model, (1 + len(aggs)) * rows.shape[1], rows), _packed_cache(model), rows, aggs)


class PartitionedProcessor(torch.nn.Module):
    """Runs a (reference-API) ``Processor`` on one rank's share of the graph.

    Generic path (any block type, any aggregator, fp32 or bf16): ghosts are refreshed before every block with a grouped NCCL
    send/recv; the block itself is unchanged (it sees ``[owned | ghosts]`` as ``[mesh | hyper]`` rows).
    Fast path (``PeerHalo`` given, and every block takes the whole-layer route of ``GraphNet``: one edge set, bf16, any of the
    'sum' / 'mean' / 'max' / 'min' / 'pna' aggregators -- the cfg5 benchmark): ``ops.graphnet_layer`` per block with the halo of that
    layer; halo rows travel as peer-memory stores issued by a kernel of the sending rank.  Every edge of an owned receiver is local,
    so the aggregates (max / min winners included) need no exchange of their own.
    HyperGraphNet path (``hyper`` = this rank's ``LocalHyperGraph``, a ``PeerHalo`` given): ``_hyper_block`` per block, with the C hyper
    rows replicated on every rank and the cluster pooling combined across ranks through a ``PeerPool`` (DESIGN.md s6.1).  Other
    hierarchical blocks raise ``HgnError``."""

    def __init__(self, processor: torch.nn.Module, plan: HaloPlan, peer: Optional[PeerHalo] = None, hyper: Optional[LocalHyperGraph] = None):
        super().__init__()
        from .migration.graphnet import PNA_OPS
        from .migration.heterographnet import HeteroGraphNet
        from .migration.hypergraphnet import HyperGraphNet
        from .migration.multiscalegraphnet import MultiScaleGraphNet
        self.processor = processor
        self.plan = plan
        self.peer = peer
        self.hyper = self.pool = None
        blocks = list(processor.graphnet_blocks)
        if hyper is not None or any(isinstance(b, (HyperGraphNet, HeteroGraphNet, MultiScaleGraphNet)) for b in blocks):
            # the generic route would read a HyperGraphNet's hyper slot as the ghosts: only the schedule of _hyper_block is right
            sets = {"mesh_edges", *HYPER_REMOTE_SETS}
            if not all(type(b) is HyperGraphNet and set(b.edge_models.keys()) == sets and b.message_passing_aggregator in PNA_OPS + ("pna",)
                       for b in blocks) or peer is None or hyper is None:
                raise HgnError(_HYPER_SCOPE)
            self.hyper = _HyperLocal(hyper, peer.device)
            self.pool = PeerPool(hyper.num_clusters, len(blocks), peer.device, peer.group)
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

    def replicated_parameters(self) -> List[torch.nn.Parameter]:
        """The parameters every rank computes redundantly from the same rows (the hyper-node MLPs and the ``inter_cluster`` edge MLP of a
        HyperGraphNet block): their gradients are complete and identical on every rank, so ``allreduce_gradients`` leaves them out."""
        if self.hyper is None:
            return []
        return [p for b in self.processor.graphnet_blocks
                for m in (b.hyper_node_model_up, b.hyper_node_model_cross, b.edge_models["inter_cluster"]) for p in m.parameters()]

    def close(self) -> None:
        """Frees the cluster exchange pool of a HyperGraphNet processor (the ``PeerHalo`` belongs to the caller)."""
        if self.pool is not None:
            self.pool.close()

    def forward(self, owned: torch.Tensor, edge_sets, hyper_nodes: Optional[torch.Tensor] = None):
        """``(owned', edge_sets')``; for HyperGraphNet blocks ``(owned', edge_sets', hyper')`` from the C replicated hyper rows
        ``hyper_nodes`` (the same on every rank), with the edge sets' local indices of ``build_local_hyper_graph``."""
        if self.hyper is not None:
            return self._hyper_forward(owned, edge_sets, hyper_nodes)
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
                owned, e = block._layer(owned, e, es.name, self.peer.s_plan, self.peer.r_plan, PeerLayerHalo(self.peer, step, layer))
            return owned.to(in_dtype), [es._replace(features=e)]
        graph = MultiGraph([owned, None], list(edge_sets))
        for block in self.processor.graphnet_blocks:
            graph.node_features[1] = halo_exchange(graph.node_features[0], self.plan)
            graph = block(graph)
        out_nodes = graph.node_features[0].to(in_dtype)
        return out_nodes, list(graph.edge_sets)      # edge latents stay in the compute dtype (see Processor.forward)

    def _hyper_forward(self, owned, edge_sets, hyper_nodes):
        from . import config
        precision = getattr(self.processor, "precision", None) or config.precision()
        names = [es.name for es in edge_sets]
        if precision != "bf16" or hyper_nodes is None or sorted(names) != sorted(("mesh_edges",) + HYPER_REMOTE_SETS):
            raise HgnError(_HYPER_SCOPE + f" (got precision {precision!r}, edge sets {names}, hyper rows {'given' if hyper_nodes is not None else 'missing'})")
        in_dtype = owned.dtype
        owned, hyper = owned.to(torch.bfloat16), hyper_nodes.to(torch.bfloat16)
        feats = {es.name: es.features.to(torch.bfloat16) for es in edge_sets}
        step = self.peer.steps_done
        self.peer.steps_done += 1
        for layer, block in enumerate(self.processor.graphnet_blocks):
            owned, hyper = self._hyper_block(block, step, layer, owned, hyper, feats)
        # edge latents stay in the compute dtype (see Processor.forward); both node lists go back, like Processor.forward's
        return owned.to(in_dtype), [es._replace(features=feats[es.name]) for es in edge_sets], hyper.to(in_dtype)

    def _hyper_block(self, block, step, layer, owned, hyper, feats):
        """One HyperGraphNet block (hypergraphnet.py) on this rank's share; ``feats`` (set name -> edge latents) is updated in place.
        The mesh phase is the fused layer with the NVLink halo; the up phase pools its owned members' edges into fp32 partials combined
        across ranks; the across phase (C rows, ~C^2 edges) runs on every rank from the same rows; the down phase is local."""
        h = self.hyper
        agg = block.message_passing_aggregator
        reducers = tuple(ops.OP_BITS) if agg == "pna" else (agg,)
        peer, pool = self.peer, self.pool
        # mesh phase (hypergraphnet.py:29-34)
        owned, feats["mesh_edges"] = block._layer(owned, feats["mesh_edges"], "mesh_edges", peer.s_plan, peer.r_plan,
                                                  PeerLayerHalo(peer, step, layer))
        # node -> hyper-node pooling (:37-39)
        _, _, s_plan, r_plan = h.up
        v = torch.cat([owned, _EnterLocal.apply(hyper, pool, step, layer, PeerPool.UP)])
        feats["intra_cluster_to_cluster"], _ = _edge(block, "intra_cluster_to_cluster", v, feats["intra_cluster_to_cluster"], s_plan, r_plan, False)
        pooled = _ClusterPool.apply(feats["intra_cluster_to_cluster"], h.cluster_plan, pool, step, layer, reducers)
        hyper = _node(block.hyper_node_model_up, hyper, list(pooled))
        # hyper-node <-> hyper-node (:42-47), on the C hyper rows alone
        _, _, s_plan, r_plan = h.across
        feats["inter_cluster"], a = _edge(block, "inter_cluster", hyper, feats["inter_cluster"], s_plan, r_plan, agg == "sum")
        hyper = _node(block.hyper_node_model_cross, hyper, [a] if agg == "sum" else ops.segment_aggregate(feats["inter_cluster"], r_plan, reducers))
        # hyper-node -> node broadcast (:50-52)
        _, _, s_plan, r_plan = h.down
        v = torch.cat([owned, _EnterLocal.apply(hyper, pool, step, layer, PeerPool.DOWN)])
        feats["intra_cluster_to_mesh"], a = _edge(block, "intra_cluster_to_mesh", v, feats["intra_cluster_to_mesh"], s_plan, r_plan, agg == "sum")
        aggs = [a] if agg == "sum" else ops.segment_aggregate(feats["intra_cluster_to_mesh"], r_plan, reducers)
        owned = _node(block.node_model_down, owned, [x[:h.n_own] for x in aggs])
        return owned, hyper


def allreduce_gradients(module: torch.nn.Module, group=None, exclude: Sequence[torch.nn.Parameter] = ()) -> None:
    """Sum the per-rank partial weight gradients (one flat fp32 all-reduce).  ``exclude``: parameters whose gradients are already
    complete on every rank (``PartitionedProcessor.replicated_parameters``)."""
    skip = {id(p) for p in exclude}
    grads = [p.grad for p in module.parameters() if p.grad is not None and id(p) not in skip]
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
    weights = synthetic.seeded_state_dict(synthetic.processor_shapes(layers, ["mesh_edges"], args.aggregator), seed=17)
    shell = MeshGraphNet(3, 128, 2, args.aggregator, layers, "none", ["mesh_edges"])
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
            "config": {"workload": f"cfg5: 1M-node / 5 992 002-edge triangulated mesh, 15 GraphNet layers, {args.aggregator} aggregator, "
                                   "processor fwd+bwd",
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
