"""Seeded synthetic meshes, latents and weights (SURVEY.md s8d "Synthetic inputs").

There is no dataset in the reference tree (``data/*/input`` are empty placeholders), so every test
and benchmark runs on the shapes below.  Everything is derived from explicit seeds with numpy's
``default_rng`` so that the build container, the GPU box and the golden fixtures agree bit for bit
without shipping weight tensors.
"""
from __future__ import annotations

import zlib
from typing import Dict, Sequence, Tuple

import numpy as np
import torch


# ----------------------------------------------------------------------------------------------
# meshes
# ----------------------------------------------------------------------------------------------
def grid_triangles(width: int, height: int) -> np.ndarray:
    """Two triangles per quad of a ``width x height`` node grid (row-major node ids), int32 [F,3].
    40x40 -> 1600 nodes / 3042 triangles / 9282 directed edges (~flag_simple)."""
    i, j = np.meshgrid(np.arange(height - 1), np.arange(width - 1), indexing="ij")
    a = (i * width + j).ravel()
    b = a + 1
    c = a + width
    d = c + 1
    tris = np.concatenate([np.stack([a, b, d], 1), np.stack([a, d, c], 1)], 0)
    return tris.astype(np.int32)


def grid_edges_two_way(width: int, height: int) -> Tuple[torch.Tensor, torch.Tensor]:
    """Closed form of ``triangles_to_edges(grid_triangles(w, h))['two_way_connectivity']`` for meshes
    too large for a sort-based ``unique`` on the host: unique (max,min) pairs in lexicographic order,
    then the reversed copies (src/util.py:60-69).  Tested against the sort-based path."""
    n = width * height
    ids = np.arange(n, dtype=np.int64)
    col = ids % width
    row = ids // width
    # for a node `hi`, the smaller-id neighbours are: hi-width-1 (diag), hi-width (up), hi-1 (left)
    cand_lo = []
    cand_hi = []
    for off, ok in ((-(width + 1), (row > 0) & (col > 0)), (-width, row > 0), (-1, col > 0)):
        cand_hi.append(ids[ok])
        cand_lo.append(ids[ok] + off)
    hi = np.concatenate(cand_hi)
    lo = np.concatenate(cand_lo)
    order = np.lexsort((lo, hi))
    s = torch.from_numpy(hi[order])
    r = torch.from_numpy(lo[order])
    return torch.cat((s, r)), torch.cat((r, s))


def cloth_frame(width: int, height: int, seed: int = 0) -> Dict[str, torch.Tensor]:
    """One flag-style frame: ``cells, mesh_pos[N,2], world_pos[N,3], prev|world_pos, target|world_pos,
    node_type[N,1]`` (first grid column = HANDLE 3, else NORMAL 0)."""
    rng = np.random.default_rng(seed)
    n = width * height
    jj, ii = np.meshgrid(np.arange(width), np.arange(height))
    mesh_pos = 0.1 * np.stack([jj.ravel(), ii.ravel()], 1).astype(np.float32)
    world = np.concatenate([mesh_pos, 0.01 * rng.standard_normal((n, 1)).astype(np.float32)], 1)
    prev = world + 0.001 * rng.standard_normal((n, 3)).astype(np.float32)
    target = world + 0.001 * rng.standard_normal((n, 3)).astype(np.float32)
    node_type = np.zeros((n, 1), np.int32)
    node_type[jj.ravel() == 0] = 3
    return {
        "cells": torch.from_numpy(grid_triangles(width, height)),
        "mesh_pos": torch.from_numpy(mesh_pos),
        "world_pos": torch.from_numpy(world.astype(np.float32)),
        "prev|world_pos": torch.from_numpy(prev.astype(np.float32)),
        "target|world_pos": torch.from_numpy(target.astype(np.float32)),
        "node_type": torch.from_numpy(node_type),
    }


def box_tetrahedra(nx: int, ny: int, nz: int) -> np.ndarray:
    """Five-free simple split: six tetrahedra per cell of an ``nx x ny x nz`` node lattice, int32 [F,4]."""
    def nid(i, j, k):
        return (k * ny + j) * nx + i
    cells = []
    for k in range(nz - 1):
        for j in range(ny - 1):
            for i in range(nx - 1):
                v = [nid(i, j, k), nid(i + 1, j, k), nid(i + 1, j + 1, k), nid(i, j + 1, k),
                     nid(i, j, k + 1), nid(i + 1, j, k + 1), nid(i + 1, j + 1, k + 1), nid(i, j + 1, k + 1)]
                for t in ((0, 1, 2, 6), (0, 2, 3, 6), (0, 3, 7, 6), (0, 7, 4, 6), (0, 4, 5, 6), (0, 5, 1, 6)):
                    cells.append([v[t[0]], v[t[1]], v[t[2]], v[t[3]]])
    return np.asarray(cells, np.int32)


def plate_frame(plate=(9, 9, 2), obstacle=(4, 4, 2), spacing: float = 0.02, gap: float = 0.012, seed: int = 0) -> Dict[str, torch.Tensor]:
    """Two-body deforming-plate frame in one index space (SURVEY.md s8d, cfg 3): a NORMAL plate lattice (its first lattice column
    HANDLE) and an OBSTACLE block hovering `gap` above it, the obstacle nodes contiguous at the end
    (src/rmp/remote_message_passing.py:82-137 requires that).  Tetrahedral cells, seeded jitter; spacing and gap are chosen so
    that mesh neighbours, plate-obstacle pairs and some non-edges all lie around the 0.03 world-edge radius (plate.py:87)."""
    rng = np.random.default_rng(seed)

    def lattice(dims, origin):
        nx, ny, nz = dims
        k, j, i = np.meshgrid(np.arange(nz), np.arange(ny), np.arange(nx), indexing="ij")
        return np.stack([i, j, k], -1).reshape(-1, 3).astype(np.float32) * np.float32(spacing) + np.asarray(origin, np.float32)

    p_pos = lattice(plate, (0.0, 0.0, 0.0))
    o_pos = lattice(obstacle, (2.3 * spacing, 1.7 * spacing, (plate[2] - 1) * spacing + gap))
    n_plate = p_pos.shape[0]
    mesh_pos = np.concatenate([p_pos, o_pos], 0)
    world_pos = mesh_pos + rng.normal(0.0, 0.1 * spacing, mesh_pos.shape).astype(np.float32)
    target = world_pos + rng.normal(0.0, 0.001, mesh_pos.shape).astype(np.float32)
    node_type = np.zeros((mesh_pos.shape[0], 1), np.int32)
    node_type[:n_plate][np.arange(n_plate) % plate[0] == 0, 0] = 3   # HANDLE
    node_type[n_plate:, 0] = 1                                     # OBSTACLE
    cells = np.concatenate([box_tetrahedra(*plate), box_tetrahedra(*obstacle) + n_plate], 0).astype(np.int32)
    return {
        "cells": torch.from_numpy(cells),
        "mesh_pos": torch.from_numpy(mesh_pos.astype(np.float32)),
        "world_pos": torch.from_numpy(world_pos.astype(np.float32)),
        "target|world_pos": torch.from_numpy(target.astype(np.float32)),
        "node_type": torch.from_numpy(node_type),
    }


def cylinder_frame(width: int, height: int, seed: int = 0) -> Dict[str, torch.Tensor]:
    """One cylinder_flow-style Eulerian frame (SURVEY.md s8d, cfg 4): a triangulated ``width x height`` rectangle whose first
    column is INFLOW (4), last column OUTFLOW (5), first / last row and a block in the middle (the obstacle's rim)
    WALL_BOUNDARY (6), everything else NORMAL (0), so that all four types of src/model/cylinder.py:71-75 occur.
    ``velocity[N,2], target|velocity[N,2], pressure[N,1]`` are seeded noise around a uniform inflow."""
    rng = np.random.default_rng(seed)
    n = width * height
    jj, ii = np.meshgrid(np.arange(width), np.arange(height))
    jj, ii = jj.ravel(), ii.ravel()
    mesh_pos = 0.05 * np.stack([jj, ii], 1).astype(np.float32)
    node_type = np.zeros((n, 1), np.int32)
    node_type[(ii == 0) | (ii == height - 1), 0] = 6
    block = (abs(jj - width // 4) <= 1) & (abs(ii - height // 2) <= 1)
    node_type[block, 0] = 6
    node_type[jj == 0, 0] = 4
    node_type[jj == width - 1, 0] = 5
    velocity = (np.asarray([1.0, 0.0], np.float32) + 0.1 * rng.standard_normal((n, 2))).astype(np.float32)
    target = (velocity + 0.01 * rng.standard_normal((n, 2))).astype(np.float32)
    pressure = (0.5 * rng.standard_normal((n, 1))).astype(np.float32)
    return {
        "cells": torch.from_numpy(grid_triangles(width, height)),
        "mesh_pos": torch.from_numpy(mesh_pos),
        "node_type": torch.from_numpy(node_type),
        "velocity": torch.from_numpy(velocity),
        "target|velocity": torch.from_numpy(target),
        "pressure": torch.from_numpy(pressure),
    }


def trajectory(frames: Sequence[Dict[str, torch.Tensor]]) -> Dict[str, torch.Tensor]:
    """``[T, N, .]`` tensors per key from T frames of one mesh: the dict ``model.rollout`` takes (src/model/flag.py:194-197; static
    fields tiled over T like src/data/preprocessing.py:52-53)."""
    return {key: torch.stack([f[key] for f in frames], 0) for key in frames[0]}


# ----------------------------------------------------------------------------------------------
# deterministic tensors
# ----------------------------------------------------------------------------------------------
def _rng_for(name: str, seed: int) -> np.random.Generator:
    return np.random.default_rng([seed, zlib.crc32(name.encode())])


def seeded_tensor(name: str, shape: Sequence[int], seed: int = 0, scale: float = 1.0) -> torch.Tensor:
    return torch.from_numpy((scale * _rng_for(name, seed).standard_normal(tuple(shape))).astype(np.float32))


def seeded_state_dict(shapes: Dict[str, Sequence[int]], seed: int = 0) -> Dict[str, torch.Tensor]:
    """Weights as a pure function of (state_dict key, shape, seed).

    ``linear_k.weight`` ~ N(0, 1/fan_in) (keeps 15 LayerNorm'd residual layers well scaled), biases
    ~ 0.1 N(0,1); LayerNorm gain = 1 + 0.1 N(0,1), LayerNorm bias = 0.1 N(0,1) so that the affine part
    of the LayerNorm is exercised."""
    out = {}
    for key, shape in shapes.items():
        shape = tuple(int(s) for s in shape)
        z = _rng_for(key, seed).standard_normal(shape)
        if key.endswith(".weight") and len(shape) == 2:
            z = z / np.sqrt(shape[1])
        elif key.endswith(".weight"):
            z = 1.0 + 0.1 * z
        else:
            z = 0.1 * z
        out[key] = torch.from_numpy(z.astype(np.float32))
    return out


def mlp_shapes(prefix: str, in_features: int, latent: int = 128, out_features: int = 128,
               layer_norm: bool = True) -> Dict[str, Tuple[int, ...]]:
    """state_dict key -> shape for one reference MLP (``_make_mlp``, meshgraphnet.py:53-60)."""
    base = f"{prefix}.0.layers" if layer_norm else f"{prefix}.layers"
    shapes = {
        f"{base}.linear_0.weight": (latent, in_features), f"{base}.linear_0.bias": (latent,),
        f"{base}.linear_1.weight": (latent, latent), f"{base}.linear_1.bias": (latent,),
        f"{base}.linear_2.weight": (out_features, latent), f"{base}.linear_2.bias": (out_features,),
    }
    if layer_norm:
        shapes[f"{prefix}.1.weight"] = (out_features,)
        shapes[f"{prefix}.1.bias"] = (out_features,)
    return shapes


def processor_shapes(num_blocks: int, edge_sets: Sequence[str], aggregator: str = "sum", latent: int = 128,
                     prefix: str = "processor") -> Dict[str, Tuple[int, ...]]:
    """Shapes of a base-``GraphNet`` processor (one node MLP + one edge MLP per set and block)."""
    k = 4 if aggregator == "pna" else 1
    shapes: Dict[str, Tuple[int, ...]] = {}
    for b in range(num_blocks):
        p = f"{prefix}.graphnet_blocks.{b}"
        shapes.update(mlp_shapes(f"{p}.node_model_cross", latent * (1 + k * len(edge_sets)), latent, latent))
        for name in edge_sets:
            shapes.update(mlp_shapes(f"{p}.edge_models.{name}", 3 * latent, latent, latent))
    return shapes


# ----------------------------------------------------------------------------------------------
# mesh-scale HyperGraphNet / HeteroGraphNet processors (their cluster segments are long)
# ----------------------------------------------------------------------------------------------
HYPER_EDGE_SETS = ("mesh_edges", "intra_cluster_to_cluster", "intra_cluster_to_mesh", "inter_cluster")


def hyper_grid_edges(width: int, height: int, num_clusters: int) -> Dict[str, Tuple[torch.Tensor, torch.Tensor]]:
    """(senders, receivers) of the four edge sets of a ``width x height`` grid mesh clustered into ``num_clusters`` bands of
    consecutive node ids, with the remote sets of ``rmp.hierarchical_connector.connector_indices`` (hyper node j = row n + j)."""
    from .rmp.hierarchical_connector import connector_indices
    n = width * height
    clusters = list(torch.arange(n, dtype=torch.int64).tensor_split(num_clusters))
    sets = connector_indices(clusters, [], n, fully_connect=True)
    return {"mesh_edges": grid_edges_two_way(width, height), **sets}


def hyper_processor_shapes(architecture: str, aggregator: str, num_blocks: int, latent: int = 128) -> Dict[str, Tuple[int, ...]]:
    """Shapes of a 'hyper' or 'hetero' processor over ``HYPER_EDGE_SETS``."""
    k = 4 if aggregator == "pna" else 1
    shapes: Dict[str, Tuple[int, ...]] = {}
    for b in range(num_blocks):
        p = f"processor.graphnet_blocks.{b}"
        for name in HYPER_EDGE_SETS:
            shapes.update(mlp_shapes(f"{p}.edge_models.{name}", 3 * latent, latent, latent))
        if architecture == "hyper":
            for m in ("node_model_cross", "hyper_node_model_up", "hyper_node_model_cross", "node_model_down"):
                shapes.update(mlp_shapes(f"{p}.{m}", latent * (1 + k), latent, latent))
        else:
            for m in ("node_model_cross", "hyper_node_model_cross"):
                shapes.update(mlp_shapes(f"{p}.{m}", latent * (1 + k * len(HYPER_EDGE_SETS)), latent, latent))
    return shapes
