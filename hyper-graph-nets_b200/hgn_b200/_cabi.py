"""ctypes binding of ``libhgn_b200.so`` (declared in ``include/hgn_b200.h``).

There is deliberately no fallback: if the shared library is missing or no sm_100 device is present the
first kernel call raises.  ``load()`` itself only needs the file (so the export check runs on CPU).
"""
from __future__ import annotations

import ctypes
import os
from ctypes import c_char_p, c_int, c_int32, c_int64, c_size_t, c_void_p, POINTER

HGN_OK = 0
HGN_F32 = 0
HGN_BF16 = 1
AGG_SUM, AGG_MEAN, AGG_MAX, AGG_MIN = 1, 2, 4, 8
HGN_MAX_CHUNKS = 24
HGN_SEGMENT_PARTIAL_WIDTH = 388
HGN_IO_ENCODER, HGN_IO_DECODER = 0, 1
ABI_VERSION = 6            # HGN_B200_ABI_VERSION of include/hgn_b200.h these signatures were written against

LIB_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "libhgn_b200.so")


class Chunks(ctypes.Structure):
    """``hgn_chunks`` (include/hgn_b200.h)."""
    _fields_ = [
        ("n_chunks", c_int32),
        ("src", c_void_p * HGN_MAX_CHUNKS),
        ("idx", c_void_p * HGN_MAX_CHUNKS),
        ("row_offset", c_int64 * HGN_MAX_CHUNKS),
    ]


class SegmentSplit(ctypes.Structure):
    """``hgn_segment_split`` (include/hgn_b200.h)."""
    _fields_ = [("num_segments", c_int64), ("num_elements", c_int64), ("n_long", c_int64), ("n_pieces", c_int64), ("n_short", c_int64),
                ("long_ids", c_void_p), ("piece_ptr", c_void_p), ("pieces", c_void_p), ("perm_short", c_void_p), ("rowptr_short", c_void_p)]


HGN_MAX_PEERS = 16


class HaloPeers(ctypes.Structure):
    """``hgn_halo_peers`` (include/hgn_b200.h)."""
    _fields_ = [("dst", c_void_p * HGN_MAX_PEERS), ("flag", c_void_p * HGN_MAX_PEERS), ("row_begin", c_int64 * (HGN_MAX_PEERS + 1))]


class HaloFlags(ctypes.Structure):
    """``hgn_halo_flags`` (include/hgn_b200.h)."""
    _fields_ = [("flag", c_void_p * HGN_MAX_PEERS)]


# name -> (restype, argtypes); every symbol the header declares
SIGNATURES = {
    "hgn_abi_version": (c_int, []),
    "hgn_last_error": (c_char_p, []),
    "hgn_device_supported": (c_int, []),
    "hgn_csr_workspace_bytes": (c_size_t, [c_int64, c_int64]),
    "hgn_csr_build": (c_int, [c_void_p, c_int64, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "hgn_segment_reduce": (c_int, [c_int, c_void_p, c_int64, c_int32, c_void_p, c_void_p, c_int64,
                                   c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p]),
    "hgn_segment_sum_pair": (c_int, [c_int, c_void_p, c_int64, c_int32, c_void_p, c_void_p, c_int64, c_void_p,
                                      c_void_p, c_void_p, c_int64, c_void_p, c_void_p]),
    "hgn_segment_reduce_bwd": (c_int, [c_int, c_int64, c_int32, c_void_p, c_void_p, c_void_p, c_int64,
                                       c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p]),
    "hgn_segment_layer_grad": (c_int, [c_int, c_int64, c_int32, c_void_p, c_void_p, c_int64] + [c_void_p] * 9 + [c_void_p]),
    "hgn_segment_split_threshold": (c_int32, []),
    "hgn_segment_split_piece": (c_int32, []),
    "hgn_segment_split_build_workspace_bytes": (c_size_t, [c_int64, c_int64]),
    "hgn_segment_split_max_long": (c_int64, [c_int64, c_int64]),
    "hgn_segment_split_max_pieces": (c_int64, [c_int64]),
    "hgn_segment_split_build": (c_int, [c_void_p, c_void_p, c_int64, c_int64] + [c_void_p] * 5 + [POINTER(c_int64), c_void_p, c_size_t, c_void_p]),
    "hgn_segment_split_reduce_workspace_bytes": (c_size_t, [POINTER(SegmentSplit)]),
    "hgn_segment_reduce_split": (c_int, [c_int, c_void_p, c_int64, c_int32, c_void_p, c_void_p, c_int64, POINTER(SegmentSplit)]
                                 + [c_void_p] * 6 + [c_int, c_void_p, c_size_t, c_void_p]),
    "hgn_segment_sum_pair_split": (c_int, [c_int, c_void_p, c_int64, c_int32, c_void_p, c_void_p, c_int64, POINTER(SegmentSplit), c_void_p,
                                           c_void_p, c_void_p, c_int64, POINTER(SegmentSplit), c_void_p, c_void_p, c_size_t, c_void_p]),
    "hgn_segment_reduce_bwd_split": (c_int, [c_int, c_int64, c_int32, c_void_p, c_void_p, c_void_p, c_int64, POINTER(SegmentSplit)]
                                     + [c_void_p] * 7 + [c_void_p]),
    "hgn_segment_layer_grad_split": (c_int, [c_int, c_int64, c_int32, c_void_p, c_void_p, c_int64, POINTER(SegmentSplit)]
                                     + [c_void_p] * 9 + [c_void_p]),
    "hgn_segment_partials": (c_int, [c_int, c_void_p, c_int64, c_int32, c_void_p, c_void_p, c_int64, POINTER(SegmentSplit), c_int]
                             + [c_void_p] * 4 + [c_size_t, c_void_p]),
    "hgn_multi_segment_sum": (c_int, [c_int, c_void_p, c_int64, c_int32, c_void_p, c_void_p, c_void_p]),
    "hgn_mlp_packed_bytes": (c_size_t, [c_int, c_int32]),
    "hgn_mlp_pack": (c_int, [c_int, c_int32] + [c_void_p] * 8 + [c_void_p, c_void_p]),
    "hgn_mlp_forward": (c_int, [c_int, c_int64, POINTER(Chunks), c_void_p, c_void_p, c_int64, c_void_p, c_void_p]),
    "hgn_mlp_backward_workspace_bytes": (c_size_t, [c_int, c_int64, c_int32]),
    "hgn_mlp_backward": (c_int, [c_int, c_int64, POINTER(Chunks), c_void_p, c_void_p, c_int32, POINTER(c_void_p)]
                         + [c_void_p] * 8 + [c_void_p, c_size_t, c_void_p]),
    "hgn_io_mlp_packed_bytes": (c_size_t, []),
    "hgn_io_mlp_pack": (c_int, [c_int32, c_int32] + [c_void_p] * 8 + [c_void_p, c_void_p]),
    "hgn_encoder_forward": (c_int, [c_int64, c_int32, c_void_p, c_void_p, c_void_p, c_void_p]),
    "hgn_encoder_backward_workspace_bytes": (c_size_t, [c_int64, c_int32]),
    "hgn_encoder_backward": (c_int, [c_int64, c_int32] + [c_void_p] * 12 + [c_void_p, c_size_t, c_void_p]),
    "hgn_decoder_forward": (c_int, [c_int64, c_int32, c_void_p, c_void_p, c_void_p, c_void_p]),
    "hgn_decoder_backward_workspace_bytes": (c_size_t, [c_int64, c_int32]),
    "hgn_decoder_backward": (c_int, [c_int64, c_int32] + [c_void_p] * 10 + [c_void_p, c_size_t, c_void_p]),
    "hgn_edge_project_forward": (c_int, [c_int, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "hgn_edge_project_backward_workspace_bytes": (c_size_t, [c_int, c_int64]),
    "hgn_edge_project_backward": (c_int, [c_int, c_int64] + [c_void_p] * 7 + [c_void_p, c_size_t, c_void_p]),
    "hgn_edge_update_forward": (c_int, [c_int, c_int64] + [c_void_p] * 7 + [c_void_p]),
    "hgn_edge_update_backward_workspace_bytes": (c_size_t, [c_int, c_int64]),
    "hgn_edge_update_backward": (c_int, [c_int, c_int64] + [c_void_p] * 18 + [c_void_p, c_size_t, c_void_p]),
    "hgn_node_update_forward": (c_int, [c_int, c_int64, c_void_p, c_int32, POINTER(c_void_p)] + [c_void_p] * 4 + [c_void_p]),
    "hgn_node_update_backward_workspace_bytes": (c_size_t, [c_int, c_int64]),
    "hgn_node_update_backward": (c_int, [c_int, c_int64, c_void_p, c_int32, POINTER(c_void_p)] + [c_void_p] * 5 + [POINTER(c_void_p)] + [c_void_p] * 8 + [c_void_p, c_size_t, c_void_p]),
    "hgn_rows_gather": (c_int, [c_int, c_void_p, c_void_p, c_int64, c_int32, c_void_p, c_void_p]),
    "hgn_rows_scatter": (c_int, [c_int, c_void_p, c_void_p, c_int64, c_int32, c_void_p, c_int, c_void_p]),
    "hgn_peer_alloc": (c_int, [c_size_t, POINTER(c_void_p), c_char_p]),
    "hgn_peer_open": (c_int, [c_char_p, POINTER(c_void_p)]),
    "hgn_peer_close": (c_int, [c_void_p]),
    "hgn_peer_free": (c_int, [c_void_p]),
    "hgn_halo_push": (c_int, [c_int, c_void_p, c_void_p, c_int32, c_void_p, c_int32, ctypes.c_uint32, c_void_p, c_void_p]),
    "hgn_halo_wait": (c_int, [c_void_p, c_int32, ctypes.c_uint32, c_void_p]),
    "hgn_cluster_combine": (c_int, [c_void_p, c_int32, c_int32, c_int64] + [c_void_p] * 7 + [c_void_p]),
    "hgn_cluster_grad_sum": (c_int, [c_int, c_void_p, c_int32, c_int64, c_int32, c_void_p, c_void_p]),
    "hgn_cluster_mean_grad": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_void_p]),
    "hgn_colsum": (c_int, [c_int, c_void_p, c_int64, c_int32, c_void_p, c_void_p, c_size_t, c_void_p]),
    "hgn_colsum_workspace_bytes": (c_size_t, [c_int64, c_int32]),
    "hgn_world_edges_workspace_bytes": (c_size_t, [c_int64, c_int64]),
    "hgn_world_edges_count": (c_int, [c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_int64, ctypes.c_float, c_int32, c_int32,
                                      c_void_p, c_size_t, POINTER(c_int64), c_void_p]),
    "hgn_world_edges_emit": (c_int, [c_void_p, c_void_p, c_int64, c_int64, ctypes.c_float, c_int32, c_void_p, c_size_t,
                                     c_void_p, c_void_p, c_int64, c_void_p]),
    "hgn_profile_enable": (c_int, [c_int]),
    "hgn_profile_reset": (c_int, []),
    "hgn_profile_report": (c_size_t, [c_char_p, c_size_t]),
    "hgn_copy_h2d": (c_int, [c_void_p, c_void_p, c_size_t, c_void_p]),
    "hgn_copy_d2h": (c_int, [c_void_p, c_void_p, c_size_t, c_void_p]),
}

_lib = None


class HgnError(RuntimeError):
    pass


def load() -> ctypes.CDLL:
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise HgnError(
                f"{LIB_PATH} not found: build it with hyper-graph-nets_b200/build.sh (or __graft_entry__.build()). "
                "hgn_b200 has no CPU / PyTorch fallback.")
        lib = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)   # AttributeError here = header and library out of sync
            fn.restype = res
            fn.argtypes = args
        if lib.hgn_abi_version() != ABI_VERSION:
            raise HgnError(f"libhgn_b200.so ABI version {lib.hgn_abi_version()} != {ABI_VERSION} expected by these bindings: rebuild")
        _lib = lib
    return _lib


def check(rc: int, what: str = "") -> None:
    if rc != HGN_OK:
        msg = load().hgn_last_error().decode(errors="replace")
        raise HgnError(f"{what or 'hgn_b200'} failed ({rc}): {msg}")


def dtype_code(torch_dtype) -> int:
    import torch
    if torch_dtype == torch.float32:
        return HGN_F32
    if torch_dtype == torch.bfloat16:
        return HGN_BF16
    raise HgnError(f"unsupported feature dtype {torch_dtype}: the kernels take float32 or bfloat16 rows")


def ptr(t) -> int:
    """Device pointer of a contiguous tensor (None -> NULL)."""
    if t is None:
        return None
    return t.data_ptr()


def stream_ptr() -> int:
    import torch
    return torch.cuda.current_stream().cuda_stream


def require_cuda(*tensors) -> None:
    import torch
    if not torch.cuda.is_available():
        raise HgnError("hgn_b200 needs a CUDA (sm_100a) device: there is no CPU fallback")
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise HgnError("hgn_b200 kernels take CUDA tensors")


def profile(enable: bool) -> None:
    """Switch the library's per-kernel CUDA-event timing on/off (clears earlier records when enabling)."""
    lib = load()
    if enable:
        lib.hgn_profile_reset()
    lib.hgn_profile_enable(1 if enable else 0)


def profile_report():
    """[{'name', 'launches', 'ms'}] since the last ``profile(True)`` (synchronises the device)."""
    import json
    lib = load()
    n = lib.hgn_profile_report(None, 0)
    buf = ctypes.create_string_buffer(n + 16)
    lib.hgn_profile_report(buf, n + 16)
    return json.loads(buf.value.decode())
