"""Process-wide switches that need no change to the reference's config schema."""
import os

_precision = os.environ.get('HGN_B200_PRECISION', 'fp32').lower()


def precision() -> str:
    """'fp32' (parity mode) or 'bf16' (tcgen05 throughput mode)."""
    return _precision


def set_precision(value: str) -> None:
    global _precision
    value = value.lower()
    if value not in ('fp32', 'bf16'):
        raise ValueError("precision must be 'fp32' or 'bf16'")
    _precision = value


_edge_storage = os.environ.get('HGN_EDGE_STORAGE', 'reference').lower()


def edge_storage() -> str:
    """Order in which the bf16 processor keeps its edge rows between entry and exit: 'reference' (as given) or
    'receiver_sorted' (stably sorted by receiver once on entry and restored on exit -- experimental, see plan.EdgeStorageOrder)."""
    return _edge_storage


def set_edge_storage(value: str) -> None:
    global _edge_storage
    value = value.lower()
    if value not in ('reference', 'receiver_sorted'):
        raise ValueError("edge storage must be 'reference' or 'receiver_sorted'")
    _edge_storage = value


_io_kernels = os.environ.get('HGN_B200_IO_KERNELS', '')


def _parse_switch(value) -> bool:
    if isinstance(value, bool):
        return value
    text = str(value).strip().lower()
    if text in ('1', 'true', 'on', 'yes'):
        return True
    if text in ('', '0', 'false', 'off', 'no'):
        return False
    raise ValueError(f"HGN_B200_IO_KERNELS must be one of 1/0, true/false, on/off, yes/no: got {value!r}")


def io_kernels() -> bool:
    """Whether the encoder and decoder MLPs run on the bf16 tcgen05 kernels (off by default).  It takes effect only where the
    precision resolves to 'bf16'; the fp32 parity mode always keeps the torch MLPs."""
    return _parse_switch(_io_kernels)


def set_io_kernels(value: bool) -> None:
    global _io_kernels
    _io_kernels = _parse_switch(value)
