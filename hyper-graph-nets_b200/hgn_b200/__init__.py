"""hgn_b200 -- B200 (sm_100a) message-passing processor behind the reference's ``src/migration`` API.

    from hgn_b200.migration.meshgraphnet import MeshGraphNet      # same ctor / state_dict keys
    from hgn_b200.util import EdgeSet, MultiGraph, unsorted_segment_operation

``install_as_reference_modules()`` aliases this package as ``src.migration.*`` / ``src.util`` hot-path
symbols so the reference's own system models (``FlagModel`` ...) run on it unchanged.
"""
from .config import io_kernels, precision, set_io_kernels, set_precision  # noqa: F401


def invalidate_packed_weights() -> None:
    """See ``hgn_b200.ops.invalidate_packed_weights`` (needed only after writes through ``Parameter.data``)."""
    from . import ops
    ops.invalidate_packed_weights()

__version__ = '0.1.0'


def install_as_reference_modules() -> None:
    """Make ``import src.migration.meshgraphnet`` etc. resolve to this package.

    Call before importing the reference's ``src.model`` / ``src.algorithms`` (INTEGRATION.md)."""
    import importlib
    import sys
    import types

    src_pkg = sys.modules.get('src')
    if src_pkg is None:
        try:
            src_pkg = importlib.import_module('src')
        except ImportError:
            src_pkg = types.ModuleType('src')
            src_pkg.__path__ = []
            sys.modules['src'] = src_pkg
    mig = importlib.import_module('hgn_b200.migration')
    sys.modules['src.migration'] = mig
    setattr(src_pkg, 'migration', mig)
    for name in ('graphnet', 'hypergraphnet', 'heterographnet', 'multiscalegraphnet', 'multigraphnet',
                 'repeatedgraphnet', 'processor', 'encoder', 'decoder', 'meshgraphnet', 'normalizer'):
        mod = importlib.import_module(f'hgn_b200.migration.{name}')
        sys.modules[f'src.migration.{name}'] = mod
        setattr(mig, name, mod)
    ours = importlib.import_module('hgn_b200.util')
    ref_util = sys.modules.get('src.util')
    if ref_util is None and getattr(src_pkg, '__path__', None):
        # a reference checkout is importable: keep ITS util module (read_yaml, detach, the namedtuple classes its models and
        # data loader construct) and swap only the hot-path function.  src/util.py:4 imports torch_scatter at module level; an
        # installation without it gets our module instead, which re-exports the same public names.
        try:
            ref_util = importlib.import_module('src.util')
        except ImportError:
            ref_util = None
    if ref_util is not None and ref_util is not ours:
        ref_util.unsorted_segment_operation = ours.unsorted_segment_operation
    else:
        sys.modules['src.util'] = ours
        setattr(src_pkg, 'util', ours)
