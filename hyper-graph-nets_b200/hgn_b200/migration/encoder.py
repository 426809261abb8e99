"""Mirror of src/migration/encoder.py.  Runs once per step on stock torch ``Linear``/``LayerNorm``
(out of the per-layer hot path, SURVEY.md s2); same attribute names and ``state_dict`` keys.

Opt-in: with the encoder and decoder kernels switched on (``hgn_b200.set_io_kernels(True)``, ``HGN_B200_IO_KERNELS=1``
or ``encoder.kernels = True``) and the precision resolving to 'bf16', every MLP runs on the bf16 tcgen05 encoder
kernel (``ops.encoder_mlp``): raw fp32 features in, bf16 latents out, which ``Processor.forward`` then takes as they
are.  ``kernels`` / ``precision`` = None follow the process settings; the fp32 parity mode always keeps the torch MLPs.
"""
from typing import Callable, List

from torch import nn

from .. import config, ops, util
from .._cabi import HgnError
from ..util import MultiGraph
from .graphnet import _mlp_parameters


def io_kernels_enabled(module: nn.Module) -> bool:
    """Whether ``module`` (an ``Encoder`` or ``Decoder``) runs its MLPs on the bf16 encoder / decoder kernels."""
    kernels = getattr(module, 'kernels', None)
    precision = getattr(module, 'precision', None) or config.precision()
    if precision not in ('fp32', 'bf16'):
        raise ValueError(f"unknown precision {precision!r} (expected 'fp32' or 'bf16')")
    return precision == 'bf16' and (config.io_kernels() if kernels is None else bool(kernels))


class Encoder(nn.Module):
    """Encodes node and edge features into latent features."""

    def __init__(self, make_mlp: Callable, latent_size: int, edge_sets: List[str], hierarchical=True):
        super().__init__()
        self._make_mlp = make_mlp
        self._latent_size = latent_size
        self.node_model = self._make_mlp(latent_size)
        self.edge_models = nn.ModuleDict({name: self._make_mlp(latent_size) for name in edge_sets})
        self.hierarchical = hierarchical
        if hierarchical:
            self.hyper_node_model = self._make_mlp(latent_size)
        self.kernels = None         # None -> hgn_b200.config.io_kernels()
        self.precision = None       # None -> hgn_b200.config.precision()

    def __getstate__(self):
        state = self.__dict__.copy()
        state.pop('_hgn_packed', None)
        return state

    def forward(self, graph: MultiGraph) -> MultiGraph:
        encode = self._encode if io_kernels_enabled(self) else (lambda name, model, x: model(x))
        nodes = [encode('node_model', self.node_model, graph.node_features[0])]
        # a second node list (hyper nodes) goes through its own MLP only for hierarchical
        # architectures (encoder.py:26-35); a missing second entry is tolerated silently
        if isinstance(graph.node_features, (list, tuple)) and len(graph.node_features) > 1:
            name = 'hyper_node_model' if self.hierarchical else 'node_model'
            nodes.append(encode(name, getattr(self, name), graph.node_features[1]))
        # edge sets without an encoder model are dropped (encoder.py:41-45)
        edge_sets = [es._replace(features=encode(f'edge_models.{es.name}', self.edge_models[es.name], es.features))
                     for es in graph.edge_sets if es.name in self.edge_models]
        return MultiGraph(nodes, edge_sets)

    def _encode(self, name: str, model: nn.Module, features):
        x = features.to(util.device)
        if x.dim() != 2 or not 1 <= x.shape[1] <= ops.D_LATENT:
            raise HgnError(f"encoder kernel: {name} takes [rows, K] features with 1 <= K <= {ops.D_LATENT}, got {tuple(x.shape)}")
        params = _mlp_parameters(model, x.shape[1], x)
        cache = self.__dict__.setdefault('_hgn_packed', {}).setdefault(name, {})
        return ops.encoder_mlp(params, cache, x)
