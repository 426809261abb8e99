"""Last stage of encode-process-decode (API mirror of src/migration/decoder.py:9-16).

The decoder MLP has no LayerNorm (meshgraphnet.py:41-43 builds it with ``layer_norm=False``), so it is outside the fused
LayerNorm kernels' contract and runs as stock torch: it touches ``[N, 128] -> [N, output_size]`` once per step, not per layer.

Opt-in: with the encoder and decoder kernels switched on (see ``encoder.py``; ``decoder.kernels`` / ``decoder.precision``
override the process settings) and the precision resolving to 'bf16', it runs on the bf16 tcgen05 decoder kernel
(``ops.decoder_mlp``): bf16 latents in, fp32 ``[N, output_size]`` out (output_size <= 16).
"""
from typing import Callable

import torch
from torch import Tensor, nn

from .. import ops
from .._cabi import HgnError
from ..util import MultiGraph
from .encoder import io_kernels_enabled


def _decoder_parameters(model: nn.Module, like: Tensor):
    """The six tensors of the reference decoder MLP ``LazyMLP([128, 128, n_out])``; lazy linears are materialised by the
    module's own forward on a zero-row input, so the Parameter objects an optimizer already holds stay valid."""
    try:
        linears = [getattr(model.layers, f'linear_{k}') for k in range(3)]
    except AttributeError as err:
        raise HgnError('the decoder kernel needs the reference MLP: LazyMLP(3 linears), no LayerNorm') from err
    if hasattr(model.layers, 'linear_3') or not all(isinstance(lin, nn.Linear) for lin in linears):
        raise HgnError('the decoder kernel needs the reference MLP: LazyMLP(3 linears), no LayerNorm')
    if any(isinstance(lin.weight, nn.parameter.UninitializedParameter) for lin in linears):
        with torch.no_grad():
            model(torch.zeros((0, ops.D_LATENT), dtype=torch.float32, device=like.device))
    return (linears[0].weight, linears[0].bias, linears[1].weight, linears[1].bias, linears[2].weight, linears[2].bias)


class Decoder(nn.Module):
    """Maps the mesh-node latents to the model output.

    ``MeshGraphNet.forward`` hands over a graph whose ``node_features`` field is already the mesh-node latent TENSOR
    (``node_features[0]`` of the processed graph); a one-element list is accepted as well."""

    def __init__(self, make_mlp: Callable, output_size: int):
        super().__init__()
        # state_dict contract: decoder.model.layers.linear_{0,1,2}.{weight,bias} -- no '.0.' level, there is no LayerNorm wrapper
        self.model = make_mlp(output_size)
        self.kernels = None         # None -> hgn_b200.config.io_kernels()
        self.precision = None       # None -> hgn_b200.config.precision()

    def __getstate__(self):
        state = self.__dict__.copy()
        state.pop('_hgn_packed', None)
        return state

    def forward(self, graph: MultiGraph) -> Tensor:
        latents = graph.node_features
        if isinstance(latents, (list, tuple)):
            latents = latents[0]
        if not io_kernels_enabled(self):
            return self.model(latents)
        params = _decoder_parameters(self.model, latents)
        return ops.decoder_mlp(params, self.__dict__.setdefault('_hgn_packed', {}), latents.to(torch.bfloat16))
