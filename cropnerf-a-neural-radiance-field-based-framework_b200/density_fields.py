"""Proposal-network density field (row a7): drop-in for ``nerfstudio/fields/density_fields.py HashMLPDensityField``
as the reference builds it at ``fruit_nerf.py:118-142`` -- same constructor kwargs, same parameter names
(``mlp_base.0.hash_table``, ``mlp_base.1.layers.*``), same ``get_density`` / ``density_fn`` interface, one fused
CUDA kernel (``csrc/density_field.cu``) underneath.
"""
from __future__ import annotations

from typing import Optional, Tuple

import torch
from torch import Tensor, nn

from . import _lib as L
from . import ops
from .field_components import MLP, HashEncoding, SceneContraction
from .rays import Frustums, RaySamples, ray_layout


class HashMLPDensityField(nn.Module):
    def __init__(self, aabb: Tensor, num_layers: int = 2, hidden_dim: int = 64, spatial_distortion: Optional[nn.Module] = None,
                 use_linear: bool = False, num_levels: int = 8, max_res: int = 1024, base_res: int = 16, log2_hashmap_size: int = 18,
                 features_per_level: int = 2, average_init_density: float = 1.0, implementation: str = "b200",
                 precision: str = "fp32") -> None:
        super().__init__()
        self.precision = precision  # "mixed": bf16 operands in the backward's MLP parameter-gradient contraction (k_density_bwd_tc<0>)
        self.register_buffer("aabb", aabb)
        self._aabb_host = aabb.detach().cpu().tolist()
        self.spatial_distortion = spatial_distortion
        self.use_linear = use_linear
        self.average_init_density = average_init_density
        self.register_buffer("max_res", torch.tensor(max_res))
        self.register_buffer("num_levels", torch.tensor(num_levels))
        self.register_buffer("log2_hashmap_size", torch.tensor(log2_hashmap_size))
        self.encoding = HashEncoding(num_levels=num_levels, min_res=base_res, max_res=max_res, log2_hashmap_size=log2_hashmap_size,
                                     features_per_level=features_per_level)
        if not use_linear:
            if num_layers != 2:
                raise ValueError("the fused proposal kernel is compiled for num_layers=2 (nerfstudio default, fruit_nerf.py:123-139)")
            if hidden_dim not in (16, 32, 64):
                raise ValueError(f"the fused proposal kernel is compiled for hidden_dim 16, 32 or 64 (got {hidden_dim})")
            network = MLP(in_dim=self.encoding.get_out_dim(), num_layers=num_layers, layer_width=hidden_dim, out_dim=1,
                          activation=nn.ReLU(), out_activation=None)
            self.mlp_base = nn.Sequential(self.encoding, network)
        else:
            self.linear = nn.Linear(self.encoding.get_out_dim(), 1)

    def _warp(self) -> L.Warp:
        if self.spatial_distortion is not None and not isinstance(self.spatial_distortion, SceneContraction):
            raise ValueError("only SceneContraction(order=inf) or None are compiled as spatial distortions")
        return L.make_warp(self.spatial_distortion is not None, self._aabb_host)

    def density_from_layout(self, layout, want_positions: bool = False):
        origins, directions, starts, ends, _cam, R, S, row_stride = layout
        if self.use_linear:
            raise NotImplementedError("use_linear proposal fields: compose HashEncoding + Linear (not on the fruit_nerf presets)")
        net = self.mlp_base[1]
        cfg = ((origins, directions, starts, ends, R, S, row_stride), self.encoding.grid_cfg(), self._warp(), float(self.average_init_density), want_positions,
               L.PREC_MIXED if self.precision == "mixed" else L.PREC_FP32)
        return ops.density_field(cfg, self.encoding.hash_table, net.layers[0].weight, net.layers[0].bias, net.layers[1].weight, net.layers[1].bias)

    def get_density(self, ray_samples: RaySamples) -> Tuple[Tensor, None]:
        layout = ray_layout(ray_samples)
        density = self.density_from_layout(layout)
        return density.view(*ray_samples.frustums.shape, 1), None

    def density_fn(self, positions: Tensor, times: Optional[Tensor] = None) -> Tensor:
        """``Field.density_fn`` (nerfstudio base_field.py): one zero-length frustum per point."""
        del times
        ray_samples = RaySamples(
            frustums=Frustums(
                origins=positions,
                directions=torch.ones_like(positions),
                starts=torch.zeros_like(positions[..., :1]),
                ends=torch.zeros_like(positions[..., :1]),
                pixel_area=torch.ones_like(positions[..., :1]),
            )
        )
        density, _ = self.get_density(ray_samples)
        return density

    def forward(self, ray_samples: RaySamples):
        density, _ = self.get_density(ray_samples)
        return {"density": density}
