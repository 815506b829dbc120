"""FruitField on the B200 kernels: drop-in for ``crop_nerf/fruit_nerf/fruit_field.py:44-302``.

Same constructor signature, same parameter / buffer names (so reference checkpoints' keys line up), same
``get_density`` / ``get_outputs`` / ``get_inference_outputs`` / ``forward`` interface.  ``forward`` is one fused
operator (``ops.fruit_field`` -> ``cnb_field_fwd``/``cnb_field_bwd``); ``get_density`` runs the same operator and
hands its rgb / semantic outputs to the ``get_outputs`` call that follows with the returned embedding, which is how
``FruitField.forward`` and ``FruitModel`` use the pair (fruit_field.py:291-299, fruit_nerf.py:480,503,551).
"""
from __future__ import annotations

from typing import Dict, Optional, Tuple

import torch
from torch import Tensor, nn

from . import _lib as L
from . import ops
from .field_components import MLP, Embedding, FieldHeadNames, HashEncoding, SceneContraction, SemanticFieldHead, SHEncoding
from .rays import RaySamples, ray_layout


class FruitField(nn.Module):
    aabb: Tensor

    def __init__(
        self,
        aabb: Tensor,
        num_images: int,
        num_layers: int = 2,
        hidden_dim: int = 64,
        geo_feat_dim: int = 15,
        num_levels: int = 16,
        base_res: int = 16,
        max_res: int = 2048,
        log2_hashmap_size: int = 19,
        num_layers_color: int = 3,
        num_layers_semantic: int = 2,
        features_per_level: int = 2,
        hidden_dim_color: int = 64,
        hidden_dim_semantics: int = 64,
        hidden_dim_transient: int = 64,
        appearance_embedding_dim: int = 32,
        use_semantics: bool = False,
        test_mode: Optional[str] = None,
        num_semantic_classes: int = 100,
        pass_semantic_gradients: bool = False,
        use_average_appearance_embedding: bool = False,
        spatial_distortion: Optional[nn.Module] = None,
        implementation: str = "b200",
        precision: str = "fp32",
        table_precision: str = "fp32",
    ) -> None:
        super().__init__()
        if not use_semantics or num_semantic_classes != 1:
            raise ValueError("the B200 FruitField is compiled for use_semantics=True, num_semantic_classes=1 (fruit_nerf.py:108-110)")
        self.register_buffer("aabb", aabb)
        self._aabb_host = aabb.detach().cpu().tolist()
        self.geo_feat_dim = geo_feat_dim
        self.register_buffer("max_res", torch.tensor(max_res))
        self.register_buffer("num_levels", torch.tensor(num_levels))
        self.register_buffer("log2_hashmap_size", torch.tensor(log2_hashmap_size))
        self.spatial_distortion = spatial_distortion
        self.num_images = num_images
        self.appearance_embedding_dim = appearance_embedding_dim
        self.embedding_appearance = Embedding(self.num_images, self.appearance_embedding_dim)
        self.use_average_appearance_embedding = use_average_appearance_embedding
        self.use_semantics = use_semantics
        self.test_mode = test_mode
        self.pass_semantic_gradients = pass_semantic_gradients
        self.base_res = base_res
        self.precision = precision
        self.direction_encoding = SHEncoding(levels=4)
        self.mlp_base_grid = HashEncoding(num_levels=num_levels, min_res=base_res, max_res=max_res, log2_hashmap_size=log2_hashmap_size,
                                          features_per_level=features_per_level)
        self.mlp_base_mlp = MLP(in_dim=self.mlp_base_grid.get_out_dim(), num_layers=num_layers, layer_width=hidden_dim,
                                out_dim=1 + self.geo_feat_dim, activation=nn.ReLU(), out_activation=None)
        self.mlp_base = nn.Sequential(self.mlp_base_grid, self.mlp_base_mlp)
        self.mlp_semantics = MLP(in_dim=self.geo_feat_dim, num_layers=num_layers_semantic, layer_width=hidden_dim_semantics,
                                 out_dim=hidden_dim_transient, activation=nn.ReLU(), out_activation=None)
        self.field_head_semantics = SemanticFieldHead(in_dim=self.mlp_semantics.get_out_dim(), num_classes=num_semantic_classes, activation=None)
        self.mlp_head = MLP(in_dim=self.direction_encoding.get_out_dim() + self.geo_feat_dim + self.appearance_embedding_dim,
                            num_layers=num_layers_color, layer_width=hidden_dim_color, out_dim=3, activation=nn.ReLU(), out_activation=nn.Sigmoid())
        self._cache: Optional[tuple] = None
        self._sample_locations: Optional[Tensor] = None
        self._density_before_activation: Optional[Tensor] = None
        self.table_precision = table_precision
        if table_precision not in ("fp32", "fp16"):
            raise ValueError(f"table_precision {table_precision!r}: 'fp32' or 'fp16'")
        if table_precision == "fp16":
            if precision != "mixed":
                raise ValueError("table_precision='fp16' needs precision='mixed': exact fp32 mode evaluates the fp32 table (it is the parity reference)")
            if self._fused_base_architecture():
                raise ValueError("table_precision='fp16' is built for fields wider than the fused base-preset kernels (the fruit_nerf_big / _huge "
                                 "presets): the base preset's 64 MiB table fits the B200's L2, where fp16 rows gather no faster than fp32 rows "
                                 "(DESIGN.md section 7)")
            # the fp16 copy the field forward gathers; the fp32 hash_table stays the parameter (optimiser, gradients, checkpoints)
            self.register_buffer("table_half", torch.zeros(self.mlp_base_grid.hash_table.shape, dtype=torch.float16), persistent=False)
            self._half_stamp: Optional[tuple] = None

    def _fused_base_architecture(self) -> bool:
        """The shapes csrc/field_mixed.cu compiles (cnb_field_mixed_supported): the base preset."""
        dims = lambda m: [m.layers[0].in_features] + [l.out_features for l in m.layers]  # noqa: E731
        return (self.mlp_base_grid.num_levels <= 16 and dims(self.mlp_base_mlp)[1:] == [64, 16] and dims(self.mlp_semantics) == [15, 64, 64]
                and dims(self.mlp_head) == [63, 64, 64, 3] and self.appearance_embedding_dim == 32 and self.geo_feat_dim == 15)

    # ------------------------------------------------------------------------------------------------
    # fp16 tables (table_precision="fp16").  The copy is kept in step by the optimiser (engine.Trainer fuses the refresh into every flat-group
    # update) and refreshed here whenever the table was written any other way: an in-place torch write (load_state_dict,
    # hash_table.copy_ under no_grad) bumps the parameter's version counter, re-homing it changes its storage.  A write through
    # ``hash_table.data`` bumps neither: call refresh_table_copy() after one.
    def _table_stamp(self) -> tuple:
        t = self.mlp_base_grid.hash_table
        return (t._version, t.data_ptr(), t.device, self.table_half.data_ptr())

    def table_copy_stale(self) -> bool:
        return self.table_precision == "fp16" and self._half_stamp != self._table_stamp()

    def refresh_table_copy(self) -> None:
        """Rewrite the fp16 copy from the fp32 hash_table (``__float2half_rn`` of every value)."""
        if self.table_precision != "fp16":
            return
        t = self.mlp_base_grid.hash_table
        if self.table_half.device != t.device:
            self.table_half = self.table_half.to(t.device)
        ops.table_to_half(t.detach(), self.table_half)
        self._half_stamp = self._table_stamp()

    def table_half_current(self) -> Optional[Tensor]:
        """The fp16 copy the field forward gathers (refreshed first when stale), or None for fp32 tables."""
        if self.table_precision != "fp16":
            return None
        if self.table_copy_stale():
            self.refresh_table_copy()
        return self.table_half

    # ------------------------------------------------------------------------------------------------
    def kernel_params(self):
        """Flat parameter list in ``ops.FIELD_PARAM_ORDER``."""
        return [
            self.mlp_base_grid.hash_table,
            *self.mlp_base_mlp.weights(), *self.mlp_base_mlp.biases(),
            *self.mlp_semantics.weights(), *self.mlp_semantics.biases(),
            self.field_head_semantics.net.weight, self.field_head_semantics.net.bias,
            *self.mlp_head.weights(), *self.mlp_head.biases(),
            self.embedding_appearance.embedding.weight,
        ]

    def _appearance_mode(self, inference: bool) -> int:
        # fruit_field.py:251-261 (get_outputs) and :219-221 (get_inference_outputs: always the mean embedding)
        if inference:
            return L.APP_MEAN
        if self.training:
            return L.APP_PER_CAMERA
        return L.APP_MEAN if self.use_average_appearance_embedding else L.APP_ZERO

    def _cfg(self, inference: bool) -> dict:
        if self.spatial_distortion is not None and not isinstance(self.spatial_distortion, SceneContraction):
            raise ValueError("only SceneContraction(order=inf) or None are compiled as spatial distortions")
        g = self.mlp_base_grid
        return {
            "nl_base": len(self.mlp_base_mlp.layers), "nl_sem": len(self.mlp_semantics.layers), "nl_rgb": len(self.mlp_head.layers),
            "num_levels": g.num_levels, "log2_hashmap_size": g.log2_hashmap_size, "scalings": tuple(g._scalings_host),
            "warp": L.make_warp(self.spatial_distortion is not None, self._aabb_host),
            "geo_feat_dim": self.geo_feat_dim,
            "appearance_mode": self._appearance_mode(inference),
            "pass_semantic_gradients": self.pass_semantic_gradients,
            "precision": L.PREC_MIXED if self.precision == "mixed" else L.PREC_FP32,
            "table_half": self.table_half_current(),
            "training": torch.is_grad_enabled(),
            "want_positions": True,
        }

    def _run(self, ray_samples: RaySamples, inference: bool, want_geo: bool = False):
        layout = ray_layout(ray_samples)
        cfg = self._cfg(inference)
        cfg["want_geo"] = want_geo
        if cfg["appearance_mode"] == L.APP_PER_CAMERA and layout[4] is None:
            raise AttributeError("Camera indices are not provided.")
        density, rgb, sem, geo, pos = ops.fruit_field(cfg, layout, self.kernel_params())
        shape = tuple(ray_samples.frustums.shape)
        self._sample_locations = pos.view(*shape, 3) if pos.numel() else None
        out = {
            "density": density.view(*shape, 1),
            "rgb": rgb.view(*shape, 3),
            "semantics": sem.view(*shape, 1),
            "geo": geo.view(*shape, -1) if geo.numel() else None,
        }
        if out["geo"] is not None:
            self._density_before_activation = out["geo"][..., :1]
        return out

    # fruit_field.py:169-194
    def get_density(self, ray_samples: RaySamples) -> Tuple[Tensor, Tensor]:
        # mixed precision: the tensor-core kernel also writes the base MLP's fp32 output row [density before activation | geo15]; the
        # embedding is returned for the caller to hand back to get_outputs (fruit_nerf.py:340,431,480,503; bayesrays/uncertainty.py:109)
        # and carries no gradient of its own there (the heads' gradients flow through the fused operator)
        inference = self.test_mode in ("inference", "export")
        out = self._run(ray_samples, inference, want_geo=True)
        embedding = out["geo"][..., 1:]
        self._cache = (ray_samples, embedding, out, inference)
        return out["density"], embedding

    def _heads_from_cache(self, ray_samples: RaySamples, density_embedding: Tensor, inference: bool) -> Dict:
        c = self._cache
        if c is None or c[0] is not ray_samples or c[1] is not density_embedding or c[3] != inference:
            raise RuntimeError(
                "cropnerf_b200 FruitField.get_outputs expects the (ray_samples, density_embedding) pair returned by the "
                "preceding get_density call -- the field is evaluated as one fused operator"
            )
        self._cache = None
        return {FieldHeadNames.SEMANTICS: c[2]["semantics"], FieldHeadNames.RGB: c[2]["rgb"]}

    # fruit_field.py:235-282
    def get_outputs(self, ray_samples: RaySamples, density_embedding: Optional[Tensor] = None) -> Dict:
        assert density_embedding is not None
        return self._heads_from_cache(ray_samples, density_embedding, False)

    # fruit_field.py:196-233
    def get_inference_outputs(self, ray_samples: RaySamples, density_embedding: Optional[Tensor] = None, render_rgb: bool = False) -> Dict:
        return self._heads_from_cache(ray_samples, density_embedding, True)

    # fruit_field.py:284-302
    def forward(self, ray_samples: RaySamples) -> Dict:
        inference = self.test_mode in ("inference", "export")
        out = self._run(ray_samples, inference)
        return {FieldHeadNames.SEMANTICS: out["semantics"], FieldHeadNames.RGB: out["rgb"], FieldHeadNames.DENSITY: out["density"]}

    def density_fn(self, positions: Tensor, times: Optional[Tensor] = None) -> Tensor:
        from .rays import Frustums

        ray_samples = RaySamples(
            frustums=Frustums(origins=positions, directions=torch.ones_like(positions), starts=torch.zeros_like(positions[..., :1]),
                              ends=torch.zeros_like(positions[..., :1]), pixel_area=torch.ones_like(positions[..., :1])),
            camera_indices=torch.zeros_like(positions[..., :1], dtype=torch.int32),
        )
        return self.forward(ray_samples)[FieldHeadNames.DENSITY]
