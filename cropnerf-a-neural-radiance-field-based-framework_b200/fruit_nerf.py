"""FruitModel on the B200 kernels: drop-in for the ray-render path of ``crop_nerf/fruit_nerf/fruit_nerf.py:71-645``.

Same module attribute names (``field``, ``proposal_networks``, ``proposal_sampler``, ``renderer_*``), same method
names and output dictionaries, same param groups (``proposal_networks`` / ``fields`` / ``camera_opt``,
fruit_nerf.py:191-196).  Out of scope here (SURVEY.md section 2): image metrics (``get_image_metrics_and_images``),
the broken ``get_projection_outputs``, and the camera-optimizer *gradient* (pose deltas are applied in the forward,
but the kernels do not return dL/d(origin, direction) yet -- a "next" row).
"""
from __future__ import annotations

from collections import defaultdict
from dataclasses import dataclass, field
from typing import Callable, Dict, List, Optional, Tuple, Union

import numpy as np
import torch
from torch import Tensor, nn
from torch.nn import Parameter

from . import _lib as L
from . import ops
from .density_fields import HashMLPDensityField
from .field_components import FieldHeadNames, SceneContraction
from .fruit_field import FruitField
from .ray_samplers import ProposalNetworkSampler, UniformSampler, UniformSamplerWithNoise
from .rays import RayBundle
from .renderers import (AccumulationRenderer, DepthRenderer, PixelLosses, RGBRenderer, SemanticRenderer, distortion_loss,
                        interlevel_loss, resolve_background)


@dataclass
class FruitNerfModelConfig:
    """``FruitNerfModelConfig(NerfactoModelConfig)`` (fruit_nerf.py:59-68) with the inherited nerfacto fields that
    reach the ray-render path, same names and defaults (SURVEY.md section 8 preamble)."""

    near_plane: float = 0.05
    far_plane: float = 1000.0
    background_color: str = "last_sample"
    hidden_dim: int = 64            # not forwarded to FruitField by the reference (fruit_nerf.py:97-112)
    hidden_dim_color: int = 64      # idem
    num_levels: int = 16
    base_res: int = 16              # idem
    max_res: int = 2048
    log2_hashmap_size: int = 19
    features_per_level: int = 2     # idem
    num_proposal_samples_per_ray: Tuple[int, ...] = (256, 96)
    num_nerf_samples_per_ray: int = 48
    proposal_update_every: int = 5
    proposal_warmup: int = 5000
    num_proposal_iterations: int = 2
    use_same_proposal_network: bool = False
    proposal_net_args_list: List[Dict] = field(
        default_factory=lambda: [
            {"hidden_dim": 16, "log2_hashmap_size": 17, "num_levels": 5, "max_res": 128, "use_linear": False},
            {"hidden_dim": 16, "log2_hashmap_size": 17, "num_levels": 5, "max_res": 256, "use_linear": False},
        ]
    )
    proposal_initial_sampler: str = "piecewise"
    interlevel_loss_mult: float = 1.0
    use_proposal_weight_anneal: bool = True
    use_average_appearance_embedding: bool = True
    proposal_weights_anneal_slope: float = 10.0
    proposal_weights_anneal_max_num_iters: int = 1000
    use_single_jitter: bool = True
    disable_scene_contraction: bool = False
    use_gradient_scaling: bool = False
    predict_normals: bool = False
    eval_num_rays_per_chunk: int = 1 << 15
    appearance_embed_dim: int = 32  # idem (not forwarded)
    camera_optimizer_mode: str = "off"
    # FruitNerfModelConfig additions
    semantic_loss_weight: float = 1.0
    pass_semantic_gradients: bool = False
    num_layers_semantic: int = 2
    hidden_dim_semantics: int = 64
    geo_feat_dim: int = 15
    # B200 selector: "fp32" (exact, 1e-4 parity) or "mixed" (fp16 tensor-core MLPs, 2e-3 parity)
    precision: str = "fp32"
    # hash-table storage the field forward gathers: "fp32", or "fp16" (a copy the optimiser keeps in step with the fp32 master table; only with
    # precision="mixed" on fields wider than the fused base-preset kernels, i.e. the big / huge presets -- FruitField raises otherwise)
    table_precision: str = "fp32"

    def setup(self, **kwargs) -> "FruitModel":
        return FruitModel(self, **kwargs)


@dataclass
class TrainingCallback:
    where_to_run: List[str]
    func: Callable
    update_every_num_iters: int = 1


class NearFarCollider(nn.Module):
    """nerfstudio scene_colliders.py NearFarCollider (fruit_nerf.py:167): pass-through when nears/fars are already set
    (lets ``get_outputs_for_projections`` inject AABB near/far, fruit_nerf.py:283,307-308)."""

    def __init__(self, near_plane: float, far_plane: float, reset_near_plane: bool = True) -> None:
        super().__init__()
        self.near_plane = near_plane
        self.far_plane = far_plane
        self.reset_near_plane = reset_near_plane

    def forward(self, ray_bundle: RayBundle) -> RayBundle:
        if ray_bundle.nears is not None and ray_bundle.fars is not None:
            return ray_bundle
        R = ray_bundle.origins.shape[0]
        near = self.near_plane if (self.training or not self.reset_near_plane) else 0.0
        ray_bundle.nears = torch.full((R, 1), float(near), device=ray_bundle.origins.device, dtype=torch.float32)
        ray_bundle.fars = torch.full((R, 1), float(self.far_plane), device=ray_bundle.origins.device, dtype=torch.float32)
        return ray_bundle


def exp_map_SO3xR3(tangent_vector: Tensor) -> Tensor:
    """nerfstudio/cameras/lie_groups.py exp_map_SO3xR3: [N,6] (translation, axis-angle) -> [N,3,4] [R|t] (Rodrigues with
    the small-angle clamp nerfstudio uses)."""
    log_rot = tangent_vector[:, 3:]
    nrms = (log_rot * log_rot).sum(1)
    rot_angles = torch.clamp(nrms, 1e-4).sqrt()
    rot_angles_inv = 1.0 / rot_angles
    fac1 = rot_angles_inv * rot_angles.sin()
    fac2 = rot_angles_inv * rot_angles_inv * (1.0 - rot_angles.cos())
    skews = torch.zeros((log_rot.shape[0], 3, 3), dtype=log_rot.dtype, device=log_rot.device)
    skews[:, 0, 1] = -log_rot[:, 2]
    skews[:, 0, 2] = log_rot[:, 1]
    skews[:, 1, 0] = log_rot[:, 2]
    skews[:, 1, 2] = -log_rot[:, 0]
    skews[:, 2, 0] = -log_rot[:, 1]
    skews[:, 2, 1] = log_rot[:, 0]
    skews_square = torch.bmm(skews, skews)
    ret = torch.zeros(tangent_vector.shape[0], 3, 4, dtype=tangent_vector.dtype, device=tangent_vector.device)
    ret[:, :3, :3] = fac1[:, None, None] * skews + fac2[:, None, None] * skews_square + torch.eye(3, dtype=log_rot.dtype, device=log_rot.device)[None]
    ret[:, :3, 3] = tangent_vector[:, :3]
    return ret


class CameraOptimizer(nn.Module):
    """nerfstudio/cameras/camera_optimizers.py CameraOptimizer as FruitModel uses it (fruit_nerf.py:114-116,547,614):
    mode "off" = identity; "SO3xR3" = per-camera pose deltas applied to the ray origins / directions in the forward pass and
    trained through the ray gradients the kernels return (row a17).  The pose algebra itself is a handful of [R,6] torch
    ops; the per-sample work (hash-grid input gradient, contraction Jacobian, per-ray reduction) is in the CUDA path."""

    def __init__(self, num_cameras: int, mode: str = "off", trans_l2_penalty: float = 1e-2, rot_l2_penalty: float = 1e-3) -> None:
        super().__init__()
        if mode not in ("off", "SO3xR3"):
            raise ValueError(f"camera optimizer mode {mode!r} not compiled (off / SO3xR3)")
        self.mode = mode
        self.num_cameras = num_cameras
        self.trans_l2_penalty = trans_l2_penalty
        self.rot_l2_penalty = rot_l2_penalty
        if mode != "off":
            self.pose_adjustment = Parameter(torch.zeros((num_cameras, 6)))

    def forward(self, indices: Tensor) -> Tensor:
        return exp_map_SO3xR3(self.pose_adjustment[indices.long(), :])

    def apply_to_raybundle(self, ray_bundle: RayBundle) -> None:
        if self.mode == "off":
            return
        correction = self(ray_bundle.camera_indices.squeeze(-1))
        ray_bundle.origins = ray_bundle.origins + correction[:, :3, 3]
        ray_bundle.directions = torch.bmm(correction[:, :3, :3], ray_bundle.directions[..., None]).squeeze(-1)

    def get_loss_dict(self, loss_dict: dict) -> None:
        if self.mode != "off":
            loss_dict["camera_opt_regularizer"] = (self.pose_adjustment[:, :3].norm(dim=-1).mean() * self.trans_l2_penalty
                                                   + self.pose_adjustment[:, 3:].norm(dim=-1).mean() * self.rot_l2_penalty)

    def get_metrics_dict(self, metrics_dict: dict) -> None:
        if self.mode != "off":
            metrics_dict["camera_opt_translation"] = self.pose_adjustment[:, :3].detach().norm()
            metrics_dict["camera_opt_rotation"] = self.pose_adjustment[:, 3:].detach().norm()

    def get_param_groups(self, param_groups: dict) -> None:
        params = list(self.parameters())
        if params:
            param_groups["camera_opt"] = params


@dataclass
class CameraOptimizerConfig:
    """nerfstudio ``CameraOptimizerConfig`` as FruitModel uses it (``self.config.camera_optimizer.setup(num_cameras=, device=)``,
    fruit_nerf.py:114-116)."""

    mode: str = "off"
    trans_l2_penalty: float = 1e-2
    rot_l2_penalty: float = 1e-3

    def setup(self, num_cameras: int, device=None, **kwargs) -> "CameraOptimizer":
        opt = CameraOptimizer(num_cameras, self.mode, self.trans_l2_penalty, self.rot_l2_penalty)
        opt.config = self
        return opt


class FruitModel(nn.Module):
    config: FruitNerfModelConfig

    def __init__(self, config: FruitNerfModelConfig, scene_box=None, num_train_data: int = 1, metadata: Optional[Dict] = None,
                 test_mode: str = "val", device: Union[str, torch.device, None] = None, **kwargs) -> None:
        super().__init__()
        self.config = config
        self.test_mode = test_mode
        self.num_train_data = num_train_data
        self.kwargs = kwargs
        aabb = getattr(scene_box, "aabb", scene_box)
        self.aabb = aabb if aabb is not None else torch.tensor([[-1.0, -1.0, -1.0], [1.0, 1.0, 1.0]])
        semantics = (metadata or {}).get("semantics")
        colors = getattr(semantics, "colors", None)
        self.register_buffer("colormap", torch.as_tensor(colors, dtype=torch.float32).clone() if colors is not None else torch.tensor([0.0, 1.0]))
        self.step = 0
        self.fused_render = True       # one-call render path for no-grad eval (set False to force the per-module operators)
        self._fused_pipeline = None
        self._pinned: Dict[tuple, Tensor] = {}
        self.populate_modules()
        if device is not None:
            self.to(device)

    @property
    def device(self) -> torch.device:
        return self.colormap.device

    # fruit_nerf.py:87-183
    def populate_modules(self) -> None:
        cfg = self.config
        scene_contraction = None if cfg.disable_scene_contraction else SceneContraction(order=float("inf"))
        self.field = FruitField(
            self.aabb,
            num_levels=cfg.num_levels,
            max_res=cfg.max_res,
            num_layers_semantic=cfg.num_layers_semantic,
            hidden_dim_semantics=cfg.hidden_dim_semantics,
            log2_hashmap_size=cfg.log2_hashmap_size,
            spatial_distortion=scene_contraction,
            num_images=self.num_train_data,
            geo_feat_dim=cfg.geo_feat_dim,
            use_average_appearance_embedding=cfg.use_average_appearance_embedding,
            use_semantics=True,
            test_mode=self.test_mode,
            num_semantic_classes=1,
            pass_semantic_gradients=cfg.pass_semantic_gradients,
            precision=cfg.precision,
            table_precision=cfg.table_precision,
        )
        self.camera_optimizer = CameraOptimizer(self.num_train_data, cfg.camera_optimizer_mode)
        self.density_fns: List[Callable] = []
        num_prop_nets = cfg.num_proposal_iterations
        self.proposal_networks = nn.ModuleList()
        if cfg.use_same_proposal_network:
            assert len(cfg.proposal_net_args_list) == 1, "Only one proposal network is allowed."
            network = HashMLPDensityField(self.aabb, spatial_distortion=scene_contraction, precision=cfg.precision, **cfg.proposal_net_args_list[0])
            self.proposal_networks.append(network)
            self.density_fns.extend([network.density_fn for _ in range(num_prop_nets)])
        else:
            for i in range(num_prop_nets):
                args = cfg.proposal_net_args_list[min(i, len(cfg.proposal_net_args_list) - 1)]
                self.proposal_networks.append(HashMLPDensityField(self.aabb, spatial_distortion=scene_contraction, precision=cfg.precision, **args))
            self.density_fns.extend([network.density_fn for network in self.proposal_networks])

        def update_schedule(step):
            return np.clip(np.interp(step, [0, cfg.proposal_warmup], [0, cfg.proposal_update_every]), 1, cfg.proposal_update_every)

        initial_sampler = None
        if cfg.proposal_initial_sampler == "uniform":
            initial_sampler = UniformSampler(single_jitter=cfg.use_single_jitter)
        self.proposal_sampler = ProposalNetworkSampler(
            num_nerf_samples_per_ray=cfg.num_nerf_samples_per_ray,
            num_proposal_samples_per_ray=cfg.num_proposal_samples_per_ray,
            num_proposal_network_iterations=cfg.num_proposal_iterations,
            single_jitter=cfg.use_single_jitter,
            update_sched=update_schedule,
            initial_sampler=initial_sampler,
        )
        self.collider = NearFarCollider(near_plane=cfg.near_plane, far_plane=cfg.far_plane)
        self.renderer_rgb = RGBRenderer(background_color=cfg.background_color)
        self.renderer_accumulation = AccumulationRenderer()
        self.renderer_depth = DepthRenderer(method="median")
        self.renderer_semantics = SemanticRenderer()
        self.pixel_losses = PixelLosses()

    # fruit_nerf.py:185-189
    def setup_inference(self, render_rgb: bool, num_inference_samples: int) -> None:
        self.render_rgb = render_rgb
        self.num_inference_samples = num_inference_samples
        self.proposal_sampler = UniformSamplerWithNoise(num_samples=self.num_inference_samples, single_jitter=False)
        self.field.spatial_distortion = None

    # fruit_nerf.py:191-196
    def get_param_groups(self) -> Dict[str, List[Parameter]]:
        param_groups: Dict[str, List[Parameter]] = {}
        param_groups["proposal_networks"] = list(self.proposal_networks.parameters())
        param_groups["fields"] = list(self.field.parameters())
        self.camera_optimizer.get_param_groups(param_groups=param_groups)
        return param_groups

    # fruit_nerf.py:198-232
    def get_training_callbacks(self, training_callback_attributes=None) -> List[TrainingCallback]:
        callbacks = []
        if self.config.use_proposal_weight_anneal:
            N = self.config.proposal_weights_anneal_max_num_iters

            def set_anneal(step):
                self.step = step
                train_frac = np.clip(step / N, 0, 1)

                def bias(x, b):
                    return b * x / ((b - 1) * x + 1)

                self.proposal_sampler.set_anneal(float(bias(train_frac, self.config.proposal_weights_anneal_slope)))

            callbacks.append(TrainingCallback(where_to_run=["BEFORE_TRAIN_ITERATION"], update_every_num_iters=1, func=set_anneal))
            callbacks.append(TrainingCallback(where_to_run=["AFTER_TRAIN_ITERATION"], update_every_num_iters=1, func=self.proposal_sampler.step_cb))
        return callbacks

    # ------------------------------------------------------------------------------------------------
    def _semantic_colormap(self, sem: Tensor) -> Tensor:
        # fruit_nerf.py:594-597: heaviside(sigmoid(sem) - 0.9, 0) -> colormap lookup, repeated to 3 channels
        labels = torch.heaviside(torch.sigmoid(sem.detach()) - 0.9, torch.zeros((), device=sem.device)).to(torch.long)
        return self.colormap.to(sem.device)[labels].repeat(1, 3)

    def _render(self, ray_bundle: RayBundle, depth_no_grad: bool, keep_lists: bool) -> Dict:
        cfg = self.config
        ray_samples, weights_list, ray_samples_list = self.proposal_sampler(ray_bundle, density_fns=self.density_fns)
        field_outputs = self.field.forward(ray_samples)
        weights = ray_samples.get_weights(field_outputs[FieldHeadNames.DENSITY])
        weights_list.append(weights)
        ray_samples_list.append(ray_samples)
        # RGB + accumulation + semantics share one compositing launch; semantic weights are detached unless
        # pass_semantic_gradients (fruit_nerf.py:586-591)
        mode, color = resolve_background(self.renderer_rgb.background_color)
        eval_mode = not self.training
        rgb, accumulation, _ = ops.render(weights, field_outputs[FieldHeadNames.RGB], None, mode, color, eval_mode)
        sem_w = weights if cfg.pass_semantic_gradients else weights.detach()
        _, _, semantics = ops.render(sem_w, None, field_outputs[FieldHeadNames.SEMANTICS], L.BG_NONE, None, False)
        depth = self.renderer_depth(weights=weights, ray_samples=ray_samples)
        outputs = {"rgb": rgb, "accumulation": accumulation, "depth": depth}
        if keep_lists:
            outputs["weights_list"] = weights_list
            outputs["ray_samples_list"] = ray_samples_list
        for i in range(cfg.num_proposal_iterations):
            outputs[f"prop_depth_{i}"] = self.renderer_depth(weights=weights_list[i], ray_samples=ray_samples_list[i])
        outputs["semantics"] = semantics
        outputs["semantics_colormap"] = self._semantic_colormap(semantics)
        return outputs

    # fruit_nerf.py:543-599
    def get_outputs(self, ray_bundle: RayBundle) -> Dict:
        self.camera_optimizer.apply_to_raybundle(ray_bundle)
        if not self.training and not torch.is_grad_enabled() and self.fused_render and ray_bundle.origins.dim() == 2 and self._fused().eligible():
            # export / projection / eval-image loops: the whole chunk in one C call (csrc/pipeline.cu)
            outputs = self._fused().render(ray_bundle, want_inds=self.proposal_sampler.pdf_sampler.keep_inds)
            if "pdf_inds" in outputs:
                self.proposal_sampler.pdf_sampler.last_inds = outputs.pop("pdf_inds")
            outputs["semantics_colormap"] = self._semantic_colormap(outputs["semantics"])
            return outputs
        return self._render(ray_bundle, depth_no_grad=True, keep_lists=self.training)

    def _fused(self):
        if self._fused_pipeline is None:
            from .pipeline import FusedPipeline

            self._fused_pipeline = FusedPipeline(self)
        return self._fused_pipeline

    # fruit_nerf.py:497-541
    def get_inference_outputs(self, ray_bundle: RayBundle) -> Dict:
        return self._render(ray_bundle, depth_no_grad=False, keep_lists=True)

    # fruit_nerf.py:476-494
    def get_export_outputs(self, ray_bundle: RayBundle) -> Dict:
        ray_samples = self.proposal_sampler(ray_bundle)
        field_outputs = self.field.forward(ray_samples)
        outputs = {
            "rgb": field_outputs[FieldHeadNames.RGB],
            "point_location": ray_samples.frustums.get_positions(),
            "semantics": field_outputs[FieldHeadNames.SEMANTICS][..., 0],
            "density": field_outputs[FieldHeadNames.DENSITY][..., 0],
        }
        sem = outputs["semantics"]
        outputs["semantics_colormap"] = torch.heaviside(torch.sigmoid(sem) - 0.9, torch.zeros((), device=sem.device)).to(torch.long)
        return outputs

    def load_state_dict(self, *args, **kwargs):
        self._params_version = getattr(self, "_params_version", 0) + 1  # cached kernel descriptors (mean appearance embedding) are stale now
        return super().load_state_dict(*args, **kwargs)

    def state_dict(self, *args, **kwargs):
        # a checkpoint writer copies the parameters on ITS stream: make that stream wait for an optimiser step still in flight on a side stream
        fence = self.__dict__.get("_param_fence")
        if fence is not None:
            fence()
        return super().state_dict(*args, **kwargs)

    # fruit_nerf.py:617-637
    def forward(self, ray_bundle: RayBundle) -> Dict:
        fence = self.__dict__.get("_param_fence")
        if fence is not None:  # an optimiser step may still be writing the field parameters on a side stream (engine.Trainer): make this stream wait
            fence()
        if self.collider is not None:
            ray_bundle = self.collider(ray_bundle)
        if self.test_mode == "inference":
            return self.get_inference_outputs(ray_bundle)
        if self.test_mode == "export":
            return self.get_export_outputs(ray_bundle)
        return self.get_outputs(ray_bundle)

    # fruit_nerf.py:601-615
    def get_loss_dict(self, outputs: Dict, batch: Dict, metrics_dict=None) -> Dict[str, Tensor]:
        image = batch["image"].to(self.device)
        mse, bce = self.pixel_losses(outputs["rgb"], outputs["semantics"], image[:, :3], batch["fruit_mask"].to(self.device),
                                     self.config.semantic_loss_weight)
        loss_dict = {"rgb_loss": mse, "semantics_loss": bce}
        if self.training:
            loss_dict["interlevel_loss"] = self.config.interlevel_loss_mult * interlevel_loss(outputs["weights_list"], outputs["ray_samples_list"])
        self.camera_optimizer.get_loss_dict(loss_dict)
        return loss_dict

    # fruit_nerf.py:639-645
    def get_metrics_dict(self, outputs: Dict, batch: Dict) -> Dict[str, Tensor]:
        image = batch["image"].to(self.device)
        mse, _ = ops.pixel_losses(outputs["rgb"].detach(), outputs["semantics"].detach(), image[:, :3], batch["fruit_mask"].to(self.device), 0.0)
        metrics = {"psnr": 10.0 * torch.log10(1.0 / mse), "distortion": distortion_loss(outputs["weights_list"], outputs["ray_samples_list"])}
        self.camera_optimizer.get_metrics_dict(metrics)
        return metrics

    # ------------------------------------------------------------------------------------------------
    # chunked image-render loops (fruit_nerf.py:320-404)
    def _chunks(self, camera_ray_bundle: RayBundle):
        n = len(camera_ray_bundle)
        step = self.config.eval_num_rays_per_chunk
        for i in range(0, n, step):
            yield camera_ray_bundle.get_row_major_sliced_ray_bundle(i, i + step).to(self.device)

    # fruit_nerf.py:320-344: accumulated opacity in front of the cluster AABB
    @torch.no_grad()
    def get_density_for_camera_ray_bundle(self, camera_ray_bundle: RayBundle) -> Tensor:
        out = []
        for ray_bundle in self._chunks(camera_ray_bundle):
            ray_samples, _, _ = self.proposal_sampler(ray_bundle, density_fns=self.density_fns)
            field_outputs = self.field.forward(ray_samples)
            weights = ray_samples.get_weights(field_outputs[FieldHeadNames.DENSITY])
            out.append(self.renderer_accumulation(weights)[:, 0])
        return torch.cat(out).cpu()

    @torch.no_grad()
    def _render_chunks(self, camera_ray_bundle: RayBundle) -> Dict[str, Tensor]:
        """Chunked render of a (host or device) ray bundle -> host tensors.  Chunks go up with non-blocking copies, every
        chunk's outputs come down with non-blocking copies into PINNED host buffers that are cached per output shape (valid
        until the next call), and the stream is synchronised once at the end -- not one ``.cpu()`` per output per chunk as in
        fruit_nerf.py:363-369."""
        n = len(camera_ray_bundle)
        step = self.config.eval_num_rays_per_chunk
        flat = camera_ray_bundle.flatten()
        host: Dict[str, Tensor] = {}
        for i in range(0, n, step):
            ray_bundle = flat._map(lambda t: t[i : i + step].to(self.device, non_blocking=True))
            outputs = self.forward(ray_bundle=ray_bundle)
            for name, output in outputs.items():
                if not isinstance(output, torch.Tensor):
                    continue
                if name not in host:
                    # one grow-only pinned buffer per output (not one per distinct ray count: jagged bundles differ call to call)
                    key = (name, tuple(output.shape[1:]), output.dtype)
                    buf = self._pinned.get(key)
                    if buf is None or buf.shape[0] < n:
                        buf = torch.empty((n, *output.shape[1:]), dtype=output.dtype, pin_memory=True)
                        self._pinned[key] = buf
                    host[name] = buf[:n]
                host[name][i : i + output.shape[0]].copy_(output, non_blocking=True)
        torch.cuda.current_stream(self.device).synchronize()
        return host

    # fruit_nerf.py:346-374
    def get_outputs_for_camera_jagged_ray_bundle(self, camera_ray_bundle: RayBundle) -> Dict[str, Tensor]:
        return self._render_chunks(camera_ray_bundle)

    # fruit_nerf.py:377-404
    def get_outputs_for_camera_ray_bundle(self, camera_ray_bundle: RayBundle) -> Dict[str, Tensor]:
        image_height, image_width = camera_ray_bundle.origins.shape[:2]
        outputs = self._render_chunks(camera_ray_bundle)
        return {name: t.view(image_height, image_width, -1) for name, t in outputs.items()}
