"""nerfstudio method plugin for the B200 path: the shape of ``crop_nerf/fruit_nerf/fruit_nerf_config.py:29-65``.

``fruit_nerf_b200_method`` is a ``MethodSpecification`` named ``fruit_nerf_b200`` with the reference's trainer / optimizer / scheduler
settings, the reference's own pipeline, data manager and data parser (``fruit_nerf.fruit_pipeline`` / ``fruit_nerf.data``: out of scope
here, used as they are), and a model config whose ``_target`` builds this package's ``FruitModel`` behind nerfstudio's ``Model`` interface.
Register it like the reference does (``README.md:79``)::

    export NERFSTUDIO_METHOD_CONFIGS="fruit_nerf_b200=cropnerf_b200.method_config:fruit_nerf_b200_method"

nerfstudio and the reference package are NOT part of this image (no network): everything below the guard is exercised only by
``tests/ref_dropin.py``-style shims (which prove the class-for-class substitution on the reference's unmodified model file); when the
imports fail, ``fruit_nerf_b200_method`` is ``None`` and ``UNAVAILABLE`` says why.  Importing this module never raises.
"""
from __future__ import annotations

from dataclasses import dataclass, field
from typing import Dict, List, Type

UNAVAILABLE = None
fruit_nerf_b200_method = None
fruit_nerf_b200_method_big = None    # fruit_nerf_config.py:66-118
fruit_nerf_b200_method_huge = None   # fruit_nerf_config.py:120-190

try:
    from nerfstudio.cameras.camera_optimizers import CameraOptimizerConfig  # type: ignore
    from nerfstudio.configs.base_config import ViewerConfig  # type: ignore
    from nerfstudio.engine.optimizers import AdamOptimizerConfig, RAdamOptimizerConfig  # type: ignore
    from nerfstudio.engine.schedulers import ExponentialDecaySchedulerConfig  # type: ignore
    from nerfstudio.engine.trainer import TrainerConfig  # type: ignore
    from nerfstudio.models.base_model import Model  # type: ignore
    from nerfstudio.models.nerfacto import NerfactoModelConfig  # type: ignore
    from nerfstudio.plugins.types import MethodSpecification  # type: ignore

    from fruit_nerf.data.cotton_nerf_dataparser import CottonNerfDataParserConfig  # type: ignore
    from fruit_nerf.data.fruit_datamanager import FruitDataManagerConfig  # type: ignore
    from fruit_nerf.fruit_pipeline import FruitPipelineConfig  # type: ignore
except Exception as e:  # nerfstudio / the reference package are absent
    UNAVAILABLE = f"{type(e).__name__}: {e}"
else:
    from . import fruit_nerf as _b200

    @dataclass
    class FruitNerfB200ModelConfig(NerfactoModelConfig):
        """``FruitNerfModelConfig`` (fruit_nerf.py:59-68) + ``precision``; ``_target`` = the adapter below."""

        _target: Type = field(default_factory=lambda: FruitModelB200)
        semantic_loss_weight: float = 1.0
        pass_semantic_gradients: bool = False
        num_layers_semantic: int = 2
        hidden_dim_semantics: int = 64
        geo_feat_dim: int = 15
        precision: str = "mixed"   # the reference preset trains with mixed_precision=True (fruit_nerf_config.py:35)

    class FruitModelB200(Model):
        """nerfstudio ``Model`` whose modules are this package's (``FruitModel.populate_modules``, fruit_nerf.py:87-183).  Every method
        nerfstudio's Trainer / Pipeline / exporter calls is forwarded to :class:`cropnerf_b200.fruit_nerf.FruitModel`."""

        config: FruitNerfB200ModelConfig

        def __init__(self, config, metadata: Dict, **kwargs) -> None:
            self._metadata = metadata
            self.test_mode = kwargs.get("test_mode", "val")
            super().__init__(config=config, **kwargs)

        def populate_modules(self):
            super().populate_modules()
            names = _b200.FruitNerfModelConfig.__dataclass_fields__
            kw = {k: getattr(self.config, k) for k in names if hasattr(self.config, k) and k != "camera_optimizer_mode"}
            kw["camera_optimizer_mode"] = getattr(getattr(self.config, "camera_optimizer", None), "mode", "off")
            self.b200 = _b200.FruitModel(_b200.FruitNerfModelConfig(**kw), scene_box=self.scene_box, num_train_data=self.num_train_data,
                                         metadata=self._metadata, test_mode=self.test_mode)
            # nerfstudio reaches for these attributes (viewer, exporter, BayesRays)
            for name in ("field", "proposal_networks", "proposal_sampler", "density_fns", "collider", "camera_optimizer", "renderer_rgb",
                         "renderer_accumulation", "renderer_depth", "renderer_semantics"):
                setattr(self, name, getattr(self.b200, name))

        def setup_inference(self, render_rgb, num_inference_samples):
            self.b200.setup_inference(render_rgb, num_inference_samples)
            self.proposal_sampler = self.b200.proposal_sampler

        def get_param_groups(self) -> Dict[str, List]:
            return self.b200.get_param_groups()

        def get_training_callbacks(self, training_callback_attributes):
            from nerfstudio.engine.callbacks import TrainingCallback, TrainingCallbackLocation  # type: ignore

            loc = {"BEFORE_TRAIN_ITERATION": TrainingCallbackLocation.BEFORE_TRAIN_ITERATION, "AFTER_TRAIN_ITERATION": TrainingCallbackLocation.AFTER_TRAIN_ITERATION}
            return [TrainingCallback(where_to_run=[loc[w] for w in cb.where_to_run], update_every_num_iters=cb.update_every_num_iters, func=cb.func)
                    for cb in self.b200.get_training_callbacks()]

        def get_outputs(self, ray_bundle):
            self.b200.train(self.training)
            return self.b200.get_outputs(ray_bundle)

        def forward(self, ray_bundle):
            self.b200.train(self.training)
            return self.b200(ray_bundle)

        def get_loss_dict(self, outputs, batch, metrics_dict=None):
            return self.b200.get_loss_dict(outputs, batch, metrics_dict)

        def get_metrics_dict(self, outputs, batch):
            return self.b200.get_metrics_dict(outputs, batch)

        def get_outputs_for_camera_ray_bundle(self, camera_ray_bundle):
            return self.b200.get_outputs_for_camera_ray_bundle(camera_ray_bundle)

        def get_image_metrics_and_images(self, outputs, batch):
            raise NotImplementedError("image metrics (psnr / ssim / lpips panels) are outside the ray-render path (SURVEY.md section 2)")

    def _opt(lr: float, lr_final: float, max_steps: int) -> dict:
        return {"optimizer": AdamOptimizerConfig(lr=lr, eps=1e-15), "scheduler": ExponentialDecaySchedulerConfig(lr_final=lr_final, max_steps=max_steps)}

    fruit_nerf_b200_method = MethodSpecification(
        config=TrainerConfig(
            method_name="fruit_nerf_b200",
            steps_per_eval_batch=500,
            steps_per_save=2000,
            max_num_iterations=40000,
            mixed_precision=False,   # the kernels carry their own precision mode (FruitNerfB200ModelConfig.precision); no autocast / GradScaler needed
            pipeline=FruitPipelineConfig(
                datamanager=FruitDataManagerConfig(dataparser=CottonNerfDataParserConfig(), train_num_rays_per_batch=4096, eval_num_rays_per_batch=4096),
                model=FruitNerfB200ModelConfig(eval_num_rays_per_chunk=1 << 15),
            ),
            optimizers={"proposal_networks": _opt(1e-2, 1e-4, 200000), "fields": _opt(1e-2, 1e-4, 200000), "camera_opt": _opt(1e-3, 1e-4, 5000)},
            viewer=ViewerConfig(num_rays_per_chunk=1 << 15),
            vis="viewer",
        ),
        description="FruitNeRF / CropNeRF ray-render path on hand-written sm_100a kernels (cropnerf_b200)",
    )

    def _ropt(lr_final, max_steps) -> dict:
        return {"optimizer": RAdamOptimizerConfig(lr=1e-2, eps=1e-15),
                "scheduler": None if lr_final is None else ExponentialDecaySchedulerConfig(lr_final=lr_final, max_steps=max_steps)}

    # The two larger presets (fruit_nerf_config.py:66-190).  Their FruitField is wider than the fused kernels (128-wide three-layer semantic MLP,
    # geo_feat_dim 30).  Registered in exact fp32 (`precision="fp32"`: layers above 64 on csrc/mlp_wide.cu); `--pipeline.model.precision mixed`
    # runs them as the reference trains them, on the tensor-core operator csrc/mlp_mixed.cu.  The optimizers are the reference's (nerfstudio's
    # RAdam; `engine.BIG_PRESET_OPTIMIZERS` is the same for this package's own Trainer).
    fruit_nerf_b200_method_big = MethodSpecification(
        config=TrainerConfig(
            method_name="fruit_nerf_b200_big", steps_per_eval_batch=500, steps_per_save=2000, max_num_iterations=100000, mixed_precision=False,
            pipeline=FruitPipelineConfig(
                datamanager=FruitDataManagerConfig(train_num_images_to_sample_from=200, train_num_times_to_repeat_images=1000,
                                                   dataparser=CottonNerfDataParserConfig(train_split_fraction=0.99),
                                                   train_num_rays_per_batch=4096 * 2, eval_num_rays_per_batch=4096),
                model=FruitNerfB200ModelConfig(eval_num_rays_per_chunk=1 << 15, num_nerf_samples_per_ray=128, num_proposal_samples_per_ray=(512, 256),
                                               hidden_dim=128, geo_feat_dim=30, hidden_dim_color=128, hidden_dim_semantics=128, num_layers_semantic=3,
                                               appearance_embed_dim=128, max_res=4096, proposal_weights_anneal_max_num_iters=5000,
                                               log2_hashmap_size=21, precision="fp32"),
            ),
            optimizers={"proposal_networks": _ropt(None, 0), "fields": _ropt(1e-4, 50000), "camera_opt": _opt(1e-3, 1e-4, 5000)},
            viewer=ViewerConfig(num_rays_per_chunk=1 << 15),
            vis="viewer",
        ),
        description="FruitNeRF-Big on the cropnerf_b200 kernels (exact fp32 mode)",
    )
    fruit_nerf_b200_method_huge = MethodSpecification(
        config=TrainerConfig(
            method_name="fruit_nerf_b200_huge", steps_per_eval_batch=500, steps_per_save=2000, max_num_iterations=100000, mixed_precision=False,
            pipeline=FruitPipelineConfig(
                datamanager=FruitDataManagerConfig(dataparser=CottonNerfDataParserConfig(), train_num_rays_per_batch=4096 * 4, eval_num_rays_per_batch=4096),
                model=FruitNerfB200ModelConfig(
                    eval_num_rays_per_chunk=1 << 15, num_nerf_samples_per_ray=64, num_proposal_samples_per_ray=(512, 512),
                    proposal_net_args_list=[{"hidden_dim": 16, "log2_hashmap_size": 17, "num_levels": 5, "max_res": 512, "use_linear": False},
                                            {"hidden_dim": 16, "log2_hashmap_size": 17, "num_levels": 7, "max_res": 2048, "use_linear": False}],
                    hidden_dim=256, hidden_dim_color=256, appearance_embed_dim=32, geo_feat_dim=30, hidden_dim_semantics=128, num_layers_semantic=3,
                    max_res=8192, proposal_weights_anneal_max_num_iters=5000, log2_hashmap_size=21, precision="fp32"),
            ),
            optimizers={"proposal_networks": _ropt(None, 0), "fields": _ropt(1e-4, 50000), "camera_opt": _opt(1e-3, 1e-4, 5000)},
            viewer=ViewerConfig(num_rays_per_chunk=1 << 15),
            vis="viewer",
        ),
        description="FruitNeRF-Huge on the cropnerf_b200 kernels (exact fp32 mode)",
    )
