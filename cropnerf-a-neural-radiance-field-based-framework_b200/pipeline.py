"""Fused ray-render pipeline: one C-ABI call per chunk of rays (``cnb_render_rays``) or per training batch
(``cnb_train_step``) instead of one call per nerfstudio module.

This is the fast path behind ``FruitModel.forward`` in no-grad mode (the export / projection / eval-image loops,
``fruit_nerf.py:320-404`` and ``export/exporter_utils_nerfacto.py:126-183``) and behind ``engine.Trainer`` (the training
step, SURVEY.md section 3.1).  The per-module operators in ``ops.py`` stay available for callers that compose the
nerfstudio modules themselves (BayesRays, custom density_fns); both routes run the same kernels.
"""
from __future__ import annotations

import ctypes as C
from typing import Dict, Optional, Tuple

import torch
from torch import Tensor

from . import _lib as L
from . import ops
from .density_fields import HashMLPDensityField
from .field_components import SceneContraction
from .renderers import resolve_background


class FusedPipeline:
    def __init__(self, model) -> None:
        self.model = model
        self._ws: Dict[Tuple[int, bool, str], Tensor] = {}
        self._tables: Dict[Tuple, Tensor] = {}
        self._ms_cache: Dict[str, tuple] = {}

    # ------------------------------------------------------------------------------------------------
    def eligible(self) -> bool:
        """True when the model is wired the way ``FruitModel.populate_modules`` wires it (fruit_nerf.py:87-183)."""
        from .ray_samplers import PDFSampler, ProposalNetworkSampler, SpacedSampler

        m = self.model
        s = m.proposal_sampler
        if not isinstance(s, ProposalNetworkSampler) or m.test_mode == "export":
            return False
        if not isinstance(s.initial_sampler, SpacedSampler) or not isinstance(s.pdf_sampler, PDFSampler):
            return False
        if s.num_proposal_network_iterations not in (1, 2) or len(m.density_fns) < s.num_proposal_network_iterations:
            return False
        for fn in m.density_fns[: s.num_proposal_network_iterations]:
            owner = getattr(fn, "__self__", None)
            if not isinstance(owner, HashMLPDensityField) or getattr(fn, "__func__", None) is not HashMLPDensityField.density_fn or owner.use_linear:
                return False
        sd = m.field.spatial_distortion
        return sd is None or isinstance(sd, SceneContraction)

    def _table(self, kind: str, n: int, dev) -> Tensor:
        key = (kind, n, str(dev))
        if key not in self._tables:  # torch.linspace on the host: bit-identical to the bins the reference samplers build
            t = torch.linspace(0.0, 1.0, n + 1) if kind == "lin" else torch.linspace(0.0, 1.0 - (1.0 / (n + 1)), steps=n + 1)
            self._tables[key] = t.to(dev)
        return self._tables[key]

    def _model_struct(self, dev, training: bool, with_grads: bool, ray_gradients: bool = False):
        """The cnb_model descriptor (pointers + hyper-parameters).  Eval / export loops call this once per chunk with unchanged parameters:
        the no-grad descriptor is cached and rebuilt only when something it depends on changes (parameter storage, a training step or
        load_state_dict -- ``model._params_version`` --, mode switches, background colour)."""
        m = self.model
        if not with_grads:
            m.field.table_half_current()  # a stale fp16 table copy is refreshed in place: the cached descriptor's pointer stays valid
            tab = m.field.mlp_base_grid.hash_table
            key = (str(dev), training, ray_gradients, m.field.test_mode, getattr(m, "_params_version", 0), tab.data_ptr(), m.field.spatial_distortion is None,
                   str(m.renderer_rgb.background_color), getattr(m.config, "precision", "fp32"), tuple(int(v) for v in m.proposal_sampler.num_proposal_samples_per_ray),
                   int(m.proposal_sampler.num_nerf_samples_per_ray), id(m.proposal_sampler), tuple(id(fn) for fn in m.density_fns))
            hit = self._ms_cache.get("eval")
            if hit is not None and hit[0] == key:
                return hit[1], hit[2]
            ms, keep = self._build_model_struct(dev, training, with_grads, ray_gradients)
            self._ms_cache["eval"] = (key, ms, keep)
            return ms, keep
        return self._build_model_struct(dev, training, with_grads, ray_gradients)

    def _build_model_struct(self, dev, training: bool, with_grads: bool, ray_gradients: bool = False):
        m = self.model
        keep = []
        field = m.field
        inference = field.test_mode in ("inference", "export")
        fcfg = field._cfg(inference)
        fcfg["training"] = training
        params = field.kernel_params()
        grads = None
        if with_grads:
            grads = []
            for p in params:
                if p.grad is None:
                    p.grad = torch.zeros_like(p)
                grads.append(p.grad)
        fs, k = ops._build_field(fcfg, params, grads)
        keep.append(k)
        ms = L.Model()
        ms.field = fs
        if fcfg["table_half"] is not None:
            ms.field_table_half = fcfg["table_half"].data_ptr()
        s = m.proposal_sampler
        n = s.num_proposal_network_iterations
        for i in range(n):
            net = m.density_fns[i].__self__
            mlp = net.mlp_base[1]
            ws, bs = [mlp.layers[0].weight, mlp.layers[1].weight], [mlp.layers[0].bias, mlp.layers[1].bias]
            tab = net.encoding.hash_table
            if with_grads:
                for p in (tab, *ws, *bs):
                    if p.grad is None:
                        p.grad = torch.zeros_like(p)
            nl, t, sc = net.encoding.grid_cfg()
            d = L.DensityField()
            d.grid = L.make_grid(tab.detach(), tab.grad if with_grads else None, nl, t, sc)
            d.mlp = L.make_mlp([w.detach() for w in ws], [b.detach() for b in bs], L.ACT_NONE, [w.grad for w in ws] if with_grads else None,
                               [b.grad for b in bs] if with_grads else None)
            d.warp = net._warp()
            d.average_init_density = float(net.average_init_density)
            d.precision = L.PREC_MIXED if getattr(m.config, "precision", "fp32") == "mixed" else L.PREC_FP32
            ms.proposal[i] = d
        sp = ms.sampler
        sp.num_proposal_iterations = n
        for i in range(n):
            sp.proposal_samples[i] = int(s.num_proposal_samples_per_ray[i])
        sp.nerf_samples = int(s.num_nerf_samples_per_ray)
        sp.initial_spacing = s.initial_sampler.spacing_kind
        sp.single_jitter = int(bool(s.initial_sampler.single_jitter))
        sp.histogram_padding = float(s.pdf_sampler.histogram_padding)
        sp.pdf_eps = 1e-5
        sp.lin_bins = self._table("lin", sp.proposal_samples[0], dev).data_ptr()
        counts = [sp.proposal_samples[i] for i in range(1, n)] + [sp.nerf_samples]
        for i, cnt in enumerate(counts):
            sp.u_base[i] = self._table("u", cnt, dev).data_ptr()
        mode, color = resolve_background(m.renderer_rgb.background_color)
        ms.bg_mode = mode
        for i in range(3):
            ms.bg_color[i] = float(color[i]) if color is not None else 0.0
        ms.ray_gradients = int(ray_gradients)
        return ms, keep

    def _rays_struct(self, ray_bundle, training: bool):
        m = self.model
        R = ray_bundle.origins.shape[0]
        keep = []

        def f32c(t):
            t = L.f32(t)
            keep.append(t)
            return t

        r = L.Rays()
        o, d = f32c(ray_bundle.origins.detach().reshape(R, 3)), f32c(ray_bundle.directions.detach().reshape(R, 3))
        r.origins, r.directions = o.data_ptr(), d.data_ptr()
        if ray_bundle.nears is not None and ray_bundle.fars is not None:
            r.nears = f32c(ray_bundle.nears.reshape(R)).data_ptr()
            r.fars = f32c(ray_bundle.fars.reshape(R)).data_ptr()
        col = m.collider
        r.near_plane = float(col.near_plane if (training or not getattr(col, "reset_near_plane", True)) else 0.0)
        r.far_plane = float(col.far_plane)
        cam = ray_bundle.camera_indices
        if cam is not None:
            cam = cam.reshape(R).to(torch.int32).contiguous()
            keep.append(cam)
            r.camera_indices = cam.data_ptr()
        r.num_rays = R
        return r, keep

    def _workspace(self, ms, R: int, training: bool, dev) -> Tensor:
        n = int(L.lib().cnb_render_workspace_floats(C.byref(ms), R, int(training)))
        # training workspaces are keyed by the exact ray count: captured CUDA graphs hold their addresses, and a trainer sees one or two
        # batch sizes.  Eval / export loops see a different remainder chunk on every call (the hit count of a projection pair, the tail
        # of an image): ONE grow-only buffer per device serves them all (the layout is computed from R inside the C call; it only needs
        # enough room), instead of one cached allocation per distinct ray count
        key = (R, True, str(dev)) if training else (0, False, str(dev))
        ws = self._ws.get(key)
        if ws is None or ws.numel() < n:
            ws = torch.empty((max(n, 1),), device=dev, dtype=torch.float32)
            self._ws[key] = ws
        return ws

    def _outputs(self, R: int, dev, n_prop: int, want_inds: bool, nerf_samples: int):
        out = L.RayOutputs()
        t = {
            "rgb": torch.empty((R, 3), device=dev, dtype=torch.float32),
            "depth": torch.empty((R, 1), device=dev, dtype=torch.float32),
            "accumulation": torch.empty((R, 1), device=dev, dtype=torch.float32),
            "semantics": torch.empty((R, 1), device=dev, dtype=torch.float32),
        }
        out.rgb, out.depth, out.accumulation, out.semantics = (t[k].data_ptr() for k in ("rgb", "depth", "accumulation", "semantics"))
        for i in range(n_prop):
            t[f"prop_depth_{i}"] = torch.empty((R, 1), device=dev, dtype=torch.float32)
            out.prop_depth[i] = t[f"prop_depth_{i}"].data_ptr()
        if want_inds:
            t["pdf_inds"] = torch.empty((R, nerf_samples + 1), device=dev, dtype=torch.int32)
            out.pdf_inds = t["pdf_inds"].data_ptr()
        return out, t

    # ------------------------------------------------------------------------------------------------
    def render(self, ray_bundle, want_inds: bool = False) -> Dict[str, Tensor]:
        """Eval-mode render of a flat bundle of rays -> the per-ray output dict of ``FruitModel.get_outputs``."""
        dev = ray_bundle.origins.device
        if dev.type != "cuda":
            raise RuntimeError("cropnerf_b200 renders on CUDA devices only; there is no CPU fallback")
        ms, keep = self._model_struct(dev, training=False, with_grads=False)
        rays, keep2 = self._rays_struct(ray_bundle, training=False)
        R = rays.num_rays
        ws = self._workspace(ms, R, False, dev)
        n_prop = ms.sampler.num_proposal_iterations
        out, tensors = self._outputs(R, dev, n_prop, want_inds, ms.sampler.nerf_samples)
        L.check(L.lib().cnb_render_rays(C.byref(ms), C.byref(rays), C.byref(out), ws.data_ptr(), L.stream_ptr(dev)), "render_rays")
        del keep, keep2
        return tensors

    def proposals_updated(self) -> bool:
        """ProposalNetworkSampler's "updated" rule (nerfstudio ray_samplers.py; SURVEY.md App. A.6)."""
        s = self.model.proposal_sampler
        return bool(s._steps_since_update > s.update_sched(s._step) or s._step < 10)

    def draw_jitter(self, R: int, dev, out: Optional[Tensor] = None) -> Tensor:
        """Jitter in the order the samplers draw it (initial sampler, then one draw per PDF resampling), flat."""
        s = self.model.proposal_sampler
        n_prop = s.num_proposal_network_iterations
        counts = [int(c) for c in s.num_proposal_samples_per_ray[:n_prop]] + [int(s.num_nerf_samples_per_ray)]
        single = bool(s.initial_sampler.single_jitter)
        fns = [s.initial_sampler.rand_fn] + [s.pdf_sampler.rand_fn] * n_prop
        if single and all(fn is torch.rand for fn in fns):
            if out is not None:
                return out.uniform_()
            return torch.rand(((n_prop + 1) * R,), device=dev, dtype=torch.float32)
        j = torch.cat([fn((R, 1) if single else (R, c + 1), dtype=torch.float32, device=dev).reshape(-1) for fn, c in zip(fns, counts)])
        return out.copy_(j) if out is not None else j

    def train_step(self, ray_bundle, batch: Dict[str, Tensor], grad_scale: float = 1.0, want_metrics: bool = True,
                   jitter: Optional[Tensor] = None, update_proposals: Optional[bool] = None, phase: int = 0,
                   state: Optional[tuple] = None, opt_groups: Optional[list] = None, camera_opt=None):
        """forward + losses + backward of one batch; gradients are accumulated into ``param.grad``.
        Returns (losses [8] device tensor: rgb, semantics, interlevel, distortion, ...; per-ray outputs)."""
        m = self.model
        dev = ray_bundle.origins.device
        s = m.proposal_sampler
        if phase in (2, 4):
            # second half of a split step (cnb_train_cfg.phase 1 -> 2, or 3 -> 4): same structs, workspace and outputs as the first call
            ms, rays, cfg, out, losses, ws, tensors, updated, keep = state
            cfg.phase = phase
            L.check(L.lib().cnb_train_step(C.byref(ms), C.byref(rays), C.byref(cfg), C.byref(out), losses.data_ptr(), ws.data_ptr(), L.stream_ptr(dev)),
                    f"train_step(phase {phase})")
            if updated:
                s._steps_since_update = 0
            return losses, tensors
        # row a17: when the ray origins / directions carry a graph (camera optimizer), the kernels also return dLoss/d rays
        ray_grads = bool(ray_bundle.origins.requires_grad or ray_bundle.directions.requires_grad)
        # camera optimizer INSIDE the step (cnb_train_cfg.pose_adjustment): the rays stay as the data manager produced them, the C call
        # applies the per-camera corrections, collects dLoss/d rays and chains them into pose_adjustment.grad (csrc/camera_opt.cu)
        fused_camopt = camera_opt is not None and getattr(camera_opt, "mode", "off") != "off"
        if fused_camopt and ray_grads:
            raise RuntimeError("rays that already carry an autograd graph cannot be combined with the in-step camera optimizer")
        ms, keep = self._model_struct(dev, training=True, with_grads=True, ray_gradients=ray_grads or fused_camopt)
        rays, keep2 = self._rays_struct(ray_bundle, training=True)
        R = rays.num_rays
        ws = self._workspace(ms, R, True, dev)
        n_prop = ms.sampler.num_proposal_iterations
        out, tensors = self._outputs(R, dev, n_prop, False, ms.sampler.nerf_samples)
        if jitter is None:
            jitter = self.draw_jitter(R, dev)
        updated = self.proposals_updated() if update_proposals is None else bool(update_proposals)
        cfg = L.TrainCfg()
        image = L.f32(batch["image"].to(dev)[:, :3])
        mask = L.f32(batch["fruit_mask"].to(dev)).reshape(R)
        cfg.image, cfg.fruit_mask, cfg.jitter = image.data_ptr(), mask.data_ptr(), jitter.data_ptr()
        cfg.anneal = float(s._anneal)
        cfg.semantic_loss_weight = float(m.config.semantic_loss_weight)
        cfg.interlevel_loss_mult = float(m.config.interlevel_loss_mult)
        cfg.grad_scale = float(grad_scale)
        cfg.update_proposals = int(bool(updated))
        cfg.want_metrics = int(want_metrics)
        cfg.phase = int(phase)
        cfg.num_opt_groups = 0
        if opt_groups:
            # optimiser stage inside the step (cnb_opt_group): (flat param, grad, exp_avg, exp_avg_sq, device scalars [8], chain)
            if len(opt_groups) > L.MAX_OPT_GROUPS:
                raise ValueError(f"at most {L.MAX_OPT_GROUPS} optimiser groups")
            for i, entry in enumerate(opt_groups):
                p_, g_, m_, v_, sc_, chain, live_ = entry[:7]
                og = cfg.opt_groups[i]
                og.live = live_.data_ptr() if live_ is not None else None
                og.param, og.grad, og.exp_avg, og.exp_avg_sq = p_.data_ptr(), g_.data_ptr(), m_.data_ptr(), v_.data_ptr()
                og.n, og.scalars, og.chain = p_.numel(), sc_.data_ptr(), int(chain)
                if len(entry) > 8 and entry[8] is not None:  # the group's fp16 table copy (engine.FlatGroup.half), refreshed by its update
                    tab_, first_, count_ = entry[8]
                    cfg.opt_half[i].table_half, cfg.opt_half[i].first, cfg.opt_half[i].count = tab_.data_ptr(), int(first_), int(count_)
                if len(entry) > 7 and entry[7] is not None:
                    # peer-memory data parallelism: this group's whole exchange runs inside the step (cnb_opt_group.peer_*); the structs are
                    # read at enqueue time, the entry keeps them alive
                    comm_struct, group_struct, flags, channel = entry[7]
                    og.peer_comm, og.peer_group = C.addressof(comm_struct), C.addressof(group_struct)
                    og.peer_flags, og.peer_channel = int(flags), int(channel)
            cfg.num_opt_groups = len(opt_groups)
        if fused_camopt:
            pose = camera_opt.pose_adjustment
            if pose.grad is None:
                pose.grad = torch.zeros_like(pose)
            ncam = int(pose.shape[0])
            key = ("camopt", R, ncam, str(dev))
            sc = self._ws.get(key)
            if sc is None:
                sc = torch.empty((12 * (R + ncam),), device=dev, dtype=torch.float32)
                self._ws[key] = sc
            if rays.camera_indices is None:
                raise AttributeError("Camera indices are not provided.")
            cfg.pose_adjustment, cfg.d_pose_adjustment, cfg.camopt_scratch = pose.data_ptr(), pose.grad.data_ptr(), sc.data_ptr()
            cfg.num_cameras = ncam
            cfg.trans_l2_penalty, cfg.rot_l2_penalty = float(camera_opt.trans_l2_penalty), float(camera_opt.rot_l2_penalty)
        d_o = d_d = None
        if ray_grads:
            if phase != 0:
                raise RuntimeError("ray gradients (camera optimizer) are not combined with the split (phase 1/2) train step")
            d_o = torch.zeros((R, 3), device=dev, dtype=torch.float32)
            d_d = torch.zeros((R, 3), device=dev, dtype=torch.float32)
            cfg.d_origins, cfg.d_directions = d_o.data_ptr(), d_d.data_ptr()
        losses = torch.empty((8,), device=dev, dtype=torch.float32)
        L.check(L.lib().cnb_train_step(C.byref(ms), C.byref(rays), C.byref(cfg), C.byref(out), losses.data_ptr(), ws.data_ptr(), L.stream_ptr(dev)),
                "train_step")
        if phase in (1, 3):
            return losses, tensors, (ms, rays, cfg, out, losses, ws, tensors, updated, (keep, keep2, image, mask, jitter))
        if updated:
            s._steps_since_update = 0
        if ray_grads:  # hand the ray gradients to whatever produced the rays (CameraOptimizer.apply_to_raybundle)
            roots = [t for t in (ray_bundle.origins, ray_bundle.directions) if t.requires_grad]
            grads = [g.view_as(t) for t, g in ((ray_bundle.origins, d_o), (ray_bundle.directions, d_d)) if t.requires_grad]
            torch.autograd.backward(roots, grads)
        del keep, keep2
        return losses, tensors
