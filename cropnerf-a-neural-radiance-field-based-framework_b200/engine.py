"""Training-step driver: what nerfstudio's ``Trainer.train_iteration`` does around the hot path for the ``fruit_nerf``
method (``fruit_nerf_config.py:29-65``; call stack SURVEY.md section 3.1), on flat parameter / gradient buffers.

* parameters of each param group (``proposal_networks`` / ``fields`` / ``camera_opt``, fruit_nerf.py:191-196) are
  re-homed as views into one contiguous fp32 buffer per group, gradients likewise -- one fused Adam launch and one
  NCCL all-reduce per group instead of one per tensor;
* data parallelism = the reference's only strategy (DDP, ``fruit_pipeline.py:119-121``): every rank renders its own
  rays, gradients are averaged with ``torch.distributed.all_reduce`` over the flat buffers (NCCL over NVLink on the
  GPU box, gloo in the CPU tests of the host logic);
* Adam(lr 1e-2, eps 1e-15) + ExponentialDecay(lr_final 1e-4, max_steps 200k) = ``fruit_nerf_config.py:45-60``.
"""
from __future__ import annotations

import math
from dataclasses import dataclass, field
from typing import Dict, List, Optional

import torch
import torch.distributed as dist
from torch import Tensor, nn

from . import ops


@dataclass
class OptimizerSpec:
    lr: float = 1e-2
    eps: float = 1e-15
    betas: tuple = (0.9, 0.999)
    lr_final: Optional[float] = 1e-4
    max_steps: int = 200000
    kind: str = "adam"   # "adam" (fruit_nerf_config.py:45-60) | "radam" (the _big / _huge presets, fruit_nerf_config.py:100-108)


DEFAULT_OPTIMIZERS = {
    "proposal_networks": OptimizerSpec(),
    "fields": OptimizerSpec(),
    "camera_opt": OptimizerSpec(lr=1e-3, lr_final=1e-4, max_steps=5000),
}


# the optimizers of `fruit_nerf_big` / `fruit_nerf_huge` (fruit_nerf_config.py:100-118,152-170): RAdam, no schedule on the proposal networks
BIG_PRESET_OPTIMIZERS = {
    "proposal_networks": OptimizerSpec(lr=1e-2, eps=1e-15, lr_final=None, kind="radam"),
    "fields": OptimizerSpec(lr=1e-2, eps=1e-15, lr_final=1e-4, max_steps=50000, kind="radam"),
    "camera_opt": OptimizerSpec(lr=1e-3, eps=1e-15, lr_final=1e-4, max_steps=5000),
}


def exponential_decay_lr(step: int, spec: OptimizerSpec) -> float:
    """nerfstudio ExponentialDecayScheduler (no warm-up): log-linear interpolation lr -> lr_final over max_steps."""
    if spec.lr_final is None:
        return spec.lr
    t = min(max(step / spec.max_steps, 0.0), 1.0)
    return math.exp(math.log(spec.lr) * (1 - t) + math.log(spec.lr_final) * t)


def step_scalars(spec: OptimizerSpec, lr: float, t: int, inv_scale: float = 1.0) -> tuple:
    """The seven per-step scalars of the flat-group update kernels, ``p -= (s0 / s4) * m / (sqrt(v) / s5 + s3)`` with m, v the Adam moments:
    ``(lr, beta1, beta2, eps, 1 - beta1^t, sqrt(1 - beta2^t), 1 / grad_scale)`` for torch.optim.Adam.  torch.optim.RAdam is the same kernel with
    other scalars: rectified steps (rho_t > 5) multiply lr by the rectification term and divide eps by sqrt(1 - beta2^t) (RAdam adds eps
    BEFORE the bias correction of the denominator); the first steps (rho_t <= 5) have no adaptive denominator, i.e. sqrt(v) / inf + 1."""
    # the kernels hold the betas as fp32: the bias corrections are taken of THOSE values (as the C entries that compute them do), otherwise
    # (1 - beta2) of the moment update and 1 - beta2^t of its correction disagree by 1e-5 relative at t = 1
    b1, b2 = (float(torch.tensor(x, dtype=torch.float32)) for x in spec.betas)
    bc1, bc2 = 1.0 - b1**t, 1.0 - b2**t
    if spec.kind == "adam":
        return (lr, b1, b2, spec.eps, bc1, math.sqrt(bc2), inv_scale)
    if spec.kind != "radam":
        raise ValueError(f"optimizer kind {spec.kind!r}: 'adam' or 'radam'")
    rho_inf = 2.0 / (1.0 - b2) - 1.0
    rho_t = rho_inf - 2.0 * t * (b2**t) / bc2
    if rho_t > 5.0:
        rect = math.sqrt((rho_t - 4.0) * (rho_t - 2.0) * rho_inf / ((rho_inf - 4.0) * (rho_inf - 2.0) * rho_t))
        return (lr * rect, b1, b2, spec.eps / math.sqrt(bc2), bc1, math.sqrt(bc2), inv_scale)
    return (lr, b1, b2, 1.0, bc1, float("inf"), inv_scale)


class GradScaler:
    """torch.amp.GradScaler semantics for the flat-group optimiser (nerfstudio Trainer: ``grad_scaler.scale(loss).backward()``,
    ``optimizer_scaler_step_all(grad_scaler)``, ``grad_scaler.update()``; enabled there whenever ``mixed_precision`` is).
    The scale multiplies the loss-gradient seed of ``cnb_train_step`` (``cnb_train_cfg.grad_scale``), the inf/NaN check over
    the flat gradients (``cnb_grad_check_finite``) and the decision to skip the Adam update (``cnb_adam_step_zero_guarded``)
    happen on the device; :meth:`update` reads the 4-byte flag back to grow / back off the scale like ``_amp_update_scale_``."""

    def __init__(self, init_scale: float = 65536.0, growth_factor: float = 2.0, backoff_factor: float = 0.5, growth_interval: int = 2000,
                 enabled: bool = True):
        self.scale = float(init_scale) if enabled else 1.0
        self.growth_factor, self.backoff_factor, self.growth_interval = growth_factor, backoff_factor, growth_interval
        self.enabled = enabled
        self.growth_tracker = 0
        self.found_inf: Optional[Tensor] = None
        self.skipped_steps = 0

    def flag(self, device) -> Tensor:
        if self.found_inf is None or self.found_inf.device != torch.device(device):
            self.found_inf = torch.zeros((1,), device=device, dtype=torch.int32)
        return self.found_inf

    def update(self) -> bool:
        """-> True when the step just taken was skipped.  Resets the flag for the next step."""
        if not self.enabled or self.found_inf is None:
            return False
        skipped = bool(self.found_inf.item())
        if skipped:
            self.scale *= self.backoff_factor
            self.growth_tracker = 0
            self.skipped_steps += 1
            self.found_inf.zero_()
        else:
            self.growth_tracker += 1
            if self.growth_tracker == self.growth_interval:
                self.scale *= self.growth_factor
                self.growth_tracker = 0
        return skipped

    def state_dict(self) -> dict:
        return {"scale": self.scale, "growth_factor": self.growth_factor, "backoff_factor": self.backoff_factor,
                "growth_interval": self.growth_interval, "_growth_tracker": self.growth_tracker}

    def load_state_dict(self, sd: dict) -> None:
        if sd:
            self.scale = float(sd.get("scale", self.scale))
            self.growth_tracker = int(sd.get("_growth_tracker", 0))


class FlatGroup:
    """One param group flattened: ``param.data`` and ``param.grad`` become views of two contiguous buffers."""

    ALIGN = 64  # floats

    def __init__(self, params: List[nn.Parameter], comm=None):
        """``comm`` (ddp.PeerComm): allocate the parameter and gradient buffers as symmetric (peer-mapped) memory."""
        uniq, seen = [], set()
        for p in params:
            if id(p) not in seen:
                seen.add(id(p))
                uniq.append(p)
        self.params = uniq
        # every tensor starts on a 256-byte boundary: the kernels use 8/16-byte vector loads and reductions on the tables
        offsets, n = [], 0
        for p in uniq:
            offsets.append(n)
            n += (p.numel() + self.ALIGN - 1) // self.ALIGN * self.ALIGN
        dev = uniq[0].device
        self.peer = None
        self.live = None
        self.half = None   # (fp16 copy, first float, float count) of a hash table in the group whose copy the update refreshes (Trainer)
        if comm is not None:
            from .ddp import PeerGroup

            self.flat, p_ptrs, mc_p = comm.alloc_floats(n)
            self.grad, g_ptrs, mc_g = comm.alloc_floats(n)
            self.peer = PeerGroup(comm, g_ptrs, p_ptrs, mc_g, mc_p)
        else:
            self.flat = torch.empty((n,), device=dev, dtype=torch.float32)
            self.grad = torch.zeros((n,), device=dev, dtype=torch.float32)
        self.exp_avg = torch.zeros_like(self.flat)
        self.exp_avg_sq = torch.zeros_like(self.flat)
        self.flat.zero_()
        for p, off in zip(uniq, offsets):
            k = p.numel()
            self.flat[off : off + k].copy_(p.data.reshape(-1))
            p.data = self.flat[off : off + k].view(p.shape)
            p.grad = self.grad[off : off + k].view(p.shape)

    def zero_grad(self) -> None:
        self.grad.zero_()

    def build_live(self, model: nn.Module) -> None:
        """Bitmap of the float4 units the optimiser has to visit (ops.reachable_bitmap): hash-table rows that no lattice corner hashes to
        have zero gradient and zero Adam moments forever, so skipping them is bit-identical to the dense pass.  Units whose moments are
        already non-zero (a resumed run of something else) are kept live."""
        from .field_components import HashEncoding

        mine = {id(p) for p in self.params}
        tables, table_ids = [], set()
        for mod in model.modules():
            if isinstance(mod, HashEncoding) and id(mod.hash_table) in mine and id(mod.hash_table) not in table_ids:
                table_ids.add(id(mod.hash_table))
                num_levels, log2_T, scalings = mod.grid_cfg()
                tables.append((mod.hash_table, num_levels, log2_T, scalings))
        others = [p for p in self.params if id(p) not in table_ids]
        self.live = ops.reachable_bitmap(self.flat, tables, others)
        self.include_nonzero_moments()
        if self.peer is not None:
            self.peer.struct.live = self.live.data_ptr()

    def include_nonzero_moments(self) -> None:
        if self.live is None:
            return
        n4 = (self.flat.numel() + 3) // 4
        nz = ((self.exp_avg != 0) | (self.exp_avg_sq != 0))
        nz = torch.nn.functional.pad(nz, (0, 4 * n4 - nz.numel())).view(n4, 4).any(dim=1)
        nz = torch.nn.functional.pad(nz, (0, 32 * self.live.numel() - n4)).view(-1, 32).to(torch.int64)
        words = (nz << torch.arange(32, device=nz.device, dtype=torch.int64)).sum(dim=1)
        words = torch.where(words >= 2**31, words - 2**32, words).to(torch.int32)
        self.live |= words

    def live_fraction(self) -> float:
        if self.live is None:
            return 1.0
        n4 = (self.flat.numel() + 3) // 4
        bits = sum(int(((self.live >> k) & 1).sum()) for k in range(32))
        return bits / n4


def _stats_views(losses: Tensor) -> Dict[str, Tensor]:
    """names of the loss buffer cnb_train_step fills (psnr / total are finalised on the device: no per-step torch kernels here)"""
    return {"rgb_loss": losses[0], "semantics_loss": losses[1], "interlevel_loss": losses[2], "distortion": losses[3], "psnr": losses[4], "loss": losses[5],
            "camera_opt_regularizer": losses[6]}


class _GraphedStep:
    """One captured CUDA graph of ``cnb_train_step`` for a fixed (ray count, proposal-update flag, anneal) combination.
    Inputs are copied into static buffers, jitter is drawn eagerly into a static buffer, then the graph is replayed: the
    ~50 kernels of a step are submitted with one launch."""

    RING = 256

    def __init__(self, trainer: "Trainer", ray_bundle, batch, update: bool):
        dev = ray_bundle.origins.device
        R = ray_bundle.origins.shape[0]
        fp = trainer.fused
        self.static = {
            "origins": torch.empty((R, 3), device=dev), "directions": torch.empty((R, 3), device=dev),
            "camera_indices": torch.empty((R, 1), device=dev, dtype=torch.int32),
            "image": torch.empty((R, 3), device=dev), "fruit_mask": torch.empty((R, 1), device=dev),
        }
        self.cam64 = torch.zeros((R, 1), device=dev, dtype=torch.int64)
        self._pending_scalars = None
        self.opt_dev = None
        self.jitter = fp.draw_jitter(R, dev).clone()
        # torch.rand inside a capture is graph-safe (the generator's philox offset advances per replay): the default jitter is drawn by the
        # graph itself; custom rand_fn feeds (tests) are drawn eagerly into the static buffer before each replay
        s_ = trainer.model.proposal_sampler
        self.jitter_in_graph = bool(s_.initial_sampler.single_jitter) and s_.initial_sampler.rand_fn is torch.rand and s_.pdf_sampler.rand_fn is torch.rand
        self._load(ray_bundle, batch)
        from .rays import RayBundle

        self.bundle = RayBundle(self.static["origins"], self.static["directions"], None, self.static["camera_indices"])
        self.batch = {"image": self.static["image"], "fruit_mask": self.static["fruit_mask"]}
        self.update = update
        # single GPU: the optimiser runs INSIDE the step -- each flat group's fused Adam + gradient clear right behind the backward chain
        # that completes its gradient, overlapping the other chain (cnb_opt_group); per-step scalars go through a small device buffer
        self.opt = None
        self.defer_fields = False
        peer = trainer.comm is not None
        cam_opt = trainer.model.camera_optimizer
        self.camera_opt = cam_opt if cam_opt.mode != "off" else None
        allowed = {"fields", "proposal_networks"} | ({"camera_opt"} if (self.camera_opt is not None and trainer.world_size == 1) else set())
        if (trainer.world_size == 1 or peer) and trainer.grad_scaler is None and set(trainer.groups) <= allowed:
            from . import _lib as L_

            # ... except the big "fields" group when the trainer pipelines it: its Adam pass (HBM bound) then runs on a side stream next to the
            # NEXT step's samplers + proposal forward (L1 bound, reads no field parameter) and only gates that step's field forward.
            # Data parallel over peer memory: the same split -- the small proposal group's exchange (barrier, reduce-scatter + Adam +
            # all-gather, barrier, clear) is a stage INSIDE the graph on the proposal chain's branch, next to the field backward; the fields
            # group's exchange runs on the library's side stream behind the step (Trainer._p2p_optimizer_step) and gates the next field forward
            self.defer_fields = (trainer.defer_fields or peer) and "fields" in trainer.groups
            names = [n for n in trainer.groups if not (self.defer_fields and n == "fields")]
            # ring of pinned rows: the host may run several steps ahead of the stream that executes the copies
            self.opt_host = torch.zeros((self.RING, len(names), 8), dtype=torch.float32, pin_memory=True)
            self.opt_np = self.opt_host.numpy()
            self.opt_dev = torch.zeros((len(names), 8), device=dev, dtype=torch.float32)
            self.opt = []
            for i, n in enumerate(names):
                g = trainer.groups[n]
                pinfo = None
                if peer:
                    zero = n == "proposal_networks" and not update   # frozen proposal networks: momentum-only step, no peer reads
                    mm = trainer.ddp == "p2p_multimem" and g.peer.has_multicast
                    pinfo = (trainer.comm.struct, g.peer.struct, (L_.P2P_GRADS_ZERO if zero else 0) | (L_.P2P_MULTIMEM if mm else 0), 2 + (i & 1))
                chain = {"fields": L_.CHAIN_FIELD, "proposal_networks": L_.CHAIN_PROPOSALS, "camera_opt": L_.CHAIN_JOIN}[n]
                self.opt.append((g.flat, g.grad, g.exp_avg, g.exp_avg_sq, self.opt_dev[i], chain, g.live, pinfo, g.half))
            self.opt_names = names
            self.inv_world = 1.0 / trainer.world_size
        self.graph = torch.cuda.CUDAGraph()
        self.graph2 = None
        self.graphB = None
        torch.cuda.synchronize()
        if trainer.world_size > 1 and trainer.comm is None:
            # data parallel over NCCL: two graphs, so the all-reduce of the field gradients (67 MB) can start after the field backward
            # and run on NCCL's stream while the proposal networks back-propagate (cnb_train_cfg.phase)
            with torch.cuda.graph(self.graph):
                self._narrow_camera_indices()
                if self.jitter_in_graph:
                    self.jitter.uniform_()
                self.losses, self.outputs, state = fp.train_step(self.bundle, self.batch, jitter=self.jitter, update_proposals=update, phase=1,
                                                                 grad_scale=trainer._loss_scale())
            self.graph2 = torch.cuda.CUDAGraph()
            with torch.cuda.graph(self.graph2, pool=self.graph.pool()):
                fp.train_step(self.bundle, self.batch, update_proposals=update, phase=2, state=state)
            self._state = state
        elif trainer.comm is not None or self.defer_fields:
            # graph A = samplers + proposal forward (reads no field parameter), graph B = the rest.  The field group's update of the PREVIOUS
            # step (peer-memory exchange, Trainer._p2p_optimizer_step; or plain Adam on one GPU) runs on a side stream and only has to land
            # before graph B
            with torch.cuda.graph(self.graph):
                self._narrow_camera_indices()
                if self.jitter_in_graph:
                    self.jitter.uniform_()
                self.losses, self.outputs, state = fp.train_step(self.bundle, self.batch, jitter=self.jitter, update_proposals=update, phase=3,
                                                                 grad_scale=trainer._loss_scale(), opt_groups=self.opt, camera_opt=self.camera_opt)
            self.graphB = torch.cuda.CUDAGraph()
            with torch.cuda.graph(self.graphB, pool=self.graph.pool()):
                fp.train_step(self.bundle, self.batch, update_proposals=update, phase=4, state=state)
            self._state = state
        else:
            with torch.cuda.graph(self.graph):
                self._narrow_camera_indices()
                if self.jitter_in_graph:
                    self.jitter.uniform_()
                self.losses, self.outputs = fp.train_step(self.bundle, self.batch, jitter=self.jitter, update_proposals=update, grad_scale=trainer._loss_scale(),
                                                          opt_groups=self.opt, camera_opt=self.camera_opt)
        self.stats = _stats_views(self.losses)
        for g in trainer.groups.values():  # whatever the capture-time warm-up left in the gradients
            g.zero_grad()

    def _load(self, ray_bundle, batch) -> None:
        st = self.static
        R = st["origins"].shape[0]
        cam = ray_bundle.camera_indices
        srcs = (ray_bundle.origins, ray_bundle.directions, cam, batch["image"], batch["fruit_mask"])
        dsts = (st["origins"], st["directions"], self.cam64, st["image"], st["fruit_mask"])
        plain = cam.dtype == torch.int64 and batch["image"].shape[-1] == 3 and all(t.is_contiguous() for t in srcs) \
            and all(t.dtype == torch.float32 for t in (srcs[0], srcs[1], srcs[3], srcs[4])) \
            and all(d.numel() * d.element_size() == t.numel() * t.element_size() for d, t in zip(dsts, srcs))
        scal = self._pending_scalars
        self._pending_scalars = None
        if plain and all((not t.is_cuda) and t.is_pinned() for t in srcs):
            # pinned host batch: raw async copies issued by ONE C call (cnb_upload), no framework dispatch per tensor; the int64 camera
            # indices go up as they are and are narrowed to the kernels' int32 inside the graph
            import ctypes as C

            from . import _lib as L

            n = len(srcs)
            d_arr = (C.c_void_p * n)(*[d.data_ptr() for d in dsts])
            s_arr = (C.c_void_p * n)(*[t.data_ptr() for t in srcs])
            b_arr = (C.c_int64 * n)(*[t.numel() * t.element_size() for t in srcs])
            L.check(L.lib().cnb_upload(d_arr, s_arr, b_arr, n, L.stream_ptr(st["origins"].device)), "upload")
            if scal is not None:
                self.opt_dev.copy_(scal, non_blocking=True)
            return
        if plain and all(t.is_cuda and t.data_ptr() % 16 == 0 for t in srcs):
            # device-resident batch: the five copies AND the optimiser's scalars in one kernel launch (cnb_stage_inputs)
            import ctypes as C

            from . import _lib as L

            n = len(srcs)
            d_arr = (C.c_void_p * n)(*[d.data_ptr() for d in dsts])
            s_arr = (C.c_void_p * n)(*[t.data_ptr() for t in srcs])
            b_arr = (C.c_int64 * n)(*[t.numel() * t.element_size() for t in srcs])
            ns = 0
            f_arr = None
            if scal is not None:
                vals = scal.reshape(-1).tolist()
                ns = len(vals)
                f_arr = (C.c_float * ns)(*vals)
            L.check(L.lib().cnb_stage_inputs(d_arr, s_arr, b_arr, n, self.opt_dev.data_ptr() if ns else None, f_arr, ns, L.stream_ptr(st["origins"].device)),
                    "stage_inputs")
            return
        st["origins"].copy_(ray_bundle.origins.reshape(R, 3), non_blocking=True)
        st["directions"].copy_(ray_bundle.directions.reshape(R, 3), non_blocking=True)
        self.cam64.copy_(cam.reshape(R, 1), non_blocking=True)
        st["image"].copy_(batch["image"][:, :3], non_blocking=True)
        st["fruit_mask"].copy_(batch["fruit_mask"].reshape(R, 1), non_blocking=True)
        if scal is not None:
            self.opt_dev.copy_(scal, non_blocking=True)

    def _narrow_camera_indices(self) -> None:
        """captured at the head of the graph: the kernels' int32 camera indices from the uploaded int64 ones (one tiny kernel)"""
        self.static["camera_indices"].copy_(self.cam64)

    def set_optimizer_scalars(self, trainer: "Trainer", step: int) -> None:
        """lr / bias corrections of THIS step for the in-graph Adam passes (one 64-byte async H2D copy)."""
        trainer.opt_step += 1
        t = trainer.opt_step
        slot = t % self.RING
        for i, name in enumerate(self.opt_names):
            spec = trainer.optimizers[name]
            b1, b2 = spec.betas
            self.opt_np[slot, i, :7] = step_scalars(spec, exponential_decay_lr(step, spec), t, self.inv_world)
        self._pending_scalars = self.opt_host[slot]   # travels with the step's inputs (_load): kernel parameters or one async H2D copy

    def run(self, trainer: "Trainer", ray_bundle, batch):
        self._load(ray_bundle, batch)
        if not self.jitter_in_graph:
            trainer.fused.draw_jitter(self.static["origins"].shape[0], self.static["origins"].device, out=self.jitter)
        probe = trainer._probe  # measurement aid (bench.py): CUDA events around the two graphs of a pipelined step
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)] if (probe is not None and self.graphB is not None) else None
        if ev:
            ev[0].record()
        self.graph.replay()
        if self.graph2 is not None:
            trainer.start_all_reduce("fields")
            self.graph2.replay()
        if self.graphB is not None:
            if ev:
                ev[1].record()
            trainer.wait_deferred_update()  # the previous step's field-group exchange must have landed before the field forward
            if ev:
                ev[2].record()
            self.graphB.replay()
            if ev:
                ev[3].record()
                probe.append(ev)
        return self.losses, self.outputs


class Trainer:
    """Minimal trainer for FruitModel: callbacks, forward, losses, backward, gradient all-reduce, Adam."""

    def __init__(self, model, optimizers: Optional[Dict[str, OptimizerSpec]] = None, world_size: int = 1, fused: bool = True,
                 cuda_graph: bool = False, force_proposal_update: bool = False, grad_scaler: Optional[GradScaler] = None, ddp: str = "auto"):
        """``ddp`` (world_size > 1): "nccl" = all-reduce of the flat gradients + local Adam (DDP as the reference does it);
        "p2p" = one reduce-scatter + Adam + all-gather kernel per group over NVLink peer mappings (csrc/ddp_p2p.cu);
        "p2p_multimem" = the same through the NVLS multicast mappings; "auto" = p2p when the symmetric-memory rendezvous works
        (CUDA, peer access), else nccl.  A GradScaler needs the global inf/NaN verdict before any update: it keeps nccl.  So do fp16 field
        tables (FruitField table_precision="fp16"): the peer-memory exchange does not refresh their copy, and "p2p*" refuses them."""
        from .pipeline import FusedPipeline

        self.model = model
        self.fused = FusedPipeline(model) if fused else None
        self.cuda_graph = cuda_graph                      # replay one captured graph per step when the step's scalars allow it
        self.force_proposal_update = force_proposal_update  # benchmark aid: every step back-propagates into the proposal networks
        self._graphs: Dict[tuple, _GraphedStep] = {}
        self._pending: Dict[str, object] = {}
        self.world_size = world_size
        self.grad_scaler = grad_scaler if (grad_scaler is not None and grad_scaler.enabled) else None
        self.optimizers = optimizers or DEFAULT_OPTIMIZERS
        self.comm = None
        self._side_stream = None
        self._ddp_steps = None
        self._deferred_event = None
        self._deferred_pending = False
        import os as _os

        self.defer_fields = _os.environ.get("CNB_NO_DEFER", "0") != "1"  # one GPU: pipeline the field group's Adam into the next step (graphed steps)
        self._probe = None                # bench.py sets a list: per-step CUDA events of the pipelined step (graph A | wait | graph B)
        self.graph_during_anneal = False  # True: capture a graph per distinct anneal value as well (tests)
        self._camopt_eager = _os.environ.get("CNB_CAMOPT_EAGER", "0") == "1"
        self.check_peers_every = 64       # peer-memory mode: read the barrier time-out flag every N steps (and before checkpoints)
        self.ddp = "nccl"
        field = getattr(model, "field", None)
        fp16_tables = getattr(field, "table_precision", "fp32") == "fp16"
        if fp16_tables and world_size > 1 and ddp in ("p2p", "p2p_multimem"):
            raise ValueError(f"ddp={ddp!r} does not refresh the fp16 copy of the field table (table_precision='fp16'): use ddp='nccl'")
        if world_size > 1 and ddp != "nccl" and self.grad_scaler is None and not fp16_tables and next(model.parameters()).is_cuda:
            try:
                from .ddp import PeerComm

                self.comm = PeerComm.create(next(model.parameters()).device)
                # measured (tests/ddp_p2p_check.py, profiles/): every rank both pulls gradients and pushes parameters, so each link direction
                # carries 2 (N-1)/N of the flat groups with peer loads / stores but only ~1x with NVLS (the switch reduces and replicates):
                # multimem wins from N = 4 up (N=8: 0.24 vs 0.30 ms), plain peer access at N = 2 (0.19 vs 0.26 ms)
                want_mm = ddp == "p2p_multimem" or (ddp == "auto" and world_size >= 4)
                self.ddp = "p2p_multimem" if (want_mm and self.comm.multicast) else "p2p"
            except Exception as e:  # no peer access / symmetric memory unavailable: the NCCL path is the alternative GPU path
                if ddp != "auto":
                    raise
                import warnings

                warnings.warn(f"peer-memory data parallelism unavailable ({type(e).__name__}: {e}); using the NCCL all-reduce path")
                self.comm = None
        self.groups: Dict[str, FlatGroup] = {name: FlatGroup(params, self.comm) for name, params in model.get_param_groups().items() if len(params) > 0}
        if _os.environ.get("CNB_NO_LIVE_MASK", "0") != "1" and next(model.parameters()).is_cuda:
            for g in self.groups.values():
                g.build_live(model)
        if fp16_tables:
            # every update of the fields group also writes the fp16 copy of the field table (from registers: one 8-byte store per float4)
            g, t = self.groups["fields"], field.mlp_base_grid.hash_table
            first = (t.data_ptr() - g.flat.data_ptr()) // 4
            if not 0 <= first <= g.flat.numel() - t.numel():
                raise RuntimeError("the field hash table is not inside the fields parameter group")
            g.half = (field.table_half, first, t.numel())
        self.callbacks = model.get_training_callbacks()
        self.opt_step = 0

    def _refresh_table_copy(self) -> None:
        """fp16 field tables: a write made outside the trainer since the last step (checkpoint load, an in-place copy) is copied into the fp16
        table before the step reads it; re-homing the parameters into the flat group counts as such a write."""
        field = getattr(self.model, "field", None)
        if field is not None and getattr(field, "table_precision", "fp32") == "fp16" and field.table_copy_stale():
            self.wait_deferred_update()
            field.refresh_table_copy()

    def _run_callbacks(self, where: str, step: int) -> None:
        for cb in self.callbacks:
            if where in cb.where_to_run and step % cb.update_every_num_iters == 0:
                cb.func(step)

    def start_all_reduce(self, name: str) -> None:
        """Launch the SUM all-reduce of one flat gradient group asynchronously (NCCL's own stream, ordered after the work
        already enqueued on the current stream)."""
        if self.world_size > 1 and self.comm is None and name in self.groups and name not in self._pending:
            self._pending[name] = dist.all_reduce(self.groups[name].grad, op=dist.ReduceOp.SUM, async_op=True)

    def all_reduce_gradients(self, proposals_updated: bool = True, wait: bool = True) -> None:
        """DDP semantics (fruit_pipeline.py:119-121): mean of the per-rank gradients.  The 1/world_size factor is
        folded into the Adam kernel (``inv_grad_scale``).  On steps where the proposal networks are frozen their gradient
        is exactly zero on every rank (the schedule is a function of the step), so that group is not communicated --
        DDP's ``find_unused_parameters=True`` behaviour."""
        self._proposals_updated = proposals_updated
        if self.world_size > 1 and self.comm is None:
            for name in self.groups:
                if name == "proposal_networks" and not proposals_updated:
                    continue
                self.start_all_reduce(name)
            if wait:  # train_iteration passes wait=False: optimizer_step then waits group by group
                for work in self._pending.values():
                    work.wait()
                self._pending.clear()

    def optimizer_step(self, step: int, pipelined: bool = False) -> None:
        """Adam over every flat group.  Groups whose all-reduce is still in flight are waited for one at a time, largest
        (launched first) first, so the Adam pass of one group hides the tail of the next group's all-reduce."""
        self.opt_step += 1
        order = sorted(self.groups, key=lambda n: -self.groups[n].flat.numel())
        if self.comm is not None:
            self._p2p_optimizer_step(step, order, pipelined=pipelined)
            return
        scaler = self.grad_scaler
        flag = None
        inv = 1.0 / self.world_size
        if scaler is not None:
            # GradScaler.step: one inf/NaN flag over ALL groups (after the all-reduce, so every rank decides alike), then every
            # group's Adam either runs or is skipped on the device
            inv /= scaler.scale
            flag = scaler.flag(self.groups[order[0]].flat.device)
            for name in order:
                work = self._pending.pop(name, None)
                if work is not None:
                    work.wait()
                ops.grad_check_finite(self.groups[name].grad, flag)
        for name in order:
            g = self.groups[name]
            work = self._pending.pop(name, None)
            if work is not None:
                work.wait()
            spec = self.optimizers[name]
            lr = exponential_decay_lr(step, spec)
            # Adam and the gradient clear of the next step in one pass over the flat group
            if spec.kind != "adam":
                if flag is not None:
                    raise NotImplementedError("RAdam with a GradScaler: the guarded update kernel computes Adam's bias corrections itself")
                ops.adam_step_scalars(g.flat, g.grad, g.exp_avg, g.exp_avg_sq, step_scalars(spec, lr, self.opt_step, inv), live=g.live, half=g.half)
                continue
            ops.adam_step(g.flat, g.grad, g.exp_avg, g.exp_avg_sq, lr, self.opt_step, spec.betas[0], spec.betas[1], spec.eps,
                          inv_grad_scale=inv, zero_grad=True, skip_flag=flag, live=g.live, half=g.half)
        self._grads_clean = True
        if scaler is not None and scaler.update():
            self.opt_step -= 1  # torch: a skipped optimizer.step() does not advance Adam's step count

    def _p2p_optimizer_step(self, step: int, order: List[str], pipelined: bool = False) -> None:
        """barrier -> one reduce-scatter + Adam + all-gather kernel per flat group over the peer mappings -> barrier -> clear the
        own gradients.  Every rank owns 1/world of each group's Adam moments (ddp.owned_range); a group whose gradient is zero on
        every rank this step (frozen proposal networks) skips the peer reads but still takes its (momentum-only) Adam step.

        ``pipelined`` (graphed steps): the big "fields" group -- 87 % of the bytes -- is exchanged on a side stream on its own barrier
        channel and only has to land before the NEXT step's field forward (graph B of _GraphedStep); the next step's samplers and
        proposal forward, which read no field parameter, overlap it.  The small groups take the synchronous route on the caller's stream.
        The whole sequence is ONE C call (cnb_ddp_optimizer_step): ~15 us of host time instead of ~0.3 ms of Python."""
        import ctypes as C

        from . import _lib as L

        comm = self.comm
        if any(self.optimizers[name].kind != "adam" for name in order):
            raise NotImplementedError("RAdam over the peer-memory exchange (its kernel computes Adam's bias corrections from the step count): use ddp='nccl'")
        if self._ddp_steps is None or len(self._ddp_steps) != len(order):
            self._ddp_steps = (L.DdpGroupStep * len(order))()
            for i, name in enumerate(order):
                g, spec, d = self.groups[name], self.optimizers[name], self._ddp_steps[i]
                d.group = C.pointer(g.peer.struct)
                d.exp_avg, d.exp_avg_sq, d.grad_own, d.n = g.exp_avg.data_ptr(), g.exp_avg_sq.data_ptr(), g.grad.data_ptr(), g.flat.numel()
                d.beta1, d.beta2, d.eps = spec.betas[0], spec.betas[1], spec.eps
                d.inv_grad_scale = 1.0 / self.world_size
        any_deferred = False
        for i, name in enumerate(order):
            g, spec, d = self.groups[name], self.optimizers[name], self._ddp_steps[i]
            zero = name == "proposal_networks" and not getattr(self, "_proposals_updated", True)
            mm = self.ddp == "p2p_multimem" and g.peer.has_multicast
            d.lr, d.step = exponential_decay_lr(step, spec), self.opt_step
            d.flags = (L.P2P_GRADS_ZERO if zero else 0) | (L.P2P_MULTIMEM if mm else 0)
            d.deferred = 1 if (pipelined and name == "fields") else 0
            any_deferred = any_deferred or bool(d.deferred)
        L.check(L.lib().cnb_ddp_optimizer_step(C.byref(comm.struct), self._ddp_steps, len(order), L.stream_ptr(comm.device)), "ddp_optimizer_step")
        if any_deferred:
            self._deferred_pending = True
            self.model._param_fence = self.wait_deferred_update  # eval / export forwards on any stream wait for it (FruitModel.forward)
        self._grads_clean = True
        if self.check_peers_every and self.opt_step % self.check_peers_every == 0:
            self.check_peers()

    def check_peers(self) -> None:
        """Peer-memory mode: a barrier that timed out (stalled or dead peer) only sets a flag on the device and lets the stream carry on,
        so the update that followed may have used stale peer gradients.  Read the flag (one 4-byte D2H read) and fail loudly instead of
        letting replicas diverge silently; called every ``check_peers_every`` steps, by ``gather_optimizer_state`` and before checkpoints."""
        if self.comm is not None and self.comm.timed_out():
            raise RuntimeError("cropnerf_b200: a peer-memory barrier timed out (stalled or dead peer): replicas may have diverged; "
                               "restart from the last checkpoint (or train with ddp='nccl')")

    def _deferred_fields_adam(self, step: int) -> None:
        """One GPU, graphed steps: the field group's fused Adam + gradient clear on a side stream, fenced by an event that the next step's
        field forward (graph B), eval forwards (FruitModel.forward) and every non-graphed path wait for."""
        dev = self.groups["fields"].flat.device
        main = torch.cuda.current_stream(dev)
        if self._side_stream is None:
            self._side_stream = torch.cuda.Stream(device=dev)
            self._deferred_event = torch.cuda.Event()
        self._side_stream.wait_stream(main)
        g = self.groups["fields"]
        spec = self.optimizers["fields"]
        with torch.cuda.stream(self._side_stream):
            if spec.kind != "adam":
                ops.adam_step_scalars(g.flat, g.grad, g.exp_avg, g.exp_avg_sq, step_scalars(spec, exponential_decay_lr(step, spec), self.opt_step), live=g.live,
                                      half=g.half)
            else:
                ops.adam_step(g.flat, g.grad, g.exp_avg, g.exp_avg_sq, exponential_decay_lr(step, spec), self.opt_step, spec.betas[0], spec.betas[1],
                              spec.eps, inv_grad_scale=1.0, zero_grad=True, live=g.live, half=g.half)
            self._deferred_event.record(self._side_stream)
        self._deferred_pending = True
        self.model._param_fence = self.wait_deferred_update

    def wait_deferred_update(self) -> None:
        """Make the current stream wait for the field group's deferred update / exchange (no-op when none is in flight)."""
        if not self._deferred_pending:
            return
        if self.comm is not None:
            from . import _lib as L

            L.check(L.lib().cnb_ddp_wait_deferred(L.stream_ptr(self.comm.device)), "ddp_wait_deferred")
        else:
            torch.cuda.current_stream().wait_event(self._deferred_event)
        # the flag stays set: several streams (the next training step, an eval forward) may have to wait for the same update, and waiting for an
        # event that has already completed costs nothing

    def gather_optimizer_state(self) -> None:
        """Peer-memory mode keeps each group's Adam moments only inside the rank's owned slice: fill in the other ranks' slices
        (one broadcast per rank and buffer) so that every rank holds the full state, e.g. before writing a checkpoint."""
        if self.comm is None:
            return
        self.wait_deferred_update()
        self.check_peers()
        from .ddp import owned_range

        for g in self.groups.values():
            for r in range(self.world_size):
                lo, hi = owned_range(g.flat.numel(), r, self.world_size)
                if hi > lo:
                    dist.broadcast(g.exp_avg[lo:hi], src=r)
                    dist.broadcast(g.exp_avg_sq[lo:hi], src=r)

    def _loss_scale(self) -> float:
        return self.grad_scaler.scale if self.grad_scaler is not None else 1.0

    def _use_fused(self) -> bool:
        return self.fused is not None and self.model.collider is not None and self.fused.eligible()

    def train_iteration(self, step: int, ray_bundle, batch: Dict[str, Tensor]) -> Dict[str, Tensor]:
        if not self.model.training:  # nn.Module.train() walks every sub-module: only when the mode actually changes
            self.model.train()
        self._run_callbacks("BEFORE_TRAIN_ITERATION", step)
        self._refresh_table_copy()
        self.model._params_version = getattr(self.model, "_params_version", 0) + 1  # invalidates the eval path's cached descriptors
        graphed = False
        if not getattr(self, "_grads_clean", False):
            for g in self.groups.values():
                g.zero_grad()
        self._grads_clean = False
        if self._use_fused():
            # one C call: samplers + proposal networks + field + renderers + losses + backward (csrc/pipeline.cu)
            fp = self.fused
            in_graph_opt = False
            updated = True if self.force_proposal_update else fp.proposals_updated()
            sampler = self.model.proposal_sampler
            cam_opt = self.model.camera_optimizer
            # row a17: the SO3xR3 camera optimizer runs INSIDE the C call (corrections applied before the samplers, dLoss/d rays chained into
            # pose_adjustment.grad together with the regulariser; csrc/camera_opt.cu) -- graph-replayable like the rest of the step.
            # CNB_CAMOPT_EAGER=1 keeps the round-1 route (torch pose algebra with autograd around the step) for A/B runs
            fused_camopt = cam_opt.mode != "off" and not self._camopt_eager
            if cam_opt.mode != "off" and not fused_camopt:
                cam_opt.apply_to_raybundle(ray_bundle)
                reg: Dict[str, Tensor] = {}
                cam_opt.get_loss_dict(reg)
                for v in reg.values():
                    v.backward()
            # rays / targets may be HOST tensors (pinned): the graphed step copies them straight into its static device buffers
            host_in = not ray_bundle.origins.is_cuda
            dev = self.model.device

            def on_device():
                if not host_in:
                    return ray_bundle, batch
                return ray_bundle.to(dev, non_blocking=True), {k: v.to(dev, non_blocking=True) for k, v in batch.items() if isinstance(v, Tensor)}

            # anneal is a kernel argument baked into the captured graph and moves every step for the first
            # proposal_weights_anneal_max_num_iters (1000) iterations: those steps run the same C call eagerly instead of
            # capturing (and throwing away) one graph per step; from then on anneal == 1 and one graph per (R, updated) is replayed
            anneal = float(sampler._anneal)
            graphable = self.cuda_graph and ray_bundle.nears is None and (cam_opt.mode == "off" or (fused_camopt and self.world_size == 1 and self.grad_scaler is None))
            if graphable and anneal != 1.0 and (int(ray_bundle.origins.shape[0]), updated, anneal, self._loss_scale()) not in self._graphs:
                graphable = self.graph_during_anneal
            if graphable:
                key = (int(ray_bundle.origins.shape[0]), updated, anneal, self._loss_scale())
                gs = self._graphs.get(key)
                if gs is None:
                    if len(self._graphs) >= 8:
                        self._graphs.pop(next(iter(self._graphs)))
                    # a deferred `fields` update (side-stream Adam / peer-memory exchange) of the previous step may still be reading and
                    # clearing the gradient buffer this warm-up accumulates into, and writing the parameters it reads
                    self.wait_deferred_update()
                    rb_d, batch_d = on_device()
                    fp.train_step(rb_d, batch_d, update_proposals=False, want_metrics=True, camera_opt=cam_opt if fused_camopt else None)  # eager warm-up (func attributes, workspace)
                    for g in self.groups.values():
                        g.zero_grad()
                    gs = self._graphs[key] = _GraphedStep(self, rb_d, batch_d, updated)
                in_graph_opt = gs.opt is not None
                graphed = True
                if in_graph_opt:
                    gs.set_optimizer_scalars(self, step)
                losses, outputs = gs.run(self, ray_bundle, batch)
                if updated:
                    sampler._steps_since_update = 0
            else:
                self.wait_deferred_update()
                rb_d, batch_d = on_device()
                losses, outputs = fp.train_step(rb_d, batch_d, update_proposals=updated, grad_scale=self._loss_scale(), camera_opt=cam_opt if fused_camopt else None)
            if in_graph_opt:
                self._grads_clean = True  # the step updated the parameters and cleared the gradients itself
                if gs.defer_fields and self.comm is not None:
                    self._proposals_updated = updated
                    self._p2p_optimizer_step(step, ["fields"], pipelined=True)   # opt_step was advanced by set_optimizer_scalars
                elif gs.defer_fields:
                    self._deferred_fields_adam(step)
            else:
                self.all_reduce_gradients(proposals_updated=updated, wait=False)
                if graphed and self.comm is not None:
                    self.optimizer_step(step, pipelined=True)
                else:
                    self.optimizer_step(step)
            self._run_callbacks("AFTER_TRAIN_ITERATION", step)
            if graphed:  # the graphed step writes the same static loss buffer every replay: its views are made once
                return gs.stats
            return _stats_views(losses)
        self.wait_deferred_update()
        outputs = self.model(ray_bundle)
        metrics = self.model.get_metrics_dict(outputs, batch)
        loss_dict = self.model.get_loss_dict(outputs, batch, metrics)
        loss = sum(loss_dict.values())
        (loss * self._loss_scale()).backward()
        self.all_reduce_gradients()
        self.optimizer_step(step)
        self._run_callbacks("AFTER_TRAIN_ITERATION", step)
        out = dict(loss_dict)
        out.update(metrics)
        out["loss"] = loss.detach()
        return out
