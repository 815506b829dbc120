"""ctypes binding of ``libcropnerf_b200.so`` (C ABI declared in ``include/cropnerf_b200.h``).

The product path has no CPU fallback: :func:`lib` raises if the shared library is missing, and every
compute wrapper raises ``RuntimeError`` with ``cnb_last_error()`` when the library reports a failure
(e.g. no CUDA device).
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
from typing import Optional, Sequence

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libcropnerf_b200.so")
CSRC = os.path.join(_HERE, "csrc")
HEADER = os.path.join(os.path.dirname(_HERE), "include", "cropnerf_b200.h")

MAX_LEVELS = 16
MAX_LAYERS = 4
MAX_WIDTH = 64        # fused (shared-memory resident) MLP operators
WIDE_MAX_WIDTH = 256  # wider layers run layer by layer in exact fp32 (csrc/mlp_wide.cu)

PREC_FP32, PREC_MIXED = 0, 1
ACT_NONE, ACT_RELU, ACT_SIGMOID = 0, 1, 2
WARP_AABB, WARP_CONTRACT_LINF = 0, 1
SPACING_UNIFORM, SPACING_LINDISP_PIECEWISE = 0, 1
BG_NONE, BG_LAST_SAMPLE, BG_CONSTANT = 0, 1, 2
APP_PER_CAMERA, APP_MEAN, APP_ZERO = 0, 1, 2


class Grid(C.Structure):
    _fields_ = [
        ("table", C.c_void_p),
        ("d_table", C.c_void_p),
        ("num_levels", C.c_int32),
        ("log2_hashmap_size", C.c_int32),
        ("scalings", C.c_float * MAX_LEVELS),
    ]


class Mlp(C.Structure):
    _fields_ = [
        ("num_layers", C.c_int32),
        ("dims", C.c_int32 * (MAX_LAYERS + 1)),
        ("out_activation", C.c_int32),
        ("_pad", C.c_int32),
        ("W", C.c_void_p * MAX_LAYERS),
        ("b", C.c_void_p * MAX_LAYERS),
        ("dW", C.c_void_p * MAX_LAYERS),
        ("db", C.c_void_p * MAX_LAYERS),
    ]


class Warp(C.Structure):
    _fields_ = [("mode", C.c_int32), ("aabb_min", C.c_float * 3), ("aabb_max", C.c_float * 3)]


class Samples(C.Structure):
    _fields_ = [
        ("origins", C.c_void_p),
        ("directions", C.c_void_p),
        ("starts", C.c_void_p),
        ("ends", C.c_void_p),
        ("camera_indices", C.c_void_p),
        ("num_rays", C.c_int64),
        ("row_stride", C.c_int64),
        ("samples_per_ray", C.c_int32),
        ("_pad", C.c_int32),
    ]


class DensityField(C.Structure):
    _fields_ = [("grid", Grid), ("mlp", Mlp), ("warp", Warp), ("average_init_density", C.c_float), ("precision", C.c_int32)]


class Field(C.Structure):
    _fields_ = [
        ("grid", Grid),
        ("base", Mlp),
        ("sem", Mlp),
        ("sem_head", Mlp),
        ("rgb", Mlp),
        ("embedding", C.c_void_p),
        ("d_embedding", C.c_void_p),
        ("mean_embedding", C.c_void_p),
        ("warp", Warp),
        ("num_images", C.c_int32),
        ("appearance_dim", C.c_int32),
        ("geo_feat_dim", C.c_int32),
        ("appearance_mode", C.c_int32),
        ("pass_semantic_gradients", C.c_int32),
        ("precision", C.c_int32),
    ]


class Camera(C.Structure):
    _fields_ = [("c2w", C.c_float * 12), ("fx", C.c_float), ("fy", C.c_float), ("cx", C.c_float), ("cy", C.c_float),
                ("width", C.c_int32), ("height", C.c_int32)]


class ImageSet(C.Structure):
    _fields_ = [("images_u8", C.c_void_p), ("images_f32", C.c_void_p), ("masks_u8", C.c_void_p), ("cameras", C.c_void_p),
                ("num_images", C.c_int32), ("height", C.c_int32), ("width", C.c_int32)]


class Rays(C.Structure):
    _fields_ = [
        ("origins", C.c_void_p),
        ("directions", C.c_void_p),
        ("nears", C.c_void_p),
        ("fars", C.c_void_p),
        ("camera_indices", C.c_void_p),
        ("num_rays", C.c_int64),
        ("near_plane", C.c_float),
        ("far_plane", C.c_float),
    ]


class Sampler(C.Structure):
    _fields_ = [
        ("num_proposal_iterations", C.c_int32),
        ("proposal_samples", C.c_int32 * 2),
        ("nerf_samples", C.c_int32),
        ("initial_spacing", C.c_int32),
        ("single_jitter", C.c_int32),
        ("histogram_padding", C.c_float),
        ("pdf_eps", C.c_float),
        ("lin_bins", C.c_void_p),
        ("u_base", C.c_void_p * 2),
    ]


class Model(C.Structure):
    _fields_ = [
        ("field", Field),
        ("proposal", DensityField * 2),
        ("sampler", Sampler),
        ("bg_mode", C.c_int32),
        ("bg_color", C.c_float * 3),
        ("ray_gradients", C.c_int32),
    ]


class RayOutputs(C.Structure):
    _fields_ = [
        ("rgb", C.c_void_p),
        ("depth", C.c_void_p),
        ("accumulation", C.c_void_p),
        ("semantics", C.c_void_p),
        ("prop_depth", C.c_void_p * 2),
        ("pdf_inds", C.c_void_p),
    ]


MAX_OPT_GROUPS = 4
CHAIN_FIELD, CHAIN_PROPOSALS, CHAIN_JOIN = 0, 1, 2


class OptGroup(C.Structure):
    _fields_ = [("param", C.c_void_p), ("grad", C.c_void_p), ("exp_avg", C.c_void_p), ("exp_avg_sq", C.c_void_p), ("n", C.c_int64), ("scalars", C.c_void_p),
                ("chain", C.c_int32), ("_pad", C.c_int32), ("live", C.c_void_p), ("peer_comm", C.c_void_p), ("peer_group", C.c_void_p),
                ("peer_flags", C.c_int32), ("peer_channel", C.c_int32)]


class TrainCfg(C.Structure):
    _fields_ = [
        ("image", C.c_void_p),
        ("fruit_mask", C.c_void_p),
        ("jitter", C.c_void_p),
        ("anneal", C.c_float),
        ("semantic_loss_weight", C.c_float),
        ("interlevel_loss_mult", C.c_float),
        ("grad_scale", C.c_float),
        ("update_proposals", C.c_int32),
        ("want_metrics", C.c_int32),
        ("d_origins", C.c_void_p),
        ("d_directions", C.c_void_p),
        ("phase", C.c_int32),
        ("num_opt_groups", C.c_int32),
        ("opt_groups", OptGroup * MAX_OPT_GROUPS),
        ("pose_adjustment", C.c_void_p),
        ("d_pose_adjustment", C.c_void_p),
        ("camopt_scratch", C.c_void_p),
        ("num_cameras", C.c_int32),
        ("trans_l2_penalty", C.c_float),
        ("rot_l2_penalty", C.c_float),
        ("_pad_camopt", C.c_int32),
    ]


MAX_PEERS = 16
P2P_GRADS_ZERO, P2P_MULTIMEM = 1, 2


class P2PComm(C.Structure):
    _fields_ = [("world", C.c_int32), ("rank", C.c_int32), ("flags", C.c_void_p * MAX_PEERS), ("state", C.c_void_p), ("timeout_ms", C.c_int32),
                ("channel", C.c_int32)]


class P2PGroup(C.Structure):
    _fields_ = [("grad", C.c_void_p * MAX_PEERS), ("param", C.c_void_p * MAX_PEERS), ("mc_grad", C.c_void_p), ("mc_param", C.c_void_p), ("live", C.c_void_p)]


class DdpGroupStep(C.Structure):
    _fields_ = [("group", C.POINTER(P2PGroup)), ("exp_avg", C.c_void_p), ("exp_avg_sq", C.c_void_p), ("grad_own", C.c_void_p), ("n", C.c_int64),
                ("lr", C.c_float), ("beta1", C.c_float), ("beta2", C.c_float), ("eps", C.c_float), ("step", C.c_int32), ("inv_grad_scale", C.c_float),
                ("flags", C.c_int32), ("deferred", C.c_int32)]


_P = C.c_void_p
_I64 = C.c_int64
_I32 = C.c_int32
_F = C.c_float

# name -> (restype, argtypes); mirrors include/cropnerf_b200.h one to one (checked by tests/test_abi.py)
SIGNATURES = {
    "cnb_version": (C.c_int, []),
    "cnb_last_error": (C.c_char_p, []),
    "cnb_device_count": (C.c_int, []),
    "cnb_hashgrid_fwd": (C.c_int, [C.POINTER(Grid), _P, _I64, _P, _P, _P]),
    "cnb_hashgrid_bwd": (C.c_int, [C.POINTER(Grid), _P, _P, _I64, _P]),
    "cnb_mlp_hidden_floats": (_I64, [C.POINTER(Mlp)]),
    "cnb_mlp_fwd": (C.c_int, [C.POINTER(Mlp), _P, _I64, _I64, _P, _P, _P]),
    "cnb_mlp_bwd": (C.c_int, [C.POINTER(Mlp), _P, _I64, _P, _P, _P, _I64, _P, _I64, _P]),
    "cnb_mlp_mixed_scratch_floats": (_I64, [C.POINTER(Mlp), _I64, _I32]),
    "cnb_mlp_mixed_fwd": (C.c_int, [C.POINTER(Mlp), _P, _I64, _I64, _P, _P, _I32, _P]),
    "cnb_mlp_mixed_bwd": (C.c_int, [C.POINTER(Mlp), _P, _I64, _P, _P, _I64, _P, _I64, _P, _P]),
    "cnb_density_field_fwd": (C.c_int, [C.POINTER(DensityField), C.POINTER(Samples), _P, _P, _P]),
    "cnb_density_field_bwd": (C.c_int, [C.POINTER(DensityField), C.POINTER(Samples), _P, _P]),
    "cnb_field_ctx_floats": (_I64, [C.POINTER(Field), _I64, _I32]),
    "cnb_field_fwd": (C.c_int, [C.POINTER(Field), C.POINTER(Samples), _P, _P, _P, _P, _P, _P, _I32, _P]),
    "cnb_field_bwd": (C.c_int, [C.POINTER(Field), C.POINTER(Samples), _P, _P, _P, _P, _P, _P]),
    "cnb_density_field_fwd_keep": (C.c_int, [C.POINTER(DensityField), C.POINTER(Samples), _P, _P, _P]),
    "cnb_density_field_bwd_kept": (C.c_int, [C.POINTER(DensityField), C.POINTER(Samples), _P, _P, _P]),
    "cnb_density_field_kept_supported": (C.c_int, [C.POINTER(DensityField)]),
    "cnb_position_grad_rays": (C.c_int, [C.POINTER(Grid), C.POINTER(Warp), C.POINTER(Samples), _P, _P, _P, _P]),
    "cnb_density_field_bwd_rays": (C.c_int, [C.POINTER(DensityField), C.POINTER(Samples), _P, _P, _P, _P, _P]),
    "cnb_field_bwd_rays": (C.c_int, [C.POINTER(Field), C.POINTER(Samples), _P, _P, _P, _P, _P, _P, _P, _P]),
    "cnb_generate_rays": (C.c_int, [C.POINTER(Camera), _P, _I64, C.POINTER(_F), _P, _P, _P, _P, _P, _P, _P]),
    "cnb_camera_opt_apply": (C.c_int, [_P, _P, _P, _P, _I64, _I32, _P, _P, _P]),
    "cnb_camera_opt_bwd": (C.c_int, [_P, _P, _P, _P, _P, _I64, _I32, _F, _F, _F, _P, _P, _P, _P]),
    "cnb_extract_points_scratch_ints": (_I64, [_I64]),
    "cnb_extract_points": (C.c_int, [_P, _P, _P, _P, _P, _I64, C.POINTER(_F), C.c_int32, _F, _P, _P, _P, _I64, _P, _P, _P, _P]),
    "cnb_generate_rays_boxes": (C.c_int, [C.POINTER(Camera), _P, C.c_int32, _I64, _P, _P, _P, _P, _P, _P, _P, _P]),
    "cnb_projection_scatter": (C.c_int, [_P, _P, _P, _I64, _F, _P, _P, _P]),
    "cnb_volume_face_rays": (C.c_int, [_F, _F, C.c_int32, _F, _F, C.c_int32, _F, C.POINTER(_F), _F, _I64, _I64, _P, _P, _P, _P, _P]),
    "cnb_sample_train_batch": (C.c_int, [C.POINTER(ImageSet), _P, _I64, _P, _P, _P, _P, _P, _P, _P, _P]),
    "cnb_sample_spaced": (C.c_int, [_P, _P, _P, _P, _I32, _I32, _I64, _I32, _P, _P, _P]),
    "cnb_sample_spaced_collide": (C.c_int, [_P, _P, _F, _F, _P, _P, _I32, _I32, _I64, _I32, _P, _P, _P, _P, _P]),
    "cnb_sample_pdf": (C.c_int, [_P, _F, _P, _P, _P, _I32, _P, _P, _I32, _I64, _I32, _I32, _F, _F, _P, _P, _P, _P]),
    "cnb_weights_fwd": (C.c_int, [_P, _P, _P, _I64, _I64, _I32, _P, _P]),
    "cnb_weights_bwd": (C.c_int, [_P, _P, _P, _I64, _I64, _I32, _P, _P, _P]),
    "cnb_render_fwd": (C.c_int, [_P, _P, _P, _P, _P, _I64, _I64, _I32, _I32, C.POINTER(_F), _I32, _P, _P, _P, _P, _P, _P]),
    "cnb_render_bwd": (C.c_int, [_P, _P, _P, _I64, _I32, _I32, C.POINTER(_F), _P, _P, _P, _I32, _P, _P, _P, _P]),
    "cnb_interlevel_fwd": (C.c_int, [_P, _P, _P, _P, _I64, _I32, _I32, _P, _P]),
    "cnb_interlevel_bwd": (C.c_int, [_P, _P, _P, _P, _I64, _I32, _I32, _F, _P, _P]),
    "cnb_distortion_fwd": (C.c_int, [_P, _P, _I64, _I32, _P, _P]),
    "cnb_pixel_losses": (C.c_int, [_P, _P, _P, _P, _I64, _F, _F, _P, _P, _P, _P]),
    "cnb_adam_step": (C.c_int, [_P, _P, _P, _P, _I64, _F, _F, _F, _F, _I32, _F, _P]),
    "cnb_adam_step_zero": (C.c_int, [_P, _P, _P, _P, _I64, _F, _F, _F, _F, _I32, _F, _P]),
    "cnb_adam_step_zero_guarded": (C.c_int, [_P, _P, _P, _P, _I64, _F, _F, _F, _F, _I32, _F, _P, _P]),
    "cnb_grad_check_finite": (C.c_int, [_P, _I64, _P, _P]),
    "cnb_hashgrid_mark_reachable": (C.c_int, [C.POINTER(Grid), _P, _I64, _P]),
    "cnb_bitmap_mark_range": (C.c_int, [_P, _I64, _I64, _P]),
    "cnb_adam_step_zero_live": (C.c_int, [_P, _P, _P, _P, _I64, _F, _F, _F, _F, _I32, _F, _P, _P]),
    "cnb_adam_step_zero_dev_live": (C.c_int, [_P, _P, _P, _P, _I64, _P, _P, _P]),
    "cnb_upload": (C.c_int, [C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.POINTER(C.c_int64), _I32, _P]),
    "cnb_stage_inputs": (C.c_int, [C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.POINTER(C.c_int64), _I32, _P, C.POINTER(_F), _I32, _P]),
    "cnb_adam_step_zero_dev": (C.c_int, [_P, _P, _P, _P, _I64, _P, _P]),
    "cnb_p2p_owned_range": (None, [_I64, _I32, _I32, C.POINTER(_I64), C.POINTER(_I64)]),
    "cnb_p2p_barrier": (C.c_int, [C.POINTER(P2PComm), _P]),
    "cnb_ddp_exchange_dev": (C.c_int, [C.POINTER(P2PComm), C.POINTER(P2PGroup), _P, _P, _P, _I64, _P, _I32, _I32, _P]),
    "cnb_ddp_optimizer_step": (C.c_int, [C.POINTER(P2PComm), C.POINTER(DdpGroupStep), _I32, _P]),
    "cnb_ddp_wait_deferred": (C.c_int, [_P]),
    "cnb_ddp_adam_update": (C.c_int, [C.POINTER(P2PComm), C.POINTER(P2PGroup), _P, _P, _I64, _F, _F, _F, _F, _I32, _F, _I32, _P]),
    "cnb_level_resample": (C.c_int, [_P, _P, _P, _P, _P, _I32, _F, _P, _P, _I32, _I64, _I32, _I32, _F, _F, _P, _P, _P, _P, _P, _P]),
    "cnb_final_composite": (C.c_int, [_P, _P, _P, _P, _I64, _I32, _I32, C.POINTER(_F), _I32, _P, _P, _P, _P, _P, _P]),
    "cnb_final_composite_bwd": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, _P, _P, _I64, _I32, _I32, C.POINTER(_F), _F, _F, _I32, _P, _P, _P, _P, _P]),
    "cnb_interlevel_fused": (C.c_int, [_P, _P, _P, _P, _P, _P, _I64, _I32, _I32, _F, _P, _P, _P]),
    "cnb_profile_enable": (None, [_I32]),
    "cnb_profile_read": (C.c_int, [C.c_char_p, _I32]),
    "cnb_render_workspace_floats": (_I64, [C.POINTER(Model), _I64, _I32]),
    "cnb_render_rays": (C.c_int, [C.POINTER(Model), C.POINTER(Rays), C.POINTER(RayOutputs), _P, _P]),
    "cnb_train_step": (C.c_int, [C.POINTER(Model), C.POINTER(Rays), C.POINTER(TrainCfg), C.POINTER(RayOutputs), _P, _P, _P]),
}

_lib: Optional["_Proxy"] = None

# kernels launched per C-ABI call (fp32 field path is a chain of kernels; see csrc/field_fp32.cu)
KERNELS_PER_CALL = {
    "cnb_hashgrid_fwd": 1, "cnb_hashgrid_bwd": 1, "cnb_mlp_fwd": 1, "cnb_mlp_bwd": 1, "cnb_density_field_fwd": 1, "cnb_density_field_bwd": 1,
    "cnb_field_fwd": 7, "cnb_field_bwd": 8, "cnb_sample_spaced": 1, "cnb_sample_pdf": 1, "cnb_weights_fwd": 1, "cnb_weights_bwd": 1,
    "cnb_render_fwd": 1, "cnb_render_bwd": 1, "cnb_interlevel_fwd": 1, "cnb_interlevel_bwd": 1, "cnb_distortion_fwd": 1, "cnb_pixel_losses": 1,
    "cnb_adam_step": 1,
}


class Profile:
    """Optional per-call instrumentation: counts every C-ABI call and, when ``timing`` is set, brackets it with CUDA
    events recorded on the launching (current) stream."""

    def __init__(self, timing: bool = False):
        self.timing = timing
        self.calls = {}
        self.events = {}

    def launches(self) -> int:
        return sum(n * KERNELS_PER_CALL.get(k, 1) for k, n in self.calls.items())

    def times_ms(self) -> dict:
        torch.cuda.synchronize()
        return {k: [a.elapsed_time(b) for a, b in v] for k, v in self.events.items()}


_profile: Optional[Profile] = None


def set_profile(p: Optional[Profile]) -> None:
    global _profile
    _profile = p


class _Proxy:
    """Attribute access returns the ctypes function wrapped with the optional profiler."""

    def __init__(self, handle: C.CDLL):
        self._h = handle
        self._cache = {}

    def __getattr__(self, name):
        c = self.__dict__["_cache"]
        if name in c:
            return c[name]
        fn = getattr(self.__dict__["_h"], name)

        def wrapped(*args, _fn=fn, _name=name):
            prof = _profile
            if prof is None:
                return _fn(*args)
            prof.calls[_name] = prof.calls.get(_name, 0) + 1
            if not prof.timing:
                return _fn(*args)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            rc = _fn(*args)
            e1.record()
            prof.events.setdefault(_name, []).append((e0, e1))
            return rc

        c[name] = wrapped
        return wrapped


def build(verbose: bool = False) -> str:
    """Compile the CUDA sources in-tree for sm_100a (``csrc/Makefile``) and return the library path."""
    res = subprocess.run(["make", "-C", CSRC, "-j", str(os.cpu_count() or 4)], capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("building libcropnerf_b200.so failed:\n" + res.stdout[-4000:] + res.stderr[-4000:])
    if verbose:
        print(res.stdout[-2000:])
    return LIB_PATH


def lib() -> "_Proxy":
    """Load (once) the shared library; fail loudly if it has not been built -- there is no fallback."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(or `make -C cropnerf-a-neural-radiance-field-based-framework_b200/csrc`). "
                "cropnerf_b200 has no CPU / PyTorch fallback for its kernels."
            )
        handle = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(handle, name)
            fn.restype = res
            fn.argtypes = args
        _lib = _Proxy(handle)
    return _lib


def last_error() -> str:
    return lib().cnb_last_error().decode("utf-8", "replace")


def check(rc: int, what: str) -> None:
    if rc != 0:
        raise RuntimeError(f"cropnerf_b200: {what} failed (status {rc}): {last_error()}")


def stream_ptr(device=None) -> int:
    return torch.cuda.current_stream(device).cuda_stream


def ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    """Device pointer of a contiguous CUDA tensor (None passes NULL)."""
    if t is None:
        return None
    if not t.is_cuda:
        raise RuntimeError("cropnerf_b200 kernels need CUDA tensors; there is no CPU fallback")
    if not t.is_contiguous():
        raise RuntimeError("cropnerf_b200: tensor must be contiguous")
    return t.data_ptr()


def f32(t: torch.Tensor) -> torch.Tensor:
    if t.dtype != torch.float32:
        t = t.float()
    return t.contiguous()


def make_grid(table: torch.Tensor, d_table: Optional[torch.Tensor], num_levels: int, log2_hashmap_size: int, scalings: Sequence[float]) -> Grid:
    g = Grid()
    g.table = ptr(table)
    g.d_table = ptr(d_table)
    g.num_levels = int(num_levels)
    g.log2_hashmap_size = int(log2_hashmap_size)
    for i in range(MAX_LEVELS):
        g.scalings[i] = float(scalings[i]) if i < len(scalings) else 0.0
    return g


def make_mlp(weights: Sequence[torch.Tensor], biases: Sequence[torch.Tensor], out_activation: int,
             d_weights: Optional[Sequence[Optional[torch.Tensor]]] = None, d_biases: Optional[Sequence[Optional[torch.Tensor]]] = None) -> Mlp:
    m = Mlp()
    n = len(weights)
    if not 1 <= n <= MAX_LAYERS:
        raise ValueError(f"MLP with {n} layers unsupported (1..{MAX_LAYERS})")
    m.num_layers = n
    m.out_activation = out_activation
    m.dims[0] = weights[0].shape[1]
    for i, (w, b) in enumerate(zip(weights, biases)):
        if w.shape[0] > WIDE_MAX_WIDTH or w.shape[1] > WIDE_MAX_WIDTH:
            raise ValueError(f"MLP layer {i} of shape {tuple(w.shape)} exceeds the compiled maximum width {WIDE_MAX_WIDTH}")
        m.dims[i + 1] = w.shape[0]
        m.W[i] = ptr(w)
        m.b[i] = ptr(b)
        m.dW[i] = ptr(d_weights[i]) if d_weights is not None else None
        m.db[i] = ptr(d_biases[i]) if d_biases is not None else None
    return m


def make_warp(contraction: bool, aabb) -> Warp:
    """``aabb``: host-side nested list [[xmin,ymin,zmin],[xmax,ymax,zmax]] (no device sync on the call path)."""
    w = Warp()
    w.mode = WARP_CONTRACT_LINF if contraction else WARP_AABB
    box = [[-1.0, -1.0, -1.0], [1.0, 1.0, 1.0]] if aabb is None else (aabb.detach().cpu().tolist() if isinstance(aabb, torch.Tensor) else aabb)
    for i in range(3):
        w.aabb_min[i] = box[0][i]
        w.aabb_max[i] = box[1][i]
    return w


def stage_profile_read() -> dict:
    """{stage: {"calls", "kernels", "ms"}} recorded by the fused pipeline since ``cnb_profile_enable(1)`` (synchronises)."""
    buf = C.create_string_buffer(8192)
    check(lib().cnb_profile_read(buf, 8192), "profile_read")
    out = {}
    for item in buf.value.decode().split(";"):
        if item:
            name, calls, kernels, ms = item.split(":")
            out[name] = {"calls": int(calls), "kernels": int(kernels), "ms": float(ms)}
    return out
