"""Operator layer: thin wrappers + ``torch.autograd.Function``s over the C ABI (``include/cropnerf_b200.h``).

Every function here enqueues hand-written sm_100a kernels on torch's current CUDA stream through ctypes; torch is
used for memory, streams and autograd bookkeeping only.  There is no CPU / eager fallback: CPU tensors raise.
"""
from __future__ import annotations

import ctypes as C
from typing import List, Optional, Sequence, Tuple

import torch
from torch import Tensor

from . import _lib as L


def _dev(t: Tensor) -> torch.device:
    if not t.is_cuda:
        raise RuntimeError("cropnerf_b200 ops need CUDA tensors; there is no CPU fallback")
    return t.device


def _p(t: Optional[Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def make_samples(origins: Tensor, directions: Tensor, starts: Tensor, ends: Tensor, cam: Optional[Tensor], R: int, S: int, row_stride: int) -> L.Samples:
    s = L.Samples()
    s.origins = origins.data_ptr()
    s.directions = directions.data_ptr()
    s.starts = starts.data_ptr()
    s.ends = ends.data_ptr()
    s.camera_indices = _p(cam)
    s.num_rays = R
    s.row_stride = row_stride
    s.samples_per_ray = S
    return s


# ---------------------------------------------------------------------------------------------------------
# a2: hash grid
# ---------------------------------------------------------------------------------------------------------


class _HashGridFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, positions: Tensor, table: Tensor, num_levels: int, log2_hashmap_size: int, scalings: Tuple[float, ...]):
        _dev(positions)
        pos = L.f32(positions.detach()).reshape(-1, 3)
        tab = table.detach()
        n = pos.shape[0]
        out = torch.empty((n, 2 * num_levels), device=pos.device, dtype=torch.float32)
        g = L.make_grid(tab, None, num_levels, log2_hashmap_size, scalings)
        L.check(L.lib().cnb_hashgrid_fwd(C.byref(g), pos.data_ptr(), n, out.data_ptr(), None, L.stream_ptr(pos.device)), "hashgrid_fwd")
        ctx.save_for_backward(pos, tab)
        ctx.cfg = (num_levels, log2_hashmap_size, scalings)
        return out.view(*positions.shape[:-1], 2 * num_levels)

    @staticmethod
    def backward(ctx, d_out: Tensor):
        pos, tab = ctx.saved_tensors
        num_levels, log2_hashmap_size, scalings = ctx.cfg
        d_table = torch.zeros_like(tab)
        d = L.f32(d_out).reshape(-1, 2 * num_levels)
        g = L.make_grid(tab, d_table, num_levels, log2_hashmap_size, scalings)
        L.check(L.lib().cnb_hashgrid_bwd(C.byref(g), pos.data_ptr(), d.data_ptr(), pos.shape[0], L.stream_ptr(pos.device)), "hashgrid_bwd")
        # positions receive no gradient: the camera-optimizer path (SURVEY.md a17) is a "next" row
        return None, d_table, None, None, None


def hashgrid_encode(positions: Tensor, table: Tensor, num_levels: int, log2_hashmap_size: int, scalings: Sequence[float]) -> Tensor:
    return _HashGridFn.apply(positions, table, num_levels, log2_hashmap_size, tuple(float(s) for s in scalings))


def hashgrid_indices(positions: Tensor, table: Tensor, num_levels: int, log2_hashmap_size: int, scalings: Sequence[float]) -> Tuple[Tensor, Tensor]:
    """Features and the [n, L, 8] int32 table rows (h0..h7 order) -- for bit-exactness tests."""
    pos = L.f32(positions.detach()).reshape(-1, 3)
    n = pos.shape[0]
    out = torch.empty((n, 2 * num_levels), device=pos.device, dtype=torch.float32)
    idx = torch.empty((n, num_levels, 8), device=pos.device, dtype=torch.int32)
    g = L.make_grid(table.detach(), None, num_levels, log2_hashmap_size, scalings)
    L.check(L.lib().cnb_hashgrid_fwd(C.byref(g), pos.data_ptr(), n, out.data_ptr(), idx.data_ptr(), L.stream_ptr(pos.device)), "hashgrid_fwd")
    return out, idx


# ---------------------------------------------------------------------------------------------------------
# a3/a4: MLP
# ---------------------------------------------------------------------------------------------------------


class _MLPFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x: Tensor, out_activation: int, *params: Tensor):
        _dev(x)
        nl = len(params) // 2
        ws = [p.detach() for p in params[:nl]]
        bs = [p.detach() for p in params[nl:]]
        x2 = L.f32(x.detach()).reshape(-1, x.shape[-1])
        n = x2.shape[0]
        out_dim = ws[-1].shape[0]
        y = torch.empty((n, out_dim), device=x2.device, dtype=torch.float32)
        m = L.make_mlp(ws, bs, out_activation)
        need_grad = any(ctx.needs_input_grad)
        hidden = None
        if need_grad and nl > 1:
            hidden = torch.empty((n * sum(w.shape[0] for w in ws[:-1]),), device=x2.device, dtype=torch.float32)
        L.check(L.lib().cnb_mlp_fwd(C.byref(m), x2.data_ptr(), x2.stride(0), n, y.data_ptr(), _p(hidden), L.stream_ptr(x2.device)), "mlp_fwd")
        ctx.save_for_backward(x2, y, hidden if hidden is not None else torch.empty(0, device=x2.device), *ws, *bs)
        ctx.nl = nl
        ctx.act = out_activation
        ctx.x_shape = x.shape
        return y.view(*x.shape[:-1], out_dim)

    @staticmethod
    def backward(ctx, dy: Tensor):
        saved = ctx.saved_tensors
        x2, y, hidden = saved[0], saved[1], saved[2]
        nl = ctx.nl
        ws, bs = list(saved[3 : 3 + nl]), list(saved[3 + nl : 3 + 2 * nl])
        dws = [torch.zeros_like(w) for w in ws]
        dbs = [torch.zeros_like(b) for b in bs]
        n = x2.shape[0]
        d = L.f32(dy).reshape(n, -1)
        dx = torch.empty_like(x2) if ctx.needs_input_grad[0] else None
        m = L.make_mlp(ws, bs, ctx.act, dws, dbs)
        L.check(
            L.lib().cnb_mlp_bwd(
                C.byref(m), x2.data_ptr(), x2.stride(0), _p(hidden) if nl > 1 else None, y.data_ptr(), d.data_ptr(), n,
                _p(dx), x2.stride(0), L.stream_ptr(x2.device),
            ),
            "mlp_bwd",
        )
        return (dx.view(ctx.x_shape) if dx is not None else None, None, *dws, *dbs)


def mlp_forward(x: Tensor, weights: Sequence[Tensor], biases: Sequence[Tensor], out_activation: int = L.ACT_NONE) -> Tensor:
    return _MLPFn.apply(x, out_activation, *weights, *biases)


# ---------------------------------------------------------------------------------------------------------
# a7: fused proposal density field
# ---------------------------------------------------------------------------------------------------------


class _DensityFieldFn(torch.autograd.Function):
    """(table, W1, b1, W2, b2) -> density [R*S].  ``cfg`` = (sample layout tuple, grid cfg, warp, avg)."""

    @staticmethod
    def forward(ctx, cfg, origins_t: Tensor, directions_t: Tensor, table: Tensor, W1: Tensor, b1: Tensor, W2: Tensor, b2: Tensor):
        (origins, directions, starts, ends, R, S, row_stride), (num_levels, log2_T, scalings), warp, avg, want_pos = cfg[:5]
        origins, directions = origins.detach(), directions.detach()
        dev = _dev(origins)
        density = torch.empty((R * S,), device=dev, dtype=torch.float32)
        pos_out = torch.empty((R * S, 3), device=dev, dtype=torch.float32) if want_pos else None
        f = L.DensityField()
        f.grid = L.make_grid(table.detach(), None, num_levels, log2_T, scalings)
        f.mlp = L.make_mlp([W1.detach(), W2.detach()], [b1.detach(), b2.detach()], L.ACT_NONE)
        f.warp = warp
        f.average_init_density = avg
        sm = make_samples(origins, directions, starts, ends, None, R, S, row_stride)
        L.check(L.lib().cnb_density_field_fwd(C.byref(f), C.byref(sm), density.data_ptr(), _p(pos_out), L.stream_ptr(dev)), "density_field_fwd")
        ctx.cfg = cfg
        ctx.rays_grad = ctx.needs_input_grad[1] or ctx.needs_input_grad[2]
        ctx.save_for_backward(table, W1, b1, W2, b2)
        ctx.mark_non_differentiable(*( [pos_out] if pos_out is not None else [] ))
        if want_pos:
            return density, pos_out
        return density

    @staticmethod
    def backward(ctx, d_density: Tensor, *unused):
        table, W1, b1, W2, b2 = ctx.saved_tensors
        (origins, directions, starts, ends, R, S, row_stride), (num_levels, log2_T, scalings), warp, avg, _ = ctx.cfg[:5]
        precision = ctx.cfg[5] if len(ctx.cfg) > 5 else L.PREC_FP32  # mixed: plain-bf16 operands in the MLP parameter-gradient contraction
        origins, directions = origins.detach(), directions.detach()
        dev = origins.device
        d_table = torch.zeros_like(table)
        dW1, db1, dW2, db2 = (torch.zeros_like(t) for t in (W1, b1, W2, b2))
        f = L.DensityField()
        f.grid = L.make_grid(table.detach(), d_table, num_levels, log2_T, scalings)
        f.mlp = L.make_mlp([W1.detach(), W2.detach()], [b1.detach(), b2.detach()], L.ACT_NONE, [dW1, dW2], [db1, db2])
        f.warp = warp
        f.average_init_density = avg
        f.precision = precision
        sm = make_samples(origins, directions, starts, ends, None, R, S, row_stride)
        d = L.f32(d_density).reshape(-1)
        d_o = d_d = None
        if ctx.rays_grad:  # row a17: the camera optimizer differentiates through the ray origins / directions
            d_o, d_d = torch.zeros_like(origins), torch.zeros_like(directions)
            scratch = torch.empty((R * S * 2 * num_levels,), device=dev, dtype=torch.float32)
            L.check(L.lib().cnb_density_field_bwd_rays(C.byref(f), C.byref(sm), d.data_ptr(), scratch.data_ptr(), d_o.data_ptr(), d_d.data_ptr(),
                                                       L.stream_ptr(dev)), "density_field_bwd_rays")
        else:
            L.check(L.lib().cnb_density_field_bwd(C.byref(f), C.byref(sm), d.data_ptr(), L.stream_ptr(dev)), "density_field_bwd")
        return None, d_o, d_d, d_table, dW1, db1, dW2, db2


def density_field(cfg, table, W1, b1, W2, b2):
    return _DensityFieldFn.apply(cfg, cfg[0][0], cfg[0][1], table, W1, b1, W2, b2)


# ---------------------------------------------------------------------------------------------------------
# a1/a5/a6: fused FruitField
# ---------------------------------------------------------------------------------------------------------

FIELD_PARAM_ORDER = ("table", "base_W", "base_b", "sem_W", "sem_b", "head_W", "head_b", "rgb_W", "rgb_b", "embedding")


def _build_field(cfg: dict, params: Sequence[Tensor], grads: Optional[Sequence[Optional[Tensor]]]) -> Tuple[L.Field, list]:
    """params: flat list [table, *base_W, *base_b, *sem_W, *sem_b, head_W, head_b, *rgb_W, *rgb_b, embedding]."""
    nb, ns, nr = cfg["nl_base"], cfg["nl_sem"], cfg["nl_rgb"]
    it = iter(range(len(params)))
    take = lambda k: [next(it) for _ in range(k)]  # noqa: E731
    i_table = take(1)[0]
    i_bw, i_bb = take(nb), take(nb)
    i_sw, i_sb = take(ns), take(ns)
    i_hw, i_hb = take(1), take(1)
    i_rw, i_rb = take(nr), take(nr)
    i_emb = take(1)[0]
    P = [p.detach() for p in params]
    G = list(grads) if grads is not None else [None] * len(params)
    sel = lambda idx, src: [src[i] for i in idx]  # noqa: E731
    f = L.Field()
    f.grid = L.make_grid(P[i_table], G[i_table], cfg["num_levels"], cfg["log2_hashmap_size"], cfg["scalings"])
    gr = grads is not None
    f.base = L.make_mlp(sel(i_bw, P), sel(i_bb, P), L.ACT_NONE, sel(i_bw, G) if gr else None, sel(i_bb, G) if gr else None)
    f.sem = L.make_mlp(sel(i_sw, P), sel(i_sb, P), L.ACT_NONE, sel(i_sw, G) if gr else None, sel(i_sb, G) if gr else None)
    f.sem_head = L.make_mlp(sel(i_hw, P), sel(i_hb, P), L.ACT_NONE, sel(i_hw, G) if gr else None, sel(i_hb, G) if gr else None)
    f.rgb = L.make_mlp(sel(i_rw, P), sel(i_rb, P), L.ACT_SIGMOID, sel(i_rw, G) if gr else None, sel(i_rb, G) if gr else None)
    f.embedding = P[i_emb].data_ptr()
    f.d_embedding = _p(G[i_emb])
    keep = []
    if cfg["appearance_mode"] == L.APP_MEAN:
        mean = P[i_emb].mean(dim=0).contiguous()
        keep.append(mean)
        f.mean_embedding = mean.data_ptr()
    f.warp = cfg["warp"]
    f.num_images = P[i_emb].shape[0]
    f.appearance_dim = P[i_emb].shape[1]
    f.geo_feat_dim = cfg["geo_feat_dim"]
    f.appearance_mode = cfg["appearance_mode"]
    f.pass_semantic_gradients = int(cfg["pass_semantic_gradients"])
    f.precision = cfg["precision"]
    return f, keep


class _FieldFn(torch.autograd.Function):
    """FruitField.forward on one launch chain: -> (density [N], rgb [N,3], sem [N], geo [N,1+geo], positions [N,3])."""

    @staticmethod
    def forward(ctx, cfg: dict, layout, origins_t: Tensor, directions_t: Tensor, *params: Tensor):
        origins, directions, starts, ends, cam, R, S, row_stride = layout
        origins, directions = origins.detach(), directions.detach()
        layout = (origins, directions, starts, ends, cam, R, S, row_stride)
        dev = _dev(origins)
        N = R * S
        training = bool(cfg["training"]) and any(ctx.needs_input_grad)
        ctx.rays_grad = ctx.needs_input_grad[2] or ctx.needs_input_grad[3]
        f, keep = _build_field(cfg, params, None)
        sm = make_samples(origins, directions, starts, ends, cam, R, S, row_stride)
        lib = L.lib()
        ctx_floats = lib.cnb_field_ctx_floats(C.byref(f), N, int(training))
        scratch = torch.empty((max(int(ctx_floats), 1),), device=dev, dtype=torch.float32)
        density = torch.empty((N,), device=dev, dtype=torch.float32)
        rgb = torch.empty((N, 3), device=dev, dtype=torch.float32)
        sem = torch.empty((N,), device=dev, dtype=torch.float32)
        # fp32: always (its gradient is accepted); mixed: only for the get_density / get_outputs split, as a non-differentiable output
        want_geo = cfg["precision"] == L.PREC_FP32 or bool(cfg.get("want_geo", False))
        geo = torch.empty((N, 1 + cfg["geo_feat_dim"]), device=dev, dtype=torch.float32) if want_geo else None
        pos = torch.empty((N, 3), device=dev, dtype=torch.float32) if cfg.get("want_positions", True) else None
        L.check(
            lib.cnb_field_fwd_half(C.byref(f), _p(cfg.get("table_half")), C.byref(sm), density.data_ptr(), _p(geo), rgb.data_ptr(), sem.data_ptr(),
                                   _p(pos), scratch.data_ptr() if ctx_floats > 0 else None, int(training), L.stream_ptr(dev)),
            "field_fwd",
        )
        ctx.cfg, ctx.layout, ctx.training = cfg, layout, training
        ctx.scratch = scratch if training else None
        ctx.save_for_backward(*params)
        outs = [density, rgb, sem, geo if geo is not None else torch.empty(0, device=dev), pos if pos is not None else torch.empty(0, device=dev)]
        ctx.mark_non_differentiable(outs[4])
        if cfg["precision"] != L.PREC_FP32:
            ctx.mark_non_differentiable(outs[3])
        return tuple(outs)

    @staticmethod
    def backward(ctx, d_density, d_rgb, d_sem, d_geo, _d_pos):
        if not ctx.training:
            raise RuntimeError("cropnerf_b200: field backward requested but forward ran in inference mode")
        params = ctx.saved_tensors
        cfg = ctx.cfg
        origins, directions, starts, ends, cam, R, S, row_stride = ctx.layout
        dev = origins.device
        grads: List[Optional[Tensor]] = [torch.zeros_like(p) if p.requires_grad else None for p in params]
        # the kernels accumulate into every buffer they are given; frozen parameters simply get none
        grads_full = [g if g is not None else torch.zeros_like(p) for g, p in zip(grads, params)]
        f, keep = _build_field(cfg, params, grads_full)
        sm = make_samples(origins, directions, starts, ends, cam, R, S, row_stride)
        dd = L.f32(d_density).reshape(-1) if d_density is not None else None
        dr = L.f32(d_rgb).reshape(-1, 3) if d_rgb is not None else None
        ds = L.f32(d_sem).reshape(-1) if d_sem is not None else None
        dg = None
        if d_geo is not None and d_geo.numel() > 0 and cfg["precision"] == L.PREC_FP32:
            dg = L.f32(d_geo).reshape(-1, 1 + cfg["geo_feat_dim"])
        scratch_ptr = ctx.scratch.data_ptr() if ctx.scratch is not None and ctx.scratch.numel() > 1 else None
        d_o = d_d = None
        if ctx.rays_grad:  # row a17: gradient with respect to the rays (camera optimizer)
            d_o, d_d = torch.zeros_like(origins), torch.zeros_like(directions)
            L.check(L.lib().cnb_field_bwd_rays_half(C.byref(f), _p(cfg.get("table_half")), C.byref(sm), _p(dd), _p(dr), _p(ds), _p(dg), scratch_ptr,
                                                    d_o.data_ptr(), d_d.data_ptr(), L.stream_ptr(dev)), "field_bwd_rays")
        else:
            L.check(L.lib().cnb_field_bwd(C.byref(f), C.byref(sm), _p(dd), _p(dr), _p(ds), _p(dg), scratch_ptr, L.stream_ptr(dev)), "field_bwd")
        # the mean-embedding gradient is not propagated (inference-only mode, fruit_field.py:219-221)
        ctx.scratch = None
        return (None, None, d_o, d_d, *grads)


def fruit_field(cfg: dict, layout, params: Sequence[Tensor]):
    return _FieldFn.apply(cfg, layout, layout[0], layout[1], *params)


# ---------------------------------------------------------------------------------------------------------
# a8/a9: samplers (no gradients: bins are detached in the reference, ray_samplers.py PDFSampler "Stop gradients")
# ---------------------------------------------------------------------------------------------------------


def sample_spaced(nears: Tensor, fars: Tensor, lin_bins: Tensor, t_rand: Optional[Tensor], spacing: int) -> Tuple[Tensor, Tensor]:
    dev = _dev(nears)
    R = nears.shape[0]
    S = lin_bins.shape[0] - 1
    nears = L.f32(nears).reshape(-1)
    fars = L.f32(fars).reshape(-1)
    sp = torch.empty((R, S + 1), device=dev, dtype=torch.float32)
    eu = torch.empty((R, S + 1), device=dev, dtype=torch.float32)
    rs = 0
    if t_rand is not None:
        t_rand = L.f32(t_rand).reshape(R, -1)
        rs = t_rand.shape[1]
    L.check(
        L.lib().cnb_sample_spaced(nears.data_ptr(), fars.data_ptr(), L.f32(lin_bins).data_ptr(), _p(t_rand), rs, spacing, R, S,
                                  sp.data_ptr(), eu.data_ptr(), L.stream_ptr(dev)),
        "sample_spaced",
    )
    return sp, eu


def sample_pdf(weights: Tensor, anneal: float, prev_spacing_bins: Tensor, nears: Tensor, fars: Tensor, spacing: int, u_base: Tensor,
               rand: Optional[Tensor], num_samples: int, histogram_padding: float = 0.01, eps: float = 1e-5,
               want_inds: bool = False) -> Tuple[Tensor, Tensor, Optional[Tensor]]:
    dev = _dev(weights)
    w = L.f32(weights.detach()).reshape(weights.shape[0], -1)
    R, Sp = w.shape
    S = num_samples
    prev = L.f32(prev_spacing_bins)
    assert prev.shape == (R, Sp + 1)
    sp = torch.empty((R, S + 1), device=dev, dtype=torch.float32)
    eu = torch.empty((R, S + 1), device=dev, dtype=torch.float32)
    inds = torch.empty((R, S + 1), device=dev, dtype=torch.int32) if want_inds else None
    rs = 0
    if rand is not None:
        rand = L.f32(rand).reshape(R, -1)
        rs = rand.shape[1]
    L.check(
        L.lib().cnb_sample_pdf(w.data_ptr(), float(anneal), prev.data_ptr(), L.f32(nears).reshape(-1).data_ptr(), L.f32(fars).reshape(-1).data_ptr(),
                               spacing, L.f32(u_base).data_ptr(), _p(rand), rs, R, Sp, S, histogram_padding, eps, sp.data_ptr(), eu.data_ptr(),
                               _p(inds), L.stream_ptr(dev)),
        "sample_pdf",
    )
    return sp, eu, inds


# ---------------------------------------------------------------------------------------------------------
# a10-a14: compositing
# ---------------------------------------------------------------------------------------------------------


def _rows(starts: Tensor, ends: Tensor) -> Tuple[Tensor, Tensor, int]:
    """[R,S,1] / [R,S] start/end tensors -> (base tensors, row stride) usable with strided addressing."""
    s = starts[..., 0] if starts.dim() == 3 else starts
    e = ends[..., 0] if ends.dim() == 3 else ends
    S = s.shape[1]
    ok = s.dtype == torch.float32 and e.dtype == torch.float32 and (S == 1 or (s.stride(1) == 1 and e.stride(1) == 1)) and s.stride(0) == e.stride(0) and s.stride(0) >= S
    if not ok:
        s, e = s.float().contiguous(), e.float().contiguous()
    return s, e, (s.stride(0) if s.shape[0] > 1 else max(S, s.stride(0)))


class _WeightsFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, density: Tensor, starts: Tensor, ends: Tensor):
        dev = _dev(density)
        s, e, stride = _rows(starts, ends)
        R, S = s.shape
        d = L.f32(density.detach()).reshape(R, S)
        w = torch.empty((R, S), device=dev, dtype=torch.float32)
        L.check(L.lib().cnb_weights_fwd(d.data_ptr(), s.data_ptr(), e.data_ptr(), stride, R, S, w.data_ptr(), L.stream_ptr(dev)), "weights_fwd")
        ctx.save_for_backward(d, s, e)
        ctx.stride = stride
        ctx.out_shape = density.shape
        return w.view(density.shape)

    @staticmethod
    def backward(ctx, d_w: Tensor):
        d, s, e = ctx.saved_tensors
        R, S = d.shape
        g = L.f32(d_w).reshape(R, S)
        dd = torch.empty_like(d)
        L.check(L.lib().cnb_weights_bwd(d.data_ptr(), s.data_ptr(), e.data_ptr(), ctx.stride, R, S, g.data_ptr(), dd.data_ptr(), L.stream_ptr(d.device)), "weights_bwd")
        return dd.view(ctx.out_shape), None, None


def ray_weights(density: Tensor, starts: Tensor, ends: Tensor) -> Tensor:
    return _WeightsFn.apply(density, starts, ends)


def _bg_args(bg_mode: int, bg_color):
    if bg_mode == L.BG_CONSTANT:
        arr = (C.c_float * 3)(*[float(v) for v in bg_color])
        return arr
    return None


class _RenderFn(torch.autograd.Function):
    """(weights, rgb, sem) -> (rgb_out [R,3], acc [R,1], sem_out [R,1]); any of rgb/sem may be None."""

    @staticmethod
    def forward(ctx, weights: Tensor, rgb: Optional[Tensor], sem: Optional[Tensor], bg_mode: int, bg_color, eval_mode: bool):
        dev = _dev(weights)
        R, S = weights.shape[0], weights.shape[1]
        w = L.f32(weights.detach()).reshape(R, S)
        c = L.f32(rgb.detach()).reshape(R, S, 3) if rgb is not None else None
        sm = L.f32(sem.detach()).reshape(R, S) if sem is not None else None
        rgb_out = torch.empty((R, 3), device=dev, dtype=torch.float32) if c is not None else None
        acc = torch.empty((R, 1), device=dev, dtype=torch.float32)
        sem_out = torch.empty((R, 1), device=dev, dtype=torch.float32) if sm is not None else None
        L.check(
            L.lib().cnb_render_fwd(w.data_ptr(), _p(c), _p(sm), None, None, S, R, S, bg_mode, _bg_args(bg_mode, bg_color), int(eval_mode),
                                   _p(rgb_out), None, acc.data_ptr(), _p(sem_out), None, L.stream_ptr(dev)),
            "render_fwd",
        )
        ctx.save_for_backward(w, c if c is not None else torch.empty(0, device=dev), sm if sm is not None else torch.empty(0, device=dev))
        ctx.cfg = (bg_mode, bg_color, c is not None, sm is not None, weights.shape, None if rgb is None else rgb.shape, None if sem is None else sem.shape)
        empty = torch.empty(0, device=dev)
        return (rgb_out if rgb_out is not None else empty, acc, sem_out if sem_out is not None else empty)

    @staticmethod
    def backward(ctx, d_rgb_out, d_acc, d_sem_out):
        w, c, sm = ctx.saved_tensors
        bg_mode, bg_color, has_rgb, has_sem, w_shape, rgb_shape, sem_shape = ctx.cfg
        R, S = w.shape
        dev = w.device
        need_w, need_rgb, need_sem = ctx.needs_input_grad[0], ctx.needs_input_grad[1] and has_rgb, ctx.needs_input_grad[2] and has_sem
        d_w = torch.empty_like(w) if need_w else None
        d_c = torch.empty((R, S, 3), device=dev, dtype=torch.float32) if need_rgb else None
        d_s = torch.empty((R, S), device=dev, dtype=torch.float32) if need_sem else None
        g_rgb = L.f32(d_rgb_out).reshape(R, 3) if has_rgb and d_rgb_out is not None and d_rgb_out.numel() else None
        g_acc = L.f32(d_acc).reshape(R) if d_acc is not None else None
        g_sem = L.f32(d_sem_out).reshape(R) if has_sem and d_sem_out is not None and d_sem_out.numel() else None
        L.check(
            L.lib().cnb_render_bwd(w.data_ptr(), c.data_ptr() if has_rgb else None, sm.data_ptr() if has_sem else None, R, S, bg_mode,
                                   _bg_args(bg_mode, bg_color), _p(g_rgb), _p(g_acc), _p(g_sem), 1, _p(d_w), _p(d_c), _p(d_s), L.stream_ptr(dev)),
            "render_bwd",
        )
        return (d_w.view(w_shape) if d_w is not None else None, d_c.view(rgb_shape) if d_c is not None else None,
                d_s.view(sem_shape) if d_s is not None else None, None, None, None)


def render(weights: Tensor, rgb: Optional[Tensor], sem: Optional[Tensor], bg_mode: int, bg_color=None, eval_mode: bool = False):
    return _RenderFn.apply(weights, rgb, sem, bg_mode, bg_color, eval_mode)


def render_median_depth(weights: Tensor, starts: Tensor, ends: Tensor, want_index: bool = False):
    """DepthRenderer(method="median") -- no gradient (a searchsorted gather; the reference calls it under no_grad
    in training, fruit_nerf.py:561-562)."""
    dev = _dev(weights)
    s, e, stride = _rows(starts, ends)
    R, S = s.shape
    w = L.f32(weights.detach()).reshape(R, S)
    depth = torch.empty((R, 1), device=dev, dtype=torch.float32)
    idx = torch.empty((R,), device=dev, dtype=torch.int32) if want_index else None
    L.check(
        L.lib().cnb_render_fwd(w.data_ptr(), None, None, s.data_ptr(), e.data_ptr(), stride, R, S, L.BG_NONE, None, 0, None, depth.data_ptr(), None, None,
                               _p(idx), L.stream_ptr(dev)),
        "render_fwd(depth)",
    )
    return (depth, idx) if want_index else depth


# ---------------------------------------------------------------------------------------------------------
# a16: losses
# ---------------------------------------------------------------------------------------------------------


class _InterlevelFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, c: Tensor, w: Tensor, cp: Tensor, wp: Tensor):
        dev = _dev(c)
        c, w, cp = L.f32(c.detach()), L.f32(w.detach()), L.f32(cp.detach())
        wpd = L.f32(wp.detach())
        R, Sc = w.shape
        Sp = wpd.shape[1]
        loss = torch.zeros((1,), device=dev, dtype=torch.float32)
        L.check(L.lib().cnb_interlevel_fwd(c.data_ptr(), w.data_ptr(), cp.data_ptr(), wpd.data_ptr(), R, Sc, Sp, loss.data_ptr(), L.stream_ptr(dev)), "interlevel_fwd")
        ctx.save_for_backward(c, w, cp, wpd)
        ctx.wp_shape = wp.shape
        return loss[0]

    @staticmethod
    def backward(ctx, g: Tensor):
        c, w, cp, wpd = ctx.saved_tensors
        R, Sc = w.shape
        Sp = wpd.shape[1]
        d_wp = torch.empty_like(wpd)
        L.check(L.lib().cnb_interlevel_bwd(c.data_ptr(), w.data_ptr(), cp.data_ptr(), wpd.data_ptr(), R, Sc, Sp, 1.0, d_wp.data_ptr(), L.stream_ptr(c.device)), "interlevel_bwd")
        return None, None, None, (d_wp * g).view(ctx.wp_shape)


def interlevel_term(c: Tensor, w: Tensor, cp: Tensor, wp: Tensor) -> Tensor:
    """mean(lossfun_outer(c, w, cp, wp)) for one proposal level; gradient flows to ``wp`` only."""
    return _InterlevelFn.apply(c, w, cp, wp)


def distortion(c: Tensor, w: Tensor) -> Tensor:
    dev = _dev(c)
    c, w = L.f32(c.detach()), L.f32(w.detach())
    R, S = w.shape
    out = torch.zeros((1,), device=dev, dtype=torch.float32)
    L.check(L.lib().cnb_distortion_fwd(c.data_ptr(), w.data_ptr(), R, S, out.data_ptr(), L.stream_ptr(dev)), "distortion_fwd")
    return out[0]


class _PixelLossFn(torch.autograd.Function):
    """-> (mse, sem_weight * bce) with analytic gradients from the same kernel pass."""

    @staticmethod
    def forward(ctx, rgb: Tensor, sem: Tensor, image: Tensor, mask: Tensor, sem_weight: float):
        dev = _dev(rgb)
        R = rgb.shape[0]
        r, s = L.f32(rgb.detach()), L.f32(sem.detach()).reshape(R)
        img, m = L.f32(image), L.f32(mask).reshape(R)
        losses = torch.zeros((2,), device=dev, dtype=torch.float32)
        d_rgb = torch.empty_like(r)
        d_sem = torch.empty_like(s)
        L.check(
            L.lib().cnb_pixel_losses(r.data_ptr(), s.data_ptr(), img.data_ptr(), m.data_ptr(), R, float(sem_weight), 1.0, losses.data_ptr(),
                                     d_rgb.data_ptr(), d_sem.data_ptr(), L.stream_ptr(dev)),
            "pixel_losses",
        )
        ctx.save_for_backward(d_rgb, d_sem)
        ctx.sem_shape = sem.shape
        return losses[0], losses[1]

    @staticmethod
    def backward(ctx, g_mse, g_bce):
        d_rgb, d_sem = ctx.saved_tensors
        return d_rgb * g_mse, (d_sem * g_bce).view(ctx.sem_shape), None, None, None


def pixel_losses(rgb: Tensor, sem: Tensor, image: Tensor, mask: Tensor, sem_weight: float = 1.0):
    return _PixelLossFn.apply(rgb, sem, image, mask, sem_weight)


# ---------------------------------------------------------------------------------------------------------
# optimiser
# ---------------------------------------------------------------------------------------------------------


def table_to_half(table: Tensor, table_half: Tensor, live: Optional[Tensor] = None, first_unit: int = 0) -> None:
    """table_half = table.half() (``__float2half_rn``); with ``live`` (a flat group's reachable bitmap, the table at 16-byte unit
    ``first_unit``) only the units the optimiser updates are written."""
    dev = _dev(table)
    if table_half.dtype != torch.float16 or table_half.numel() != table.numel() or not table_half.is_contiguous() or not table.is_contiguous():
        raise ValueError("table_to_half: table_half must be a contiguous float16 tensor with the table's size")
    L.check(L.lib().cnb_table_to_half(table.data_ptr(), table.numel(), _p(live), int(first_unit), table_half.data_ptr(), L.stream_ptr(dev)), "table_to_half")


def adam_step(param: Tensor, grad: Tensor, exp_avg: Tensor, exp_avg_sq: Tensor, lr: float, step: int, beta1: float = 0.9, beta2: float = 0.999,
              eps: float = 1e-15, inv_grad_scale: float = 1.0, zero_grad: bool = False, skip_flag: Optional[Tensor] = None,
              live: Optional[Tensor] = None, half: Optional[tuple] = None) -> None:
    """``half`` = (fp16 table copy, first float, float count) of a hash table inside the group (engine.FlatGroup.half): the update also stores
    every table value it writes into the copy."""
    dev = _dev(param)
    if half is not None:
        if not zero_grad:
            raise ValueError("adam_step: the fp16 table refresh is fused into the update + gradient-clear pass (zero_grad=True)")
        tab, first, count = half
        L.check(L.lib().cnb_adam_step_zero_half(param.data_ptr(), grad.data_ptr(), exp_avg.data_ptr(), exp_avg_sq.data_ptr(), param.numel(), lr, beta1,
                                                beta2, eps, int(step), inv_grad_scale, _p(skip_flag), _p(live), tab.data_ptr(), int(first), int(count),
                                                L.stream_ptr(dev)), "adam_step_half")
        return
    if live is not None and zero_grad and skip_flag is None:  # skip the units no hash-grid corner can reach (bit-identical, see reachable_bitmap)
        L.check(L.lib().cnb_adam_step_zero_live(param.data_ptr(), grad.data_ptr(), exp_avg.data_ptr(), exp_avg_sq.data_ptr(), param.numel(), lr, beta1,
                                                beta2, eps, int(step), inv_grad_scale, live.data_ptr(), L.stream_ptr(dev)), "adam_step_live")
        return
    if skip_flag is not None:  # GradScaler.step: device-side "skip on inf/NaN" (always clears the gradient)
        L.check(L.lib().cnb_adam_step_zero_guarded(param.data_ptr(), grad.data_ptr(), exp_avg.data_ptr(), exp_avg_sq.data_ptr(), param.numel(), lr, beta1,
                                                   beta2, eps, int(step), inv_grad_scale, skip_flag.data_ptr(), L.stream_ptr(dev)), "adam_step_guarded")
        return
    fn = L.lib().cnb_adam_step_zero if zero_grad else L.lib().cnb_adam_step
    L.check(
        fn(param.data_ptr(), grad.data_ptr(), exp_avg.data_ptr(), exp_avg_sq.data_ptr(), param.numel(), lr, beta1, beta2, eps,
                              int(step), inv_grad_scale, L.stream_ptr(dev)),
        "adam_step",
    )


def adam_step_scalars(param: Tensor, grad: Tensor, exp_avg: Tensor, exp_avg_sq: Tensor, scalars, live: Optional[Tensor] = None,
                      half: Optional[tuple] = None) -> None:
    """The flat-group update + gradient clear with the step's seven scalars given explicitly (engine.step_scalars: Adam or RAdam):
    ``p -= (s0 / s4) * m / (sqrt(v) / s5 + s3)``.  The scalars travel as one 28-byte device tensor (cnb_adam_step_zero_dev[_live])."""
    dev = _dev(param)
    sc = torch.tensor([float(x) for x in scalars] + [0.0], dtype=torch.float32).to(dev, non_blocking=False)
    if half is not None:  # (fp16 table copy, first float, float count): see adam_step
        tab, first, count = half
        L.check(L.lib().cnb_adam_step_zero_dev_half(param.data_ptr(), grad.data_ptr(), exp_avg.data_ptr(), exp_avg_sq.data_ptr(), param.numel(),
                                                    sc.data_ptr(), _p(live), tab.data_ptr(), int(first), int(count), L.stream_ptr(dev)), "adam_step_dev_half")
    elif live is not None:
        L.check(L.lib().cnb_adam_step_zero_dev_live(param.data_ptr(), grad.data_ptr(), exp_avg.data_ptr(), exp_avg_sq.data_ptr(), param.numel(),
                                                    sc.data_ptr(), live.data_ptr(), L.stream_ptr(dev)), "adam_step_dev_live")
    else:
        L.check(L.lib().cnb_adam_step_zero_dev(param.data_ptr(), grad.data_ptr(), exp_avg.data_ptr(), exp_avg_sq.data_ptr(), param.numel(),
                                               sc.data_ptr(), L.stream_ptr(dev)), "adam_step_dev")
    sc.record_stream(torch.cuda.current_stream(dev))


def grad_check_finite(grad: Tensor, found_inf: Tensor) -> None:
    """found_inf (device int32 [1]) |= any(!isfinite(grad))  -- torch.amp.GradScaler's inf check over one flat gradient group."""
    dev = _dev(grad)
    L.check(L.lib().cnb_grad_check_finite(grad.data_ptr(), grad.numel(), found_inf.data_ptr(), L.stream_ptr(dev)), "grad_check_finite")


def reachable_bitmap(flat: Tensor, tables: Sequence[Tuple[Tensor, int, int, Sequence[float]]], others: Sequence[Tensor]) -> Tensor:
    """One bit per float4 of the flat group ``flat``: 1 where the optimiser has work.  ``tables`` = (hash_table parameter, num_levels,
    log2_hashmap_size, scalings) of every hash grid living in the group (views of ``flat``): only rows some lattice corner hashes to are
    marked (``cnb_hashgrid_mark_reachable``); ``others`` = all remaining parameters (marked whole).  Padding between tensors stays 0."""
    dev = _dev(flat)
    n4 = (flat.numel() + 3) // 4
    bitmap = torch.zeros(((n4 + 31) // 32,), device=dev, dtype=torch.int32)
    base = flat.data_ptr()
    for table, num_levels, log2_T, scalings in tables:
        off = (table.data_ptr() - base) // 4
        if off % 4 != 0:
            raise ValueError("hash table must start on a 16-byte boundary of its flat group")
        g = L.make_grid(table.detach(), None, num_levels, log2_T, scalings)
        L.check(L.lib().cnb_hashgrid_mark_reachable(C.byref(g), bitmap.data_ptr(), off // 4, L.stream_ptr(dev)), "hashgrid_mark_reachable")
    for t in others:
        off = (t.data_ptr() - base) // 4
        first, last = off // 4, (off + t.numel() + 3) // 4
        L.check(L.lib().cnb_bitmap_mark_range(bitmap.data_ptr(), first, last - first, L.stream_ptr(dev)), "bitmap_mark_range")
    return bitmap
