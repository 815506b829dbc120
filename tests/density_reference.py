"""Float64 reference of the proposal-network density operator (``csrc/density_field.cu``), beside the oracle
(``oracle/nerfstudio_torch.py``), which restates nerfstudio's ``HashMLPDensityField.get_density`` in float32.

Split at the point where the kernels stop being bit-exact with torch:

* float32, on the CPU, with the oracle's own functions: ``Frustums.get_positions``, ``HashMLPDensityField.normalised_positions``
  (contraction or AABB, selector) and ``HashEncoding.corner_indices`` (table rows and offsets).  The kernels evaluate these with
  separately rounded float32 operations, so the reference picks the corners and offsets the kernels pick, bit for bit.
* float64 (any device): the trilinear blend in the oracle's corner order, ``W1``, ReLU, ``W2``, ``avg * exp(out)`` times the
  selector, and the backward through autograd with ``_TruncExp``'s clamp: table gradient, MLP parameter gradients, the gradient
  reaching the encoded features and, with ``ray_grads``, the gradient reaching the ray origins and directions.

For the ray gradients the offsets are made differentiable in the float64 positions with the floors held fixed: the offset is
``t(o, d) * scale - floor + delta``, where ``t`` is the normalised (contracted) float64 position and ``delta`` is the constant that
makes the value equal the float32 offset at the given rays.  The derivative is then that of the float64 warp, and the value that of
the kernels' cell.
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Dict, Optional, Sequence

import torch
from torch import Tensor

from oracle import nerfstudio_torch as ns


@dataclass
class DensityCase:
    """One call of the operator: rays (per-ray origins / directions, [R, S] starts / ends), grid, warp and parameters."""

    origins: Tensor  # [R, 3] float32
    directions: Tensor  # [R, 3] float32
    starts: Tensor  # [R, S] float32
    ends: Tensor  # [R, S] float32
    num_levels: int
    log2_hashmap_size: int
    scalings: Sequence[float]
    contraction: bool
    aabb: Tensor  # [2, 3] float32
    avg: float
    table: Tensor  # [L * 2^T, 2] float32
    W1: Tensor  # [H, 2L]
    b1: Tensor  # [H]
    W2: Tensor  # [1, H]
    b2: Tensor  # [1]

    @property
    def R(self) -> int:
        return self.starts.shape[0]

    @property
    def S(self) -> int:
        return self.starts.shape[1]


class _Grid:
    """The oracle's HashEncoding index path on explicit scalings (no table: the reference gathers from the case's own)."""

    hash_fn = ns.HashEncoding.hash_fn
    corner_indices = ns.HashEncoding.corner_indices

    def __init__(self, num_levels: int, log2_hashmap_size: int, scalings: Sequence[float]):
        self.scalings = torch.tensor([float(s) for s in scalings[:num_levels]], dtype=torch.float32)
        self.hash_table_size = 2**log2_hashmap_size
        self.hash_offset = torch.arange(num_levels) * self.hash_table_size


class _Warp:
    """The oracle's HashMLPDensityField normalisation (contraction or AABB, then the selector)."""

    normalised_positions = ns.HashMLPDensityField.normalised_positions

    def __init__(self, contraction: bool, aabb: Tensor):
        self.spatial_distortion = ns.SceneContraction() if contraction else None
        self.aabb = aabb


def corners(case: DensityCase) -> Dict[str, Tensor]:
    """The float32 part, on the CPU: world positions [N, 3], normalised positions, selector [N], rows [N, L, 8], offsets [N, L, 3]."""
    R, S = case.R, case.S
    fr = ns.Frustums(case.origins.cpu()[:, None, :].expand(R, S, 3), case.directions.cpu()[:, None, :].expand(R, S, 3),
                     case.starts.cpu()[..., None], case.ends.cpu()[..., None], torch.ones(R, S, 1))
    pos = fr.get_positions().reshape(-1, 3)
    normed, sel = _Warp(case.contraction, case.aabb.cpu()).normalised_positions(pos)
    rows, offsets = _Grid(case.num_levels, case.log2_hashmap_size, case.scalings).corner_indices(normed)
    return {"positions": pos, "normalised": normed, "selector": sel, "rows": rows, "offsets": offsets}


def _normalise64(case: DensityCase, pos: Tensor, inside: Tensor) -> Tensor:
    """The warp in float64; ``inside`` (the float32 ``|p|_inf < 1``) picks the contraction branch, as the kernels picked it."""
    if case.contraction:
        mag = torch.where(inside[:, None], torch.ones_like(pos[:, :1]), pos.abs().amax(dim=-1, keepdim=True))  # no 0/0 in the branch not taken
        pos = torch.where(inside[:, None], pos, (2 - 1 / mag) * (pos / mag))
        return (pos + 2.0) / 4.0
    box = case.aabb.to(pos)
    return (pos - box[0]) / (box[1] - box[0])


def blend(table: Tensor, rows: Tensor, off: Tensor) -> Tensor:
    """HashEncoding.pytorch_fwd's trilinear blend: rows [N, L, 8], offsets [N, L, 3] -> features [N, 2L]."""
    f = table[rows]  # [N, L, 8, 2]
    ox, oy, oz = off[..., 0:1], off[..., 1:2], off[..., 2:3]
    f_03 = f[..., 0, :] * ox + f[..., 3, :] * (1 - ox)
    f_12 = f[..., 1, :] * ox + f[..., 2, :] * (1 - ox)
    f_56 = f[..., 5, :] * ox + f[..., 6, :] * (1 - ox)
    f_47 = f[..., 4, :] * ox + f[..., 7, :] * (1 - ox)
    f0312 = f_03 * oy + f_12 * (1 - oy)
    f4756 = f_47 * oy + f_56 * (1 - oy)
    return torch.flatten(f0312 * oz + f4756 * (1 - oz), start_dim=-2)


def _scaled(case: DensityCase, idx: Dict[str, Tensor], origins: Tensor, directions: Tensor) -> Tensor:
    """float64 ``t * scale`` [N, L, 3] of the sample positions of the given rays (``t``: normalised position, zero where not selected)."""
    S = case.S
    mid = ((case.starts.to(origins) + case.ends.to(origins)) / 2).reshape(-1, 1)
    pos = origins.repeat_interleave(S, dim=0) + directions.repeat_interleave(S, dim=0) * mid
    inside = idx["positions"].abs().amax(dim=-1).to(origins.device) < 1
    t = _normalise64(case, pos, inside) * idx["selector"].to(origins)[:, None]
    return t[:, None, :] * _Grid(case.num_levels, case.log2_hashmap_size, case.scalings).scalings.to(origins)[None, :, None]


def forward(case: DensityCase, idx: Dict[str, Tensor], table: Tensor, W1: Tensor, b1: Tensor, W2: Tensor, b2: Tensor,
            origins: Optional[Tensor] = None, directions: Optional[Tensor] = None):
    """(density [N], features [N, 2L], pre-activation [N]) in the parameters' dtype and device, differentiable in the parameters and,
    when ``origins`` / ``directions`` are given, in the rays (floors held at the float32 cell of ``case``'s own rays)."""
    dtype, device = table.dtype, table.device
    off = idx["offsets"].to(device=device, dtype=dtype)
    if origins is not None:
        grid = _Grid(case.num_levels, case.log2_hashmap_size, case.scalings)
        floor = torch.floor(idx["normalised"][:, None, :] * grid.scalings.view(-1, 1)).to(off)  # the float32 cell, as corner_indices found it
        with torch.no_grad():
            nominal = _scaled(case, idx, case.origins.to(off), case.directions.to(off))
        off = _scaled(case, idx, origins, directions) - floor + (off - (nominal - floor))  # value: the float32 offset at case's rays
    feat = blend(table, idx["rows"].to(device), off)
    hid = torch.relu(feat @ W1.t() + b1)
    out = (hid @ W2.t() + b2)[:, 0]
    density = case.avg * ns.trunc_exp(out) * idx["selector"].to(device=device, dtype=dtype)
    return density, feat, out


def evaluate(case: DensityCase, d_density: Optional[Tensor] = None, ray_grads: bool = False, dtype=torch.float64,
             device: Optional[torch.device] = None, idx: Optional[Dict[str, Tensor]] = None) -> Dict[str, Tensor]:
    """Densities [N] and, given ``d_density`` [N], the gradients of ``sum(density * d_density)``: ``table``, ``W1``, ``b1``, ``W2``,
    ``b2``, ``d_feat`` [N, 2L] (the gradient reaching the encoded features) and, with ``ray_grads``, ``origins`` / ``directions``.
    Also returns ``feat`` [N, 2L] and the pre-activation ``out`` [N].  ``dtype=float32`` evaluates the oracle's arithmetic."""
    device = device if device is not None else torch.device("cpu")
    idx = idx if idx is not None else corners(case)
    cast = lambda t: t.detach().to(device=device, dtype=dtype)  # noqa: E731
    grad = d_density is not None
    params = {k: cast(getattr(case, k)).requires_grad_(grad) for k in ("table", "W1", "b1", "W2", "b2")}
    rays = {k: cast(getattr(case, k)).requires_grad_(True) for k in ("origins", "directions")} if ray_grads else {}
    density, feat, out = forward(case, idx, **params, **rays)
    res = {"density": density.detach(), "feat": feat.detach(), "out": out.detach()}
    if not grad:
        return res
    feat.retain_grad()
    (density * cast(d_density)).sum().backward()
    res.update({k: p.grad for k, p in params.items()})
    res.update({k: p.grad for k, p in rays.items()})
    res["d_feat"] = feat.grad
    return res


def make_case(R: int, S: int, num_levels: int, hidden: int, contraction: bool, seed: int = 0, log2_hashmap_size: int = 14,
              max_res: int = 2048, avg: float = 1.0, out_shift: float = 0.0) -> DensityCase:
    """Seeded rays and parameters.  Rays start inside the unit box and run up to 2.5 units, so without contraction part of every ray
    leaves the box (selector 0); ray 1 runs out to 2000 (the contraction's outer shell), ray 2 has zero-length frustums.  Features are
    O(0.5) with hash collisions on the fine levels (2^14 rows per level); ``out_shift`` moves the MLP output (``trunc_exp``'s clamp)."""
    g = torch.Generator().manual_seed(seed)
    u = lambda *shape: torch.rand(shape, generator=g) * 2 - 1  # noqa: E731
    origins = u(R, 3) * 0.6
    directions = torch.nn.functional.normalize(torch.randn((R, 3), generator=g), dim=-1)
    edges = torch.sort(torch.rand((R, S + 1), generator=g) * 2.5, dim=-1).values
    if R > 1:
        edges[1] = torch.linspace(0.0, 2000.0, S + 1)
    starts, ends = edges[:, :-1].contiguous(), edges[:, 1:].contiguous()
    if R > 2:
        ends[2] = starts[2]
    L, H, T = num_levels, hidden, 2**log2_hashmap_size
    return DensityCase(
        origins=origins, directions=directions, starts=starts, ends=ends, num_levels=L, log2_hashmap_size=log2_hashmap_size,
        scalings=ns.hash_scalings(L, 16, max_res).tolist(), contraction=contraction, aabb=torch.tensor([[-1.0] * 3, [1.0] * 3]), avg=avg,
        table=u(L * T, 2) * 0.5, W1=u(H, 2 * L) * (6.0 / (2 * L)) ** 0.5, b1=u(H) * 0.2, W2=u(1, H) * (6.0 / H) ** 0.5,
        b2=u(1) * 0.2 + out_shift)
