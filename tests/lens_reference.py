"""Reference for lens distortion in ray generation, beside the oracle (``oracle/nerfstudio_torch.py``), which restates the
pinhole path: nerfstudio 1.1.3 ``cameras/camera_utils.py`` ``_compute_residual_and_jacobian`` / ``radial_and_tangential_undistort``
and the undistortion step of ``cameras/cameras.py`` ``Cameras._generate_rays_from_coords``.

[verify]: restated from the published nerfstudio 1.1.3 source, not line-checked (nerfstudio is absent here), like the rest of
the oracle.  Every expression keeps nerfstudio's operation order: torch evaluates it op by op, left to right, so the float32
results are what the reference computes and what ``csrc/lens.cuh`` reproduces.

``generate_pinhole_rays`` and ``next_train_batch`` are the oracle's functions of the same names with an optional
``distortion_params``; with None they return exactly what the oracle's return (tested in ``test_lens_distortion_cpu.py``).
"""
from typing import Optional

import torch
from torch import Tensor


def _compute_residual_and_jacobian(x: Tensor, y: Tensor, xd: Tensor, yd: Tensor, distortion_params: Tensor):
    """camera_utils._compute_residual_and_jacobian: residual of the OPENCV forward model at (x, y) against the distorted point
    (xd, yd), and its Jacobian.  distortion_params [..., 6] = [k1, k2, k3, k4, p1, p2]."""
    k1 = distortion_params[..., 0]
    k2 = distortion_params[..., 1]
    k3 = distortion_params[..., 2]
    k4 = distortion_params[..., 3]
    p1 = distortion_params[..., 4]
    p2 = distortion_params[..., 5]
    r = x * x + y * y
    d = 1.0 + r * (k1 + r * (k2 + r * (k3 + r * k4)))
    fx = d * x + 2 * p1 * x * y + p2 * (r + 2 * x * x) - xd
    fy = d * y + 2 * p2 * x * y + p1 * (r + 2 * y * y) - yd
    d_r = k1 + r * (2.0 * k2 + r * (3.0 * k3 + r * 4.0 * k4))
    d_x = 2.0 * x * d_r
    d_y = 2.0 * y * d_r
    fx_x = d + d_x * x + 2.0 * p1 * y + 6.0 * p2 * x
    fx_y = d_y * x + 2.0 * p1 * x + 2.0 * p2 * y
    fy_x = d_x * y + 2.0 * p2 * y + 2.0 * p1 * x
    fy_y = d + d_y * y + 2.0 * p2 * x + 6.0 * p1 * y
    return fx, fy, fx_x, fx_y, fy_x, fy_y


def radial_and_tangential_undistort(coords: Tensor, distortion_params: Tensor, eps: float = 1e-3, max_iterations: int = 10) -> Tensor:
    """camera_utils.radial_and_tangential_undistort: Newton's method from the distorted point; coords [..., 2]."""
    x = coords[..., 0]
    y = coords[..., 1]
    for _ in range(max_iterations):
        fx, fy, fx_x, fx_y, fy_x, fy_y = _compute_residual_and_jacobian(x=x, y=y, xd=coords[..., 0], yd=coords[..., 1],
                                                                        distortion_params=distortion_params)
        denominator = fy_x * fx_y - fx_x * fy_y
        x_numerator = fx * fy_y - fy * fx_y
        y_numerator = fy * fx_x - fx * fy_x
        step_x = torch.where(torch.abs(denominator) > eps, x_numerator / denominator, torch.zeros_like(denominator))
        step_y = torch.where(torch.abs(denominator) > eps, y_numerator / denominator, torch.zeros_like(denominator))
        x = x + step_x
        y = y + step_y
    return torch.stack([x, y], dim=-1)


def distort(coords: Tensor, distortion_params: Tensor) -> Tensor:
    """The OPENCV forward model the solve inverts: undistorted (x, y) -> distorted (xd, yd)."""
    zero = torch.zeros_like(coords[..., 0])
    fx, fy = _compute_residual_and_jacobian(coords[..., 0], coords[..., 1], zero, zero, distortion_params)[:2]
    return torch.stack([fx, fy], dim=-1)


def _undistort_stack(coord_stack: Tensor, distortion_params: Optional[Tensor]) -> Tensor:
    """The distortion step of _generate_rays_from_coords for perspective cameras: the [3, n, 2] stack (ray, x offset, y offset) is
    undistorted as a whole when any parameter of the batch is non-zero."""
    if distortion_params is not None and bool((distortion_params != 0).any()):
        coord_stack = radial_and_tangential_undistort(coord_stack.reshape(3, -1, 2), distortion_params).reshape(coord_stack.shape)
    return coord_stack


def generate_pinhole_rays(c2w: Tensor, fx: float, fy: float, cx: float, cy: float, coords_yx: Tensor, distortion_params: Optional[Tensor] = None):
    """oracle ``generate_pinhole_rays`` plus nerfstudio's undistortion; distortion_params [6] or None."""
    y, x = coords_yx[..., 0], coords_yx[..., 1]
    coord = torch.stack([(x - cx) / fx, -(y - cy) / fy], -1)
    coord_x_offset = torch.stack([(x - cx + 1) / fx, -(y - cy) / fy], -1)
    coord_y_offset = torch.stack([(x - cx) / fx, -(y - cy + 1) / fy], -1)
    coord_stack = torch.stack([coord, coord_x_offset, coord_y_offset], dim=0)
    coord_stack = _undistort_stack(coord_stack, None if distortion_params is None else torch.as_tensor(distortion_params, dtype=coord_stack.dtype))
    directions_stack = torch.cat([coord_stack, -torch.ones_like(coord_stack[..., :1])], dim=-1)
    rotation = c2w[:3, :3]
    directions_stack = torch.sum(directions_stack[..., None, :] * rotation, dim=-1)
    norm = torch.linalg.norm(directions_stack, dim=-1, keepdim=True)
    directions_stack = directions_stack / norm
    directions = directions_stack[0]
    dx = torch.sqrt(torch.sum((directions - directions_stack[1]) ** 2, dim=-1))
    dy = torch.sqrt(torch.sum((directions - directions_stack[2]) ** 2, dim=-1))
    pixel_area = (dx * dy)[..., None]
    origins = c2w[:3, 3].expand(directions.shape)
    return origins, directions, pixel_area


def next_train_batch(rand3: Tensor, images: Tensor, masks: Optional[Tensor], c2w: Tensor, fx: Tensor, fy: Tensor, cx: Tensor, cy: Tensor,
                     distortion_params: Optional[Tensor] = None):
    """oracle ``next_train_batch`` plus nerfstudio's undistortion; distortion_params [N,6] (per camera) or None."""
    from oracle import nerfstudio_torch as ns

    n, h, w = images.shape[:3]
    idx = ns.pixel_sampler_indices(rand3, n, h, w)
    c, y, x = idx[:, 0], idx[:, 1], idx[:, 2]
    image = images[c, y, x]
    mask = masks[c, y, x][:, None].to(images.dtype) if masks is not None else torch.zeros((idx.shape[0], 1), dtype=images.dtype)
    coords = torch.stack([y.to(rand3.dtype) + 0.5, x.to(rand3.dtype) + 0.5], -1)
    yy, xx = coords[:, 0], coords[:, 1]
    fxc, fyc, cxc, cyc = fx[c], fy[c], cx[c], cy[c]
    coord = torch.stack([(xx - cxc) / fxc, -(yy - cyc) / fyc], -1)
    coord_x_offset = torch.stack([(xx - cxc + 1) / fxc, -(yy - cyc) / fyc], -1)
    coord_y_offset = torch.stack([(xx - cxc) / fxc, -(yy - cyc + 1) / fyc], -1)
    coord_stack = torch.stack([coord, coord_x_offset, coord_y_offset], dim=0)
    coord_stack = _undistort_stack(coord_stack, None if distortion_params is None else distortion_params.to(coord_stack.dtype)[c])
    directions_stack = torch.cat([coord_stack, -torch.ones_like(coord_stack[..., :1])], dim=-1)
    rotation = c2w[c][:, :3, :3]
    directions_stack = torch.sum(directions_stack[..., None, :] * rotation, dim=-1)
    directions_stack = directions_stack / torch.linalg.norm(directions_stack, dim=-1, keepdim=True)
    directions = directions_stack[0]
    dx = torch.sqrt(torch.sum((directions - directions_stack[1]) ** 2, dim=-1))
    dy = torch.sqrt(torch.sum((directions - directions_stack[2]) ** 2, dim=-1))
    return idx, c2w[c][:, :3, 3], directions, (dx * dy)[..., None], image, mask
