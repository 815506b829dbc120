"""Export / projection render loops (callers of the hot path), sharded by ray range across ranks with no data-path
collective (SURVEY.md section 8e).

* :func:`generate_point_cloud` -- the render loop of ``export/exporter_utils_nerfacto.py:126-183`` (``ns-export
  pointcloud`` as patched by ``debug/exporter_nerfacto.py``): render a batch of training rays, back-project the median
  depth, keep rays whose semantic label is "fruit" (``sigmoid(sem) > 0.9``) and that fall inside the crop OBB, until
  ``num_points`` are collected.  The open3d outlier removal / normal estimation that follows in the reference is CPU
  geometry-library work and out of scope.
* :func:`render_cluster_projection` -- the per-(camera, cluster AABB) step of ``FruitModel.get_outputs_for_projections``
  (``fruit_nerf.py:283-315``): un-occluded semantic render of the rays hitting the box, and the opacity accumulated in
  front of the box (occluded where >= 0.5).
* :func:`write_ply` -- ``semantics_pc.ply`` in the layout ``segmentation/segmenter.py:210`` reads (float xyz, uchar rgb).
* :func:`generate_rays` -- device-side ``cam.generate_rays(aabb_box=...)`` (pixel -> ray -> slab test in one kernel), with
  nerfstudio's OPENCV lens undistortion when the camera has non-zero ``distortion_params``.
* :func:`cameras_from_nerfstudio` -- nerfstudio ``Cameras`` -> :class:`PinholeCamera` list (perspective only; others are refused).
* :func:`project_clusters` -- the whole ``get_outputs_for_projections`` loop (``fruit_nerf.py:254-318``) writing the
  ``super_cluster_k/cam_j/{wo_occ,visible}_cluster_i.png`` tree ``segmentation/merger.py`` reads, sharded over ranks.
"""
from __future__ import annotations

import struct
from dataclasses import dataclass
from typing import Callable, Dict, List, Optional, Sequence, Tuple

import pickle

import numpy as np
import torch
from torch import Tensor

from .rays import RayBundle


def shard_range(n: int, rank: int, world_size: int) -> Tuple[int, int]:
    """Contiguous, disjoint, covering split of ``range(n)`` -- how rays / cameras are divided across ranks."""
    return (n * rank) // world_size, (n * (rank + 1)) // world_size


@dataclass
class OrientedBox:
    """nerfstudio ``OrientedBox`` (R, T, S) with ``within`` as used at exporter_utils_nerfacto.py:170-176."""

    R: Tensor  # [3,3]
    T: Tensor  # [3]
    S: Tensor  # [3]

    @staticmethod
    def from_params(pos, rpy, scale) -> "OrientedBox":
        r, p, y = rpy
        cr, sr, cp, sp, cy, sy = np.cos(r), np.sin(r), np.cos(p), np.sin(p), np.cos(y), np.sin(y)
        rx = np.array([[1, 0, 0], [0, cr, -sr], [0, sr, cr]])
        ry = np.array([[cp, 0, sp], [0, 1, 0], [-sp, 0, cp]])
        rz = np.array([[cy, -sy, 0], [sy, cy, 0], [0, 0, 1]])
        return OrientedBox(torch.tensor(rz @ ry @ rx, dtype=torch.float32), torch.tensor(pos, dtype=torch.float32), torch.tensor(scale, dtype=torch.float32))

    def within(self, pts: Tensor) -> Tensor:
        R, T, S = self.R.to(pts), self.T.to(pts), self.S.to(pts)
        local = (pts - T) @ R  # == (R^T (p - T))^T
        return ((local > -S / 2) & (local < S / 2)).all(dim=-1)


def _obb_array(crop_obb: Optional["OrientedBox"]):
    import ctypes as C

    if crop_obb is None:
        return None
    vals = [float(v) for v in crop_obb.R.detach().cpu().reshape(-1).tolist()] + [float(v) for v in crop_obb.T.detach().cpu().tolist()] \
        + [float(v) for v in crop_obb.S.detach().cpu().tolist()]
    return (C.c_float * 15)(*vals)


def generate_point_cloud(model, next_rays: Callable[[int], RayBundle], num_points: int, crop_obb: Optional[OrientedBox] = None,
                         only_semantics: bool = True, rank: int = 0, world_size: int = 1, max_batches: int = 1 << 30, lag: int = 2) -> Dict[str, Tensor]:
    """Rank-local share of the export (export/exporter_utils_nerfacto.py:126-183): collects ``num_points / world_size`` kept points.
    ``next_rays(i)`` returns the i-th ray batch of this rank (ranks draw disjoint ray streams).

    Per batch: the fused render, then ONE C call (``cnb_extract_points``) does depth -> point -> semantic mask -> OBB test ->
    order-preserving append into the output arrays, with the running count kept in device memory.  The host never waits for a batch it has
    just launched: the count of batch ``i - lag`` (an asynchronous 4-byte copy into pinned memory) decides whether batch ``i`` is still
    needed, so at most ``lag`` batches are rendered beyond the one that completes the cloud -- their points fall past ``num_points`` and are
    dropped, so the result is exactly the first ``num_points / world_size`` kept points of the ray stream, in stream order, as in the
    reference's loop.  ``rays_needed`` counts the rays up to the completing batch (what the reference renders), ``rays_rendered`` all of them."""
    import ctypes as C

    from . import _lib as L

    dev = model.device
    if dev.type != "cuda":
        raise RuntimeError("cropnerf_b200.generate_point_cloud runs on CUDA devices only; there is no CPU fallback")
    lo, hi = shard_range(num_points, rank, world_size)
    want = hi - lo
    points = torch.empty((want, 3), device=dev, dtype=torch.float32)
    rgbs = torch.empty((want, 3), device=dev, dtype=torch.float32)
    dirs = torch.empty((want, 3), device=dev, dtype=torch.float32)
    counters = torch.zeros((2,), device=dev, dtype=torch.int32)
    ring = lag + 2
    host_counts = torch.zeros((ring,), dtype=torch.int32, pin_memory=True)
    events = [torch.cuda.Event() for _ in range(ring)]
    obb = _obb_array(crop_obb)
    lib = L.lib()
    scratch = None
    cum: List[int] = []      # kept points after batch j (filled as the counts arrive)
    sizes: List[int] = []
    i = 0

    def collect(j: int) -> int:
        events[j % ring].synchronize()
        cum.append(int(host_counts[j % ring]))
        return cum[-1]

    stream = torch.cuda.current_stream(dev)
    while want > 0 and i < max_batches:
        if i >= lag and collect(i - lag) >= want:
            break
        with torch.no_grad():
            ray_bundle = next_rays(i)
            outputs = model(ray_bundle)
        n = len(ray_bundle)
        sizes.append(n)
        need = int(lib.cnb_extract_points_scratch_ints(n))
        if scratch is None or scratch.numel() < need:
            scratch = torch.empty((max(need, 1),), device=dev, dtype=torch.int32)
        o, d = L.f32(ray_bundle.origins.reshape(n, 3)), L.f32(ray_bundle.directions.reshape(n, 3))
        depth, sem, rgb = L.f32(outputs["depth"].reshape(n)), L.f32(outputs["semantics"].reshape(n)), L.f32(outputs["rgb"].reshape(n, 3))
        L.check(lib.cnb_extract_points(o.data_ptr(), d.data_ptr(), depth.data_ptr(), sem.data_ptr(), rgb.data_ptr(), n, obb, int(only_semantics), 0.9,
                                       scratch.data_ptr(), counters[i & 1 :].data_ptr(), counters[(i + 1) & 1 :].data_ptr(), want, points.data_ptr(),
                                       rgbs.data_ptr(), dirs.data_ptr(), L.stream_ptr(dev)), "extract_points")
        host_counts[i % ring : i % ring + 1].copy_(counters[(i + 1) & 1 : ((i + 1) & 1) + 1], non_blocking=True)
        events[i % ring].record(stream)
        i += 1
    for j in range(len(cum), i):
        collect(j)
    have = min(cum[-1], want) if cum else 0
    needed = next((k + 1 for k, c in enumerate(cum) if c >= want), len(cum))
    return {"points": points[:have], "rgbs": rgbs[:have], "view_directions": dirs[:have], "rays_rendered": int(sum(sizes)),
            "rays_needed": int(sum(sizes[:needed])), "batches": i}


def write_ply(path: str, points: Tensor, rgbs: Tensor) -> None:
    """Binary little-endian PLY: float x y z, uchar red green blue (debug/exporter_nerfacto.py:140-146)."""
    pts = points.detach().cpu().numpy().astype("<f4")
    col = (rgbs.detach().cpu().clamp(0, 1).numpy() * 255).astype(np.uint8)
    n = pts.shape[0]
    header = ("ply\nformat binary_little_endian 1.0\n" f"element vertex {n}\n" "property float x\nproperty float y\nproperty float z\n"
              "property uchar red\nproperty uchar green\nproperty uchar blue\nend_header\n")
    rec = np.empty(n, dtype=[("p", "<f4", 3), ("c", "u1", 3)])
    rec["p"], rec["c"] = pts, col
    with open(path, "wb") as f:
        f.write(header.encode("ascii"))
        f.write(rec.tobytes())


def generate_rays(c2w: Tensor, fx: float, fy: float, cx: float, cy: float, width: int, height: int, device, aabb: Optional[Tensor] = None,
                  pixel_yx: Optional[Tensor] = None, camera_index: int = 0, count_valid: bool = False, distortion_params: Optional[Tensor] = None):
    """``cam.generate_rays(camera_indices=0, keep_shape=True, aabb_box=aabb)`` (fruit_nerf.py:283) for one perspective camera
    on the device: one kernel does pixel -> direction -> normalisation -> pixel_area -> AABB slab test (``cnb_generate_rays``).
    Returns a flat RayBundle of width*height rays (or of the given integer ``pixel_yx`` [n,2]); with ``aabb`` ([2,3] or [6])
    ``nears``/``fars`` are set and misses carry 1e10 (``valid = nears < 1e10``, fruit_nerf.py:286).  ``count_valid`` also
    returns the number of rays that hit the box as a device int32 tensor (no host sync).  ``distortion_params`` (6 values,
    nerfstudio's ``[k1, k2, k3, k4, p1, p2]``) undistorts every pixel coordinate as nerfstudio does (``cnb_generate_rays_lens``);
    None or all zero gives the pinhole rays."""
    import ctypes as C

    from . import _lib as L

    dev = torch.device(device)
    if dev.type != "cuda":
        raise RuntimeError("cropnerf_b200.generate_rays runs on CUDA devices only; there is no CPU fallback")
    cam = L.Camera()
    m = c2w.detach().cpu().float().reshape(-1)[:12].tolist()
    for i in range(12):
        cam.c2w[i] = m[i]
    cam.fx, cam.fy, cam.cx, cam.cy, cam.width, cam.height = float(fx), float(fy), float(cx), float(cy), int(width), int(height)
    pix = None
    n = int(width) * int(height)
    if pixel_yx is not None:
        pix = pixel_yx.to(dev, torch.int32).contiguous()
        n = pix.shape[0]
    box = None
    if aabb is not None:
        box = (C.c_float * 6)(*[float(v) for v in aabb.detach().cpu().reshape(-1).tolist()])
    o = torch.empty((n, 3), device=dev, dtype=torch.float32)
    d = torch.empty((n, 3), device=dev, dtype=torch.float32)
    area = torch.empty((n, 1), device=dev, dtype=torch.float32)
    nears = torch.empty((n, 1), device=dev, dtype=torch.float32) if aabb is not None else None
    fars = torch.empty((n, 1), device=dev, dtype=torch.float32) if aabb is not None else None
    cnt = torch.zeros((1,), device=dev, dtype=torch.int32) if (count_valid and aabb is not None) else None
    lens = _lens_struct(distortion_params)
    if lens is None:
        L.check(L.lib().cnb_generate_rays(C.byref(cam), L.ptr(pix), n, box, o.data_ptr(), d.data_ptr(), area.data_ptr(), L.ptr(nears), L.ptr(fars),
                                          L.ptr(cnt), L.stream_ptr(dev)), "generate_rays")
    else:
        L.check(L.lib().cnb_generate_rays_lens(C.byref(cam), C.byref(lens), L.ptr(pix), n, box, o.data_ptr(), d.data_ptr(), area.data_ptr(),
                                               L.ptr(nears), L.ptr(fars), L.ptr(cnt), L.stream_ptr(dev)), "generate_rays_lens")
    rb = RayBundle(origins=o, directions=d, pixel_area=area, camera_indices=torch.full((n, 1), int(camera_index), device=dev, dtype=torch.int32),
                   nears=nears, fars=fars)
    return (rb, cnt) if count_valid else rb


def aabb_near_far(origins: Tensor, directions: Tensor, aabb: Tensor, invalid: float = 1e10) -> Tuple[Tensor, Tensor]:
    """nerfstudio ``intersect_aabb`` (utils/math.py; what ``cam.generate_rays(aabb_box=...)`` sets, fruit_nerf.py:283) for an arbitrary flat
    ray bundle, in torch ops (the per-camera path uses the fused kernel, :func:`generate_rays`): slab test against an AABB [2,3], both
    distances clamped to [0, 1e10], rays with ``t_max <= t_min`` are misses and get nears = fars = ``invalid``."""
    lo, hi = aabb[0].to(origins), aabb[1].to(origins)
    t0 = (lo - origins) / directions
    t1 = (hi - origins) / directions
    tmin = torch.minimum(t0, t1).amax(dim=-1, keepdim=True).clamp(min=0.0, max=1e10)
    tmax = torch.maximum(t0, t1).amin(dim=-1, keepdim=True).clamp(min=0.0, max=1e10)
    miss = tmax <= tmin
    return torch.where(miss, torch.full_like(tmin, invalid), tmin), torch.where(miss, torch.full_like(tmax, invalid), tmax)


def render_cluster_projection(model, rays: RayBundle, aabb: Tensor) -> Dict[str, Tensor]:
    """One (camera, cluster) step of fruit_nerf.py:283-315 on a flat ray bundle [N]: returns per-ray ``valid``,
    ``semantics`` (un-occluded render between the box's near/far) and ``front_opacity`` (sum of weights on [0, near])."""
    dev = model.device
    o, d = rays.origins.to(dev), rays.directions.to(dev)
    nears, fars = aabb_near_far(o, d, aabb.to(dev))
    valid = nears[:, 0] < 1e10
    n = o.shape[0]
    sem = torch.zeros((n, 3), device=dev)
    front = torch.zeros((n,), device=dev)
    if int(valid.sum()) >= 10:  # fruit_nerf.py:293: fewer than 10 valid rays -> black images
        sub = RayBundle(origins=o[valid], directions=d[valid], pixel_area=None if rays.pixel_area is None else rays.pixel_area.to(dev)[valid],
                        camera_indices=None if rays.camera_indices is None else rays.camera_indices.to(dev)[valid],
                        nears=nears[valid], fars=fars[valid])
        with torch.no_grad():
            out = model.get_outputs_for_camera_jagged_ray_bundle(sub)
            sem[valid] = out["semantics"].to(dev).expand(-1, 3)
            sub.fars = sub.nears
            sub.nears = torch.zeros_like(sub.nears)
            front[valid] = model.get_density_for_camera_ray_bundle(sub).to(dev)
    visible = sem.clone()
    visible[front >= 0.5] = 0.0
    return {"valid": valid, "semantics": sem, "front_opacity": front, "visible": visible}


# ---------------------------------------------------------------------------------------------------------------------
# "next" row f3: the files the downstream stages read (segmentation/segmenter.py, segmentation/merger.py)


@dataclass
class PinholeCamera:
    """What the projection loop needs of one nerfstudio ``Cameras`` entry: a perspective camera, optionally with OPENCV lens
    distortion (``distortion_params``: 6 values in nerfstudio's order ``[k1, k2, k3, k4, p1, p2]``; None = none)."""

    c2w: Tensor  # [3,4]
    fx: float
    fy: float
    cx: float
    cy: float
    width: int
    height: int
    distortion_params: Optional[Tensor] = None


# nerfstudio cameras/cameras.py CameraType (enum auto() values); only PERSPECTIVE is generated here
_CAMERA_TYPES = {1: "PERSPECTIVE", 2: "FISHEYE", 3: "EQUIRECTANGULAR", 4: "OMNIDIRECTIONALSTEREO_L", 5: "OMNIDIRECTIONALSTEREO_R", 6: "VR180_L",
                 7: "VR180_R", 8: "ORTHOPHOTO", 9: "FISHEYE624"}
_PERSPECTIVE = 1


def check_perspective(camera_type, what: str) -> None:
    """Raise ``ValueError`` naming the type unless every entry of ``camera_type`` (a nerfstudio ``camera_type`` tensor, a
    ``CameraType`` member or an int; None = perspective) is ``CameraType.PERSPECTIVE``.  Other projection models are refused,
    not rendered as pinholes."""
    if camera_type is None:
        return
    values = torch.as_tensor(getattr(camera_type, "value", camera_type)).reshape(-1).tolist()
    for v in values:
        if int(v) != _PERSPECTIVE:
            raise ValueError(f"{what}: camera type {_CAMERA_TYPES.get(int(v), int(v))} is not supported; only perspective cameras "
                             "(with or without OPENCV k1..k4, p1, p2 distortion) are")


def lens_values(distortion_params) -> Optional[List[float]]:
    """nerfstudio ``distortion_params`` of one camera -> its 6 floats (None stays None)."""
    if distortion_params is None:
        return None
    t = torch.as_tensor(distortion_params).detach().cpu().to(torch.float32).reshape(-1)
    if t.numel() != 6:
        raise ValueError(f"distortion_params must hold 6 values [k1, k2, k3, k4, p1, p2], got {t.numel()}")
    return t.tolist()


def _lens_struct(distortion_params):
    from . import _lib as L

    v = lens_values(distortion_params)
    return None if v is None else L.Lens(*v)


def cameras_from_nerfstudio(cameras) -> List[PinholeCamera]:
    """nerfstudio ``Cameras`` (batch [N], or one row) -> one :class:`PinholeCamera` per camera, read by attribute name so that
    nerfstudio need not be importable: ``camera_to_worlds`` [N,3,4], ``fx, fy, cx, cy, width, height`` [N,1],
    ``distortion_params`` [N,6] or None, ``camera_type`` [N,1].  Raises ``ValueError`` on a camera that is not perspective
    (fisheye, equirectangular, fisheye624, orthophoto, ...) and on unexpected shapes."""
    c2w = torch.as_tensor(cameras.camera_to_worlds).detach().cpu().to(torch.float32)
    single = c2w.dim() == 2
    if single:
        c2w = c2w[None]
    if c2w.dim() != 3 or tuple(c2w.shape[1:]) != (3, 4):
        raise ValueError(f"cameras.camera_to_worlds has shape {tuple(cameras.camera_to_worlds.shape)}, expected [N,3,4]")
    n = int(c2w.shape[0])

    def per_camera(name, width):
        t = torch.as_tensor(getattr(cameras, name)).detach().cpu()
        want = (width,) if single else (n, width)
        if tuple(t.shape) != want:
            raise ValueError(f"cameras.{name} has shape {tuple(t.shape)}, expected {list(want)}")
        return t.reshape(n, width)

    camera_type = getattr(cameras, "camera_type", None)
    if camera_type is not None:
        if isinstance(camera_type, Tensor):
            per_camera("camera_type", 1)
        check_perspective(camera_type, "cameras_from_nerfstudio")
    fx, fy, cx, cy = (per_camera(k, 1).to(torch.float32) for k in ("fx", "fy", "cx", "cy"))
    width, height = per_camera("width", 1), per_camera("height", 1)
    dist = per_camera("distortion_params", 6).to(torch.float32) if getattr(cameras, "distortion_params", None) is not None else None
    return [PinholeCamera(c2w=c2w[i].clone(), fx=float(fx[i, 0]), fy=float(fy[i, 0]), cx=float(cx[i, 0]), cy=float(cy[i, 0]),
                          width=int(width[i, 0]), height=int(height[i, 0]), distortion_params=None if dist is None else dist[i].clone())
            for i in range(n)]


class _NumpyOnlyUnpickler(pickle.Unpickler):
    """The cluster-info file is a pickled object array (the reference writes it with ``np.save(..., allow_pickle=True)``): dicts, lists, ints and
    numpy arrays.  Unpickling is restricted to the numpy reconstruction helpers, so a crafted file cannot run code (ADVICE r1)."""

    _ALLOWED = {
        ("numpy.core.multiarray", "_reconstruct"), ("numpy._core.multiarray", "_reconstruct"), ("numpy", "ndarray"), ("numpy", "dtype"),
        ("numpy.core.multiarray", "scalar"), ("numpy._core.multiarray", "scalar"), ("numpy.core.numeric", "_frombuffer"),
        ("numpy._core.numeric", "_frombuffer"),
    }

    def find_class(self, module, name):
        if (module, name) in self._ALLOWED:
            return super().find_class(module, name)
        raise pickle.UnpicklingError(f"cluster info: refusing to unpickle {module}.{name}")


def load_cluster_info(path: str, allow_pickle: bool = False) -> List[dict]:
    """``all_super_cluster_info_nsub_*.npy`` written by segmentation/segmenter.py:153-181: a pickled list of
    ``{'aabb': float[k,2,3] (min,max per sub-cluster), 'pcd': {sub_id: float[n,3]}}`` (read at fruit_nerf.py:265).
    By default only numpy arrays / plain containers are unpickled; ``allow_pickle=True`` is the reference's unrestricted ``np.load``."""
    if allow_pickle:
        data = np.load(path, allow_pickle=True)
    else:
        with open(path, "rb") as f:
            version = np.lib.format.read_magic(f)
            shape, fortran, dtype = np.lib.format.read_array_header_1_0(f) if version == (1, 0) else np.lib.format.read_array_header_2_0(f)
            if dtype.hasobject:
                data = _NumpyOnlyUnpickler(f).load()
            else:
                f.seek(0)
                data = np.load(f, allow_pickle=False)
    out = []
    for item in list(data):
        aabb = np.asarray(item["aabb"], dtype=np.float32)
        if aabb.ndim != 3 or aabb.shape[1:] != (2, 3):
            raise ValueError(f"{path}: cluster aabb has shape {aabb.shape}, expected [k,2,3]")
        out.append({"aabb": aabb, "pcd": item.get("pcd", {})})
    return out


def save_cluster_info(path: str, clusters: List[dict]) -> None:
    np.save(path, np.asarray(clusters, dtype=object), allow_pickle=True)


def to_png_bytes(image: Tensor) -> np.ndarray:
    """torchvision.utils.save_image quantisation (used at fruit_nerf.py:295-315): ``clamp(x*255 + 0.5, 0, 255)`` -> uint8 HxWx3."""
    img = image.detach().float().cpu()
    if img.dim() == 2:
        img = img[..., None].expand(-1, -1, 3)
    return img.mul(255).add_(0.5).clamp_(0, 255).to(torch.uint8).numpy()


def write_png(path: str, image: Tensor) -> None:
    import cv2

    arr = to_png_bytes(image)
    if not cv2.imwrite(path, np.ascontiguousarray(arr[..., ::-1])):  # cv2 wants BGR
        raise IOError(f"could not write {path}")


def _camera_struct(cam: "PinholeCamera"):
    from . import _lib as L

    c = L.Camera()
    m = torch.as_tensor(cam.c2w).detach().cpu().float().reshape(-1)[:12].tolist()
    for i in range(12):
        c.c2w[i] = m[i]
    c.fx, c.fy, c.cx, c.cy, c.width, c.height = float(cam.fx), float(cam.fy), float(cam.cx), float(cam.cy), int(cam.width), int(cam.height)
    return c


def _render_on_device(model, bundle: RayBundle, keys: Sequence[str]) -> Dict[str, Tensor]:
    """Chunked no-grad render of a flat DEVICE bundle; the requested outputs stay on the device (no pinned-host round trip)."""
    n = len(bundle)
    step = int(model.config.eval_num_rays_per_chunk)
    parts: Dict[str, List[Tensor]] = {k: [] for k in keys}
    with torch.no_grad():
        for i in range(0, n, step):
            out = model(bundle._map(lambda t: t[i : i + step]))
            for k in keys:
                parts[k].append(out[k])
    return {k: (torch.cat(v, dim=0) if len(v) != 1 else v[0]) for k, v in parts.items()}


def project_camera_boxes(model, cam: "PinholeCamera", boxes: Tensor, min_valid_rays: int = 10, occlusion_threshold: float = 0.5,
                         capacity: Optional[int] = None) -> Dict[str, Tensor]:
    """One (super-cluster, camera) pair of ``get_outputs_for_projections`` (fruit_nerf.py:276-315) with ALL ``k`` sub-cluster boxes in
    one pass: ``cnb_generate_rays_boxes`` builds the compacted list of (pixel, box) hits, two fused renders over that list give the
    un-occluded semantics (between each box's near / far) and the opacity in front of the box (0 .. near), and
    ``cnb_projection_scatter`` writes the quantised pixels into the k ``wo_occ`` / ``visible`` images.  One host read-back (the hit
    count) per pair; images are returned as device uint8 ``[k, H, W]`` (single channel: the reference's three channels are equal)."""
    import ctypes as C

    from . import _lib as L

    dev = model.device
    if dev.type != "cuda":
        raise RuntimeError("cropnerf_b200.project_camera_boxes runs on CUDA devices only; there is no CPU fallback")
    boxes_d = L.f32(torch.as_tensor(boxes, dtype=torch.float32).reshape(-1, 6).to(dev))
    k = int(boxes_d.shape[0])
    npix = int(cam.width) * int(cam.height)
    cap = int(capacity) if capacity is not None else min(k * npix, max(npix, 1 << 21))
    check_perspective(getattr(cam, "camera_type", None), "project_camera_boxes")
    cs = _camera_struct(cam)
    lens = _lens_struct(getattr(cam, "distortion_params", None))
    lib = L.lib()
    while True:
        o = torch.empty((cap, 3), device=dev)
        d = torch.empty((cap, 3), device=dev)
        area = torch.empty((cap, 1), device=dev)
        nears = torch.empty((cap, 1), device=dev)
        fars = torch.empty((cap, 1), device=dev)
        tags = torch.empty((cap,), device=dev, dtype=torch.int32)
        count = torch.zeros((1,), device=dev, dtype=torch.int32)
        L.check(lib.cnb_generate_rays_boxes_lens(C.byref(cs), None if lens is None else C.byref(lens), boxes_d.data_ptr(), k, cap, o.data_ptr(),
                                                 d.data_ptr(), area.data_ptr(), nears.data_ptr(), fars.data_ptr(), tags.data_ptr(), count.data_ptr(),
                                                 L.stream_ptr(dev)), "generate_rays_boxes")
        n = int(count.item())  # the one host read-back of the pair
        if n <= cap:
            break
        cap = n                # more overlapping boxes than the first guess: once more with room for every hit
    wo_occ = torch.zeros((k, int(cam.height), int(cam.width)), device=dev, dtype=torch.uint8)
    visible = torch.zeros_like(wo_occ)
    rays = 0
    if n > 0:
        o, d, area, nears, fars, tags = o[:n], d[:n], area[:n], nears[:n], fars[:n], tags[:n]
        box_of = torch.div(tags, npix, rounding_mode="floor")
        per_box = torch.bincount(box_of, minlength=k)
        if bool((per_box < min_valid_rays).any()):  # fruit_nerf.py:293: fewer than 10 hit rays -> that box's images stay black
            keep = per_box[box_of.long()] >= min_valid_rays
            o, d, area, nears, fars, tags = o[keep], d[keep], area[keep], nears[keep], fars[keep], tags[keep]
            n = int(tags.shape[0])
    if n > 0:
        cam_idx = torch.zeros((n, 1), device=dev, dtype=torch.int32)
        bundle = RayBundle(origins=o, directions=d, pixel_area=area, camera_indices=cam_idx, nears=nears, fars=fars)
        sem = _render_on_device(model, bundle, ("semantics",))["semantics"]
        front_bundle = RayBundle(origins=o, directions=d, pixel_area=area, camera_indices=cam_idx, nears=torch.zeros_like(nears), fars=nears)
        front = _render_on_device(model, front_bundle, ("accumulation",))["accumulation"]
        L.check(lib.cnb_projection_scatter(tags.contiguous().data_ptr(), L.f32(sem.reshape(n)).data_ptr(), L.f32(front.reshape(n)).data_ptr(), n,
                                           float(occlusion_threshold), wo_occ.data_ptr(), visible.data_ptr(), L.stream_ptr(dev)), "projection_scatter")
        rays = 2 * n
    return {"wo_occ": wo_occ, "visible": visible, "rays": rays, "hits": n}


def write_png_u8(path: str, image_u8: np.ndarray) -> None:
    """uint8 [H,W] -> the 3-channel PNG ``save_image`` writes for a gray [3,H,W] tensor."""
    import cv2

    if not cv2.imwrite(path, np.ascontiguousarray(np.repeat(image_u8[..., None], 3, axis=-1))):
        raise IOError(f"could not write {path}")


def project_clusters(model, cameras: Sequence[PinholeCamera], clusters: List[dict], out_dir: Optional[str], rank: int = 0, world_size: int = 1,
                     segmentation_files: Optional[Sequence[str]] = None) -> Dict[str, int]:
    """``FruitModel.get_outputs_for_projections`` (fruit_nerf.py:254-318) with the (super-cluster, camera) pairs sharded over
    the ranks (no communication).  Every pair is one :func:`project_camera_boxes` call (all sub-cluster boxes of the super-cluster in one
    ray-generation pass and two batched renders); the uint8 images come down in one copy per pair and are written as
    ``super_cluster_{k}/cam_{j}/wo_occ_cluster_{i}.png`` / ``visible_cluster_{i}.png`` -- the layout segmentation/merger.py:219-333 reads.
    ``out_dir=None`` renders without writing files (benchmarks).  Returns counters (pairs, images, rays rendered).
    ``cameras`` may also be a nerfstudio ``Cameras`` batch (see :func:`cameras_from_nerfstudio`); lens distortion is applied, and a
    camera that is not perspective raises ``ValueError`` before anything is rendered."""
    import os
    import shutil

    if hasattr(cameras, "camera_to_worlds"):
        cameras = cameras_from_nerfstudio(cameras)
    for cam in cameras:
        check_perspective(getattr(cam, "camera_type", None), "project_clusters")

    stats = {"pairs": 0, "images": 0, "rays": 0}
    pair = 0
    for i_sc, cluster in enumerate(clusters):
        boxes = torch.as_tensor(cluster["aabb"], dtype=torch.float32)
        for cam_idx, cam in enumerate(cameras):
            mine = pair % world_size == rank
            pair += 1
            if not mine:
                continue
            res = project_camera_boxes(model, cam, boxes)
            stats["pairs"] += 1
            stats["rays"] += int(res["rays"])
            stats["images"] += 2 * int(boxes.shape[0])
            if out_dir is None:
                continue
            cam_dir = os.path.join(out_dir, f"super_cluster_{i_sc}", f"cam_{cam_idx}")
            os.makedirs(cam_dir, exist_ok=True)
            wo, vis = res["wo_occ"].cpu().numpy(), res["visible"].cpu().numpy()
            for i in range(boxes.shape[0]):
                write_png_u8(os.path.join(cam_dir, f"wo_occ_cluster_{i}.png"), wo[i])
                write_png_u8(os.path.join(cam_dir, f"visible_cluster_{i}.png"), vis[i])
            if segmentation_files is not None:
                shutil.copy(segmentation_files[cam_idx], cam_dir)
    return stats


# ---------------------------------------------------------------------------------------------------------------------
# "next" row f4: volumetric export (scripts/exporter.py ExportSemanticPointCloud -> export/exporter_utils.py sample_volume)


def aabb_corners(aabb) -> Tensor:
    """``get_corners_of_aabb`` (data/fruit_datamanager.py:42-68): the 8 corners, x fastest, then y, then z."""
    lo, hi = [float(v) for v in aabb[0]], [float(v) for v in aabb[1]]
    return torch.tensor([[(hi if i & 1 else lo)[0], (hi if i & 2 else lo)[1], (hi if i & 4 else lo)[2]] for i in range(8)], dtype=torch.float32)


def volume_surface_rays(aabb, num_points_per_side: int) -> Tuple[Tensor, Tensor, float]:
    """``sample_surface_points`` + ``OrthographicRayGenerator`` (data/fruit_datamanager.py:71-120,
    components/ray_generators.py:35-64): a regular grid on the z = z_min face of the box (``int(dx/dz*n)`` x ``int(dy/dz*n)``
    points, ``torch.linspace`` + ij-meshgrid order) and the common ray direction / length.  Returns (origins [M,3],
    direction [3], far).  The reference's quirks are kept: the ray length is ``sign(z_max)*|z_min| + |z_max|`` (= z_max - z_min
    only when the box straddles z = 0)."""
    c = aabb_corners(aabb)
    c1, c2, c3, c4 = c[0], c[1], c[2], c[-1]
    ext = (c.max(dim=0).values - c.min(dim=0).values).abs()
    const_axis = int(torch.argmax(((c1 == c2) & (c2 == c3)).to(torch.int)))
    ax_x = int(torch.argmax((c1 - c2).abs()))
    ax_y = int(torch.argmax((c1 - c3).abs()))
    x = torch.linspace(float(c1[ax_x]), float(c2[ax_x]), int(ext[0] / ext[const_axis] * num_points_per_side), dtype=torch.float32)
    y = torch.linspace(float(c1[ax_y]), float(c3[ax_y]), int(ext[1] / ext[const_axis] * num_points_per_side), dtype=torch.float32)
    xx, yy = torch.meshgrid(x, y, indexing="ij")
    origins = torch.column_stack((xx.flatten(), yy.flatten(), torch.full_like(xx.flatten(), float(c3[const_axis]))))
    plane = torch.tensor([0.0, 0.0, float(torch.sign(c4[const_axis]) * c1[const_axis].abs() + c4[const_axis].abs())])
    far = float(torch.linalg.norm(plane))
    direction = torch.nn.functional.normalize(plane[None])[0]
    return origins, direction, far


def volume_face_grid(aabb, num_points_per_side: int) -> Dict[str, float]:
    """The parameters of :func:`volume_surface_rays`'s grid (same quirks), for the device generator ``cnb_volume_face_rays``."""
    c = aabb_corners(aabb)
    c1, c2, c3, c4 = c[0], c[1], c[2], c[-1]
    ext = (c.max(dim=0).values - c.min(dim=0).values).abs()
    const_axis = int(torch.argmax(((c1 == c2) & (c2 == c3)).to(torch.int)))
    ax_x = int(torch.argmax((c1 - c2).abs()))
    ax_y = int(torch.argmax((c1 - c3).abs()))
    plane = torch.tensor([0.0, 0.0, float(torch.sign(c4[const_axis]) * c1[const_axis].abs() + c4[const_axis].abs())])
    direction = torch.nn.functional.normalize(plane[None])[0]
    return {"x0": float(c1[ax_x]), "x1": float(c2[ax_x]), "nx": int(ext[0] / ext[const_axis] * num_points_per_side),
            "y0": float(c1[ax_y]), "y1": float(c3[ax_y]), "ny": int(ext[1] / ext[const_axis] * num_points_per_side),
            "z": float(c3[const_axis]), "direction": [float(v) for v in direction.tolist()], "far": float(torch.linalg.norm(plane))}


def volume_face_rays_device(grid: Dict[str, float], first: int, n: int, device) -> RayBundle:
    """Rays ``first .. first + n`` of the export face (``OrthographicRayGenerator``, components/ray_generators.py:46-66) written by one
    kernel: origins on the grid (bit-equal to ``torch.linspace`` + ij-meshgrid), the common direction, nears = 0, fars = ray length."""
    import ctypes as C

    from . import _lib as L

    dev = torch.device(device)
    if dev.type != "cuda":
        raise RuntimeError("cropnerf_b200.volume_face_rays_device runs on CUDA devices only; there is no CPU fallback")
    o = torch.empty((n, 3), device=dev)
    d = torch.empty((n, 3), device=dev)
    nears = torch.empty((n, 1), device=dev)
    fars = torch.empty((n, 1), device=dev)
    direction = (C.c_float * 3)(*grid["direction"])
    L.check(L.lib().cnb_volume_face_rays(grid["x0"], grid["x1"], grid["nx"], grid["y0"], grid["y1"], grid["ny"], grid["z"], direction, grid["far"],
                                         int(first), int(n), o.data_ptr(), d.data_ptr(), nears.data_ptr(), fars.data_ptr(), L.stream_ptr(dev)),
            "volume_face_rays")
    return RayBundle(origins=o, directions=d, pixel_area=torch.zeros((n, 1), device=dev), camera_indices=None, nears=nears, fars=fars)


def sample_volume(model, aabb, num_points_per_side: int, num_rays_per_batch: int = 512, rank: int = 0, world_size: int = 1,
                  semantic_threshold: float = 3.0, density_threshold: float = 70.0, colormap_threshold: float = 0.999) -> Dict[str, Dict[str, Tensor]]:
    """The render loop of ``sample_volume`` (export/exporter_utils.py:88-172) for a model in ``test_mode='export'`` after
    ``setup_inference`` (uniform sampler, contraction off): orthographic rays from the z_min face, ``num_inference_samples``
    field evaluations per ray (no compositing), per-SAMPLE thresholds ``semantic >= 3``, ``density >= 70``,
    ``semantics_colormap >= 0.999``.  The rays of the face are split across ranks by contiguous range, no communication.
    Thresholding and compaction run on the device; only kept points are copied to the host.  Returns the three clouds of the
    reference -- ``semantic_colormap``, ``semantic``, ``density`` -- as {'points' [n,3], 'colors' [n,4] = (rgb, sigmoid(.))};
    the open3d rescaling / PLY writing that follows in the reference is :func:`rescale_to_dataparser` + :func:`write_ply`."""
    if model.test_mode != "export":
        raise RuntimeError("sample_volume needs a model built with test_mode='export' and setup_inference() applied (scripts/exporter.py:88-91)")
    dev = model.device
    grid = volume_face_grid(aabb, num_points_per_side)
    total = grid["nx"] * grid["ny"]
    lo, hi = shard_range(total, rank, world_size)
    clouds = {k: {"points": [], "colors": []} for k in ("semantic_colormap", "semantic", "density")}
    n_samples = 0
    for start in range(lo, hi, num_rays_per_batch):
        n = min(num_rays_per_batch, hi - start)
        rb = volume_face_rays_device(grid, start, n, dev)   # OrthographicRayGenerator batch, generated on the device
        with torch.no_grad():
            out = model(rb)
        pts = out["point_location"].reshape(-1, 3)
        sem = out["semantics"].reshape(-1)
        den = out["density"].reshape(-1)
        rgb = out["rgb"].reshape(-1, 3)
        label = out["semantics_colormap"].reshape(-1).to(sem.dtype)
        n_samples += int(sem.shape[0])
        m_den = den >= density_threshold
        m_sem = (sem >= semantic_threshold) & m_den
        m_cm = (label >= colormap_threshold) & m_den
        for key, mask, alpha in (("semantic_colormap", m_cm, torch.sigmoid(sem)), ("semantic", m_sem, torch.sigmoid(sem)), ("density", m_den, torch.sigmoid(den))):
            idx = torch.nonzero(mask)[:, 0]
            clouds[key]["points"].append(pts[idx].cpu())
            clouds[key]["colors"].append(torch.cat([rgb[idx], alpha[idx, None]], dim=-1).cpu())
    result = {}
    for key, parts in clouds.items():
        result[key] = {"points": torch.cat(parts["points"]) if parts["points"] else torch.empty((0, 3)),
                       "colors": torch.cat(parts["colors"]) if parts["colors"] else torch.empty((0, 4))}
    result["stats"] = {"rays": int(hi - lo), "samples": n_samples}
    return result


def rescale_to_dataparser(points: Tensor, dataparser_scale: float) -> Tensor:
    """``pcd.scale(1/scale).scale(2)`` about the origin (export/exporter_utils.py:186-193): back to the capture's metric frame."""
    return points * (2.0 / float(dataparser_scale))
