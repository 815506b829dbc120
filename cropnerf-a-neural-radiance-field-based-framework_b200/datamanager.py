"""Device-resident training batches: ``FruitDataManager.next_train`` (``data/fruit_datamanager.py:188-197``) in one kernel.

The reference draws a batch as ``batch = train_pixel_sampler.sample(image_batch)`` (nerfstudio ``PixelSampler``: random
``(camera, y, x)`` indices, then ``value[c, y, x]`` of the image and the fruit mask on the HOST copy of all images) followed by
``ray_bundle = train_ray_generator(batch["indices"])`` (nerfstudio ``RayGenerator``: pixel centres -> ``Cameras.generate_rays``).
Here the images of the split stay in HBM (uint8 RGB: 300 x 1080p = 1.9 GB, masks 0.6 GB) and ``cnb_sample_train_batch``
(``csrc/train_batch.cu``) does index -> pixel gather -> per-camera pinhole ray -> pixel area, one thread per ray, writing exactly
the tensors the training step reads.  SURVEY.md section 8, "next" row f1 (pixel sampler).  Cameras with OPENCV lens distortion
(nerfstudio ``distortion_params``) get nerfstudio's undistortion in the same kernel (``cnb_sample_train_batch_lens``).

Parity: ``tests/test_train_batch_gpu.py`` (indices and gathered pixels bit-exact against the oracle, uint8 and float32 storage);
``bench.py``'s end-to-end leg ``e2e_device_batches`` trains from it (images resident in HBM, no host ray traffic at all).
"""
from __future__ import annotations

import ctypes as C
from typing import Dict, Optional, Sequence, Tuple

import torch
from torch import Tensor

from . import _lib as L
from .export import cameras_from_nerfstudio, check_perspective, lens_values
from .rays import RayBundle


class DeviceTrainBatches:
    """``next_train(step) -> (RayBundle, batch)`` with nerfstudio's batch keys (``image``, ``fruit_mask``, ``indices``).

    ``images``: ``[N,H,W,3]`` uint8 (value / 255 is the float image ``cotton_dataset.py`` produces) or float32; ``fruit_masks``:
    ``[N,H,W]`` uint8 / bool (non-zero = fruit) or None.  ``cameras``: either N objects with ``c2w`` ``[3,4]``, ``fx, fy, cx, cy``
    and optionally ``distortion_params`` (6 values, nerfstudio order) and ``camera_type`` (``export.PinholeCamera``), or a
    nerfstudio ``Cameras`` batch of N cameras, which is read through ``export.cameras_from_nerfstudio`` (``camera_to_worlds``,
    intrinsics, ``distortion_params``, ``camera_type``).  Only perspective cameras are accepted; any other ``camera_type`` raises
    ``ValueError``.  If some camera has non-zero distortion, the ``[N,6]`` parameters are uploaded once here and every batch is
    undistorted as nerfstudio's ``RayGenerator`` does.  ``rand_fn(shape, device)`` is injectable so that tests feed the oracle
    the same numbers; default ``torch.rand`` on the device with this object's generator."""

    def __init__(self, images: Tensor, fruit_masks: Optional[Tensor], cameras: Sequence, num_rays_per_batch: int = 4096, device="cuda",
                 seed: int = 0, rand_fn=None):
        dev = torch.device(device)
        if dev.type != "cuda":
            raise RuntimeError("cropnerf_b200.DeviceTrainBatches runs on CUDA devices only; there is no CPU fallback")
        if images.dim() != 4 or images.shape[-1] != 3 or images.dtype not in (torch.uint8, torch.float32):
            raise ValueError(f"images must be [N,H,W,3] uint8 or float32, got {tuple(images.shape)} {images.dtype}")
        n, h, w = images.shape[:3]
        if hasattr(cameras, "camera_to_worlds"):         # a nerfstudio Cameras batch
            cameras = cameras_from_nerfstudio(cameras)
        if len(cameras) != n:
            raise ValueError(f"{len(cameras)} cameras for {n} images")
        self.device = dev
        self.images = images.to(dev).contiguous()
        self.masks = None
        if fruit_masks is not None:
            if tuple(fruit_masks.shape) != (n, h, w):
                raise ValueError(f"fruit_masks must be [N,H,W] = {(n, h, w)}, got {tuple(fruit_masks.shape)}")
            self.masks = (fruit_masks != 0).to(dev, torch.uint8).contiguous()
        cam_host = (L.Camera * n)()
        lenses = torch.zeros((n, 6), dtype=torch.float32)
        for i, cam in enumerate(cameras):
            check_perspective(getattr(cam, "camera_type", None), "DeviceTrainBatches")
            dist = lens_values(getattr(cam, "distortion_params", None))
            if dist is not None:
                lenses[i] = torch.tensor(dist, dtype=torch.float32)
            m = torch.as_tensor(cam.c2w).detach().cpu().float().reshape(-1)[:12].tolist()
            for k in range(12):
                cam_host[i].c2w[k] = m[k]
            cam_host[i].fx, cam_host[i].fy, cam_host[i].cx, cam_host[i].cy = float(cam.fx), float(cam.fy), float(cam.cx), float(cam.cy)
            cam_host[i].width, cam_host[i].height = int(w), int(h)
        raw = torch.frombuffer(bytearray(bytes(cam_host)), dtype=torch.uint8)
        self._cameras = raw.to(dev)                      # device array of cnb_camera records (72 bytes each)
        # device array of cnb_lens records [N,6], only when some camera is distorted (otherwise the pinhole kernel runs)
        self._lenses = lenses.to(dev) if bool((lenses != 0).any()) else None
        self.num_rays_per_batch = int(num_rays_per_batch)
        self.generator = torch.Generator(device=dev)
        self.generator.manual_seed(int(seed))
        self.rand_fn = rand_fn
        self.train_count = 0
        self._set = L.ImageSet()
        self._set.images_u8 = self.images.data_ptr() if self.images.dtype == torch.uint8 else None
        self._set.images_f32 = self.images.data_ptr() if self.images.dtype == torch.float32 else None
        self._set.masks_u8 = self.masks.data_ptr() if self.masks is not None else None
        self._set.cameras = self._cameras.data_ptr()
        self._set.num_images, self._set.height, self._set.width = int(n), int(h), int(w)

    def next_train(self, step: int) -> Tuple[RayBundle, Dict[str, Tensor]]:
        """``FruitDataManager.next_train`` (fruit_datamanager.py:188-197)."""
        self.train_count += 1
        R, dev = self.num_rays_per_batch, self.device
        if self.rand_fn is not None:
            rand3 = self.rand_fn((R, 3), dev).to(dev, torch.float32).contiguous()
        else:
            rand3 = torch.rand((R, 3), device=dev, dtype=torch.float32, generator=self.generator)
        indices = torch.empty((R, 3), device=dev, dtype=torch.int32)
        origins = torch.empty((R, 3), device=dev, dtype=torch.float32)
        directions = torch.empty((R, 3), device=dev, dtype=torch.float32)
        pixel_area = torch.empty((R, 1), device=dev, dtype=torch.float32)
        camera_indices = torch.empty((R, 1), device=dev, dtype=torch.int32)
        image = torch.empty((R, 3), device=dev, dtype=torch.float32)
        fruit_mask = torch.empty((R, 1), device=dev, dtype=torch.float32)
        if self._lenses is None:
            L.check(L.lib().cnb_sample_train_batch(C.byref(self._set), rand3.data_ptr(), R, indices.data_ptr(), origins.data_ptr(), directions.data_ptr(),
                                                   pixel_area.data_ptr(), camera_indices.data_ptr(), image.data_ptr(), fruit_mask.data_ptr(),
                                                   L.stream_ptr(dev)), "sample_train_batch")
        else:
            L.check(L.lib().cnb_sample_train_batch_lens(C.byref(self._set), self._lenses.data_ptr(), rand3.data_ptr(), R, indices.data_ptr(),
                                                        origins.data_ptr(), directions.data_ptr(), pixel_area.data_ptr(), camera_indices.data_ptr(),
                                                        image.data_ptr(), fruit_mask.data_ptr(), L.stream_ptr(dev)), "sample_train_batch_lens")
        bundle = RayBundle(origins=origins, directions=directions, pixel_area=pixel_area, camera_indices=camera_indices)
        return bundle, {"image": image, "fruit_mask": fruit_mask, "indices": indices}
