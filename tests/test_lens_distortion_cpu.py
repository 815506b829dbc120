"""CPU tests for lens distortion in ray generation: the restated nerfstudio undistortion (tests/lens_reference.py) converges and
agrees with OpenCV, zero / absent distortion leaves the oracle's rays untouched, nerfstudio ``Cameras`` are converted and
non-perspective ones refused, and the ctypes ``Lens`` mirrors ``cnb_lens``."""
import os
import subprocess
import tempfile
from types import SimpleNamespace

import ctypes as C
import cv2
import numpy as np
import pytest
import torch

import lens_reference as lr
from helpers import ROOT

from cropnerf_b200 import _lib as L
from cropnerf_b200 import export
from oracle import nerfstudio_torch as ns

FULL = [-0.12, 0.03, -0.004, 0.0005, 1e-3, -5e-4]   # k1, k2, k3, k4, p1, p2


def _normalised_grid(dtype, w=1920, h=1080, f=1000.0, step=37):
    """(x, -y) of pixel centres of a w x h camera (principal point at the centre), the four corners included."""
    xs = torch.cat([torch.arange(0, w, step, dtype=dtype), torch.tensor([w - 1], dtype=dtype)]) + 0.5
    ys = torch.cat([torch.arange(0, h, step, dtype=dtype), torch.tensor([h - 1], dtype=dtype)]) + 0.5
    yy, xx = torch.meshgrid(ys, xs, indexing="ij")
    return torch.stack([(xx - w / 2) / f, -(yy - h / 2) / f], -1).reshape(-1, 2)


def test_undistort_converges_to_the_forward_model_inverse():
    pts = _normalised_grid(torch.float64)
    corners = [pts[0], pts[-1]]
    assert abs(float(corners[0][0])) > 0.95 and abs(float(corners[0][1])) > 0.53
    params = torch.tensor(FULL, dtype=torch.float64)
    und = lr.radial_and_tangential_undistort(pts, params)
    assert (und - pts).abs().max() > 1e-2, "the lens must move the border pixels"
    back = lr.distort(und, params)
    assert (back - pts).abs().max() <= 1e-6


def test_undistort_matches_opencv_for_radial_lenses():
    """Radial-only lenses are symmetric under nerfstudio's y flip, so OpenCV's iterative undistortion of (x, y) is the flip of the
    reference's undistortion of (x, -y)."""
    pts = _normalised_grid(torch.float64)
    for k1, k2, k3 in ((-0.12, 0.03, -0.004), (0.08, -0.02, 0.003), (-0.25, 0.06, 0.0)):
        params = torch.tensor([k1, k2, k3, 0.0, 0.0, 0.0], dtype=torch.float64)
        ref = lr.radial_and_tangential_undistort(pts, params).numpy()
        src = np.stack([pts[:, 0].numpy(), -pts[:, 1].numpy()], -1)[:, None, :]
        crit = (cv2.TERM_CRITERIA_COUNT | cv2.TERM_CRITERIA_EPS, 200, 1e-15)
        got = cv2.undistortPointsIter(src, np.eye(3), np.array([k1, k2, 0.0, 0.0, k3]), np.eye(3), np.eye(3), crit)[:, 0, :]
        assert np.abs(got[:, 0] - ref[:, 0]).max() <= 1e-5
        assert np.abs(-got[:, 1] - ref[:, 1]).max() <= 1e-5


def test_zero_lens_is_the_identity_bit_for_bit():
    pts = _normalised_grid(torch.float32)
    assert torch.equal(lr.radial_and_tangential_undistort(pts, torch.zeros(6)), pts)


def test_no_or_zero_distortion_gives_todays_rays():
    g = torch.Generator().manual_seed(3)
    q, _ = torch.linalg.qr(torch.randn(3, 3, generator=g))
    c2w = torch.cat([q, torch.rand(3, 1, generator=g)], 1)
    coords = torch.stack([torch.randint(0, 61, (300,), generator=g), torch.randint(0, 97, (300,), generator=g)], -1).float() + 0.5
    want = ns.generate_pinhole_rays(c2w, 80.0, 82.0, 48.5, 30.25, coords)
    for dist in (None, torch.zeros(6)):
        got = lr.generate_pinhole_rays(c2w, 80.0, 82.0, 48.5, 30.25, coords, distortion_params=dist)
        assert all(torch.equal(a, b) for a, b in zip(got, want))
    lensed = lr.generate_pinhole_rays(c2w, 80.0, 82.0, 48.5, 30.25, coords, distortion_params=torch.tensor(FULL))
    assert (lensed[1] - want[1]).abs().max() > 1e-3

    n, h, w = 3, 6, 8
    images = torch.rand((n, h, w, 3), generator=g)
    masks = (torch.rand((n, h, w), generator=g) < 0.3).float()
    c2ws = torch.stack([c2w] * n)
    fx, fy = torch.tensor([10.0, 11.0, 12.0]), torch.tensor([11.0, 10.5, 10.0])
    cx, cy = torch.full((n,), w / 2.0), torch.full((n,), h / 2.0)
    rand3 = torch.rand((64, 3), generator=g)
    want = ns.next_train_batch(rand3, images, masks, c2ws, fx, fy, cx, cy)
    for dist in (None, torch.zeros(n, 6)):
        got = lr.next_train_batch(rand3, images, masks, c2ws, fx, fy, cx, cy, distortion_params=dist)
        assert all(torch.equal(a, b) for a, b in zip(got, want))


def test_train_batch_reference_undistorts_each_ray_with_its_camera():
    g = torch.Generator().manual_seed(4)
    n, h, w = 3, 6, 8
    c2w = torch.zeros(n, 3, 4)
    for i in range(n):
        c2w[i, :, :3] = torch.linalg.qr(torch.randn(3, 3, generator=g))[0]
    fx, fy = torch.tensor([5.0, 6.0, 7.0]), torch.tensor([6.0, 5.5, 5.0])
    cx, cy = torch.full((n,), w / 2.0), torch.full((n,), h / 2.0)
    dist = torch.tensor([FULL, [0.0] * 6, [0.05, 0.0, 0.0, 0.0, 0.0, 2e-3]])
    rand3 = torch.rand((40, 3), generator=g)
    idx, o, d, area, _, _ = lr.next_train_batch(rand3, torch.zeros((n, h, w, 3)), None, c2w, fx, fy, cx, cy, distortion_params=dist)
    for i in range(rand3.shape[0]):
        c, y, x = idx[i].tolist()
        _, d1, a1 = lr.generate_pinhole_rays(c2w[c], float(fx[c]), float(fy[c]), float(cx[c]), float(cy[c]), torch.tensor([[y + 0.5, x + 0.5]]),
                                             distortion_params=dist[c])
        assert torch.equal(d1[0], d[i]) and torch.equal(a1[0], area[i])


def _ns_cameras(n=4, camera_type=None, dist=True):
    """A stand-in for nerfstudio's Cameras with its attribute names and shapes."""
    g = torch.Generator().manual_seed(5)
    c2w = torch.rand((n, 3, 4), generator=g)
    col = lambda v: torch.full((n, 1), v)  # noqa: E731
    return SimpleNamespace(camera_to_worlds=c2w, fx=col(900.0) + torch.arange(n)[:, None], fy=col(905.0), cx=col(640.0), cy=col(360.0),
                           width=torch.full((n, 1), 1280, dtype=torch.int64), height=torch.full((n, 1), 720, dtype=torch.int64),
                           distortion_params=torch.rand((n, 6), generator=g) * 0.01 if dist else None,
                           camera_type=torch.ones((n, 1), dtype=torch.int64) if camera_type is None else camera_type)


def test_cameras_from_nerfstudio():
    ns_cams = _ns_cameras()
    cams = export.cameras_from_nerfstudio(ns_cams)
    assert len(cams) == 4
    for i, cam in enumerate(cams):
        assert torch.equal(cam.c2w, ns_cams.camera_to_worlds[i])
        assert (cam.fx, cam.fy, cam.cx, cam.cy, cam.width, cam.height) == (900.0 + i, 905.0, 640.0, 360.0, 1280, 720)
        assert torch.equal(cam.distortion_params, ns_cams.distortion_params[i])
    assert all(c.distortion_params is None for c in export.cameras_from_nerfstudio(_ns_cameras(dist=False)))
    # one row of a Cameras batch (cameras[i]): [3,4] pose, [1] intrinsics, [6] distortion
    row = SimpleNamespace(**{k: (v[1] if v is not None else None) for k, v in vars(ns_cams).items()})
    one = export.cameras_from_nerfstudio(row)
    assert len(one) == 1 and one[0].fx == 901.0 and torch.equal(one[0].distortion_params, ns_cams.distortion_params[1])


@pytest.mark.parametrize("type_value,name", [(2, "FISHEYE"), (3, "EQUIRECTANGULAR"), (8, "ORTHOPHOTO"), (9, "FISHEYE624")])
def test_non_perspective_cameras_are_refused(type_value, name):
    ct = torch.ones((4, 1), dtype=torch.int64)
    ct[2] = type_value
    with pytest.raises(ValueError, match=name):
        export.cameras_from_nerfstudio(_ns_cameras(camera_type=ct))
    fisheye = SimpleNamespace(camera_type=type_value, **vars(export.PinholeCamera(torch.eye(3, 4), 10.0, 10.0, 4.0, 3.0, 8, 6)))
    with pytest.raises(ValueError, match=name):   # checked before any rendering: no model or GPU is reached
        export.project_clusters(None, [fisheye], [{"aabb": np.zeros((1, 2, 3), np.float32)}], None)
    with pytest.raises(ValueError, match=name):
        export.project_clusters(None, _ns_cameras(camera_type=ct), [], None)


def test_cameras_from_nerfstudio_refuses_bad_shapes():
    bad = _ns_cameras()
    bad.camera_to_worlds = torch.zeros((4, 4, 4))
    with pytest.raises(ValueError, match="camera_to_worlds"):
        export.cameras_from_nerfstudio(bad)
    bad = _ns_cameras()
    bad.fx = torch.full((4,), 900.0)
    with pytest.raises(ValueError, match="fx"):
        export.cameras_from_nerfstudio(bad)
    bad = _ns_cameras()
    bad.distortion_params = torch.zeros((4, 4))
    with pytest.raises(ValueError, match="distortion_params"):
        export.cameras_from_nerfstudio(bad)
    bad = _ns_cameras()
    bad.camera_type = torch.ones((3, 1), dtype=torch.int64)
    with pytest.raises(ValueError, match="camera_type"):
        export.cameras_from_nerfstudio(bad)
    with pytest.raises(ValueError, match="6 values"):
        export.lens_values(torch.zeros(5))


def test_pinhole_camera_keeps_its_seven_positional_fields():
    cam = export.PinholeCamera(torch.eye(3, 4), 10.0, 11.0, 4.0, 3.0, 8, 6)
    assert (cam.fx, cam.fy, cam.cx, cam.cy, cam.width, cam.height) == (10.0, 11.0, 4.0, 3.0, 8, 6)
    assert cam.distortion_params is None
    assert export._lens_struct(cam.distortion_params) is None
    lens = export._lens_struct(torch.tensor(FULL))
    assert [lens.k1, lens.k2, lens.k3, lens.k4, lens.p1, lens.p2] == torch.tensor(FULL).tolist()


def test_lens_struct_matches_c_compiler():
    prog = r"""
#include <stddef.h>
#include <stdio.h>
#include "cropnerf_b200.h"
int main(void){ printf("%zu %zu %zu %zu\n", sizeof(cnb_lens), offsetof(cnb_lens, k4), offsetof(cnb_lens, p2), sizeof(cnb_camera)); return 0; }
"""
    with tempfile.TemporaryDirectory() as d:
        src = os.path.join(d, "s.c")
        open(src, "w").write(prog)
        exe = os.path.join(d, "s")
        subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), src, "-o", exe])
        sizes = [int(v) for v in subprocess.check_output([exe]).split()]
    assert sizes == [C.sizeof(L.Lens), L.Lens.k4.offset, L.Lens.p2.offset, C.sizeof(L.Camera)] == [24, 12, 20, 72]


def test_lens_entries_refuse_bad_arguments_without_a_device():
    if torch.cuda.is_available():
        pytest.skip("CUDA present")
    lib = L.lib()
    assert lib.cnb_generate_rays_lens(None, None, None, 4, None, None, None, None, None, None, None, None) != 0
    assert b"generate_rays" in lib.cnb_last_error()
    assert lib.cnb_sample_train_batch_lens(None, None, None, 16, None, None, None, None, None, None, None, None) != 0
    assert b"sample_train_batch" in lib.cnb_last_error()
