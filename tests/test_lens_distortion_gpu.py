"""GPU parity of lens distortion in the three device ray generators (cnb_generate_rays_lens, cnb_sample_train_batch_lens,
cnb_generate_rays_boxes_lens; csrc/lens.cuh) against the reference's undistortion (tests/lens_reference.py), with the bounds of
the pinhole tests: test_generate_rays_and_aabb_clip, test_device_train_batch_matches_oracle,
test_generate_rays_boxes_equals_one_box_at_a_time and test_project_clusters_png_tree_matches_oracle."""
import ctypes as C
import os
from types import SimpleNamespace

import cv2
import numpy as np
import pytest
import torch

import lens_reference as lr
from helpers import assert_close, product_model

from cropnerf_b200 import _lib as L
from cropnerf_b200 import engine, export, synthetic
from oracle import cases
from oracle import nerfstudio_torch as ns

pytestmark = pytest.mark.gpu

FULL = torch.tensor([-0.12, 0.03, -0.004, 0.0005, 1e-3, -5e-4])   # k1, k2, k3, k4, p1, p2


@pytest.mark.parametrize("with_aabb", [False, True])
def test_generate_rays_lens_matches_oracle(dev, with_aabb):
    W, H = 97, 61
    c2w = synthetic.make_cameras(5, seed=3)[2]
    fx, fy, cx, cy = 80.0, 82.0, 48.5, 30.25
    aabb = torch.tensor([[-0.3, -0.2, -0.25], [0.2, 0.3, 0.15]])
    yy, xx = torch.meshgrid(torch.arange(H), torch.arange(W), indexing="ij")
    coords = torch.stack([yy, xx], -1).reshape(-1, 2).float() + 0.5
    o_ref, d_ref, a_ref = lr.generate_pinhole_rays(c2w, fx, fy, cx, cy, coords, distortion_params=FULL)
    if with_aabb:
        rb, cnt = export.generate_rays(c2w, fx, fy, cx, cy, W, H, dev, aabb=aabb, count_valid=True, distortion_params=FULL)
    else:
        rb = export.generate_rays(c2w, fx, fy, cx, cy, W, H, dev, distortion_params=FULL)
        assert rb.nears is None
    assert_close(rb.origins, o_ref, 1e-6, "origins")
    assert_close(rb.directions, d_ref, 2e-6, "directions", floor=1e-2)
    assert_close(rb.pixel_area, a_ref, 2e-3, "pixel_area", floor=1e-9)
    assert torch.allclose(rb.directions.norm(dim=-1).cpu(), torch.ones(rb.directions.shape[0]), atol=1e-5)
    pinhole = export.generate_rays(c2w, fx, fy, cx, cy, W, H, dev, aabb=aabb if with_aabb else None)
    assert (rb.directions - pinhole.directions).abs().max().item() > 1e-2, "the lens must visibly move the border rays"
    if with_aabb:
        tmin, tmax = ns.intersect_aabb(o_ref, d_ref, aabb.reshape(-1))
        hit_ref = tmin < 1e10
        hit = rb.nears[:, 0].cpu() < 1e10
        assert (hit == hit_ref).float().mean().item() >= 0.999
        both = hit & hit_ref
        assert both.sum() > 50, "test scene should hit the box"
        assert_close(rb.nears[:, 0].cpu()[both], tmin[both], 1e-4, "nears", floor=1e-2)
        assert_close(rb.fars[:, 0].cpu()[both], tmax[both], 1e-4, "fars", floor=1e-2)
        assert int(cnt.item()) == int(hit.sum().item())
    # a zero lens is the pinhole kernel, bit for bit
    zero = export.generate_rays(c2w, fx, fy, cx, cy, W, H, dev, aabb=aabb if with_aabb else None, distortion_params=torch.zeros(6))
    for name in ("origins", "directions", "pixel_area", "nears", "fars"):
        a, b = getattr(zero, name), getattr(pinhole, name)
        assert (a is None and b is None) or torch.equal(a, b), name


def test_generate_rays_lens_pixel_list_and_no_pixel_area(dev):
    """Given pixels, and without a pixel_area output (the offsets are then not undistorted): the same rays as the full image."""
    W, H = 97, 61
    c2w = synthetic.make_cameras(5, seed=3)[1]
    cam = export.PinholeCamera(c2w, 80.0, 82.0, 48.5, 30.25, W, H)
    full = export.generate_rays(c2w, cam.fx, cam.fy, cam.cx, cam.cy, W, H, dev, distortion_params=FULL)
    g = torch.Generator().manual_seed(1)
    pix = torch.stack([torch.randint(0, H, (500,), generator=g), torch.randint(0, W, (500,), generator=g)], -1)
    sub = export.generate_rays(c2w, cam.fx, cam.fy, cam.cx, cam.cy, W, H, dev, pixel_yx=pix, distortion_params=FULL)
    flat = (pix[:, 0] * W + pix[:, 1]).to(dev)
    assert torch.equal(sub.directions, full.directions[flat]) and torch.equal(sub.pixel_area, full.pixel_area[flat])
    cs = export._camera_struct(cam)
    lens = export._lens_struct(FULL)
    n = W * H
    o = torch.empty((n, 3), device=dev)
    d = torch.empty((n, 3), device=dev)
    L.check(L.lib().cnb_generate_rays_lens(C.byref(cs), C.byref(lens), None, n, None, o.data_ptr(), d.data_ptr(), None, None, None, None,
                                           L.stream_ptr(dev)), "generate_rays_lens")
    assert torch.equal(d, full.directions) and torch.equal(o, full.origins)


def _train_scene(n, h, w, g):
    c2w = torch.zeros(n, 3, 4)
    for i in range(n):
        q, _ = torch.linalg.qr(torch.randn(3, 3, generator=g))
        c2w[i, :, :3] = q
        c2w[i, :, 3] = torch.rand(3, generator=g) - 0.5
    fx = torch.full((n,), 72.0) + torch.arange(n)
    fy = torch.full((n,), 71.0) - torch.arange(n) * 0.5
    cx, cy = torch.full((n,), w / 2.0), torch.full((n,), h / 2.0)
    return c2w, fx, fy, cx, cy


@pytest.mark.parametrize("storage", ["uint8", "float32"])
def test_device_train_batch_with_lenses_matches_oracle(storage):
    from cropnerf_b200.datamanager import DeviceTrainBatches

    g = torch.Generator().manual_seed(0)
    n, h, w, R = 7, 54, 96, 4096
    images = torch.randint(0, 256, (n, h, w, 3), generator=g, dtype=torch.uint8)
    masks = (torch.rand((n, h, w), generator=g) < 0.1).to(torch.uint8)
    c2w, fx, fy, cx, cy = _train_scene(n, h, w, g)
    dist = torch.zeros(n, 6)
    dist[0] = FULL
    dist[2] = torch.tensor([0.2, -0.05, 0.0, 0.0, 0.0, 0.0])
    dist[3] = torch.tensor([0.0, 0.0, 0.0, 0.0, 3e-3, -2e-3])
    dist[5] = FULL * 1.5
    rand3 = torch.rand((R, 3), generator=g)
    rand3[0] = torch.tensor([0.0, 0.0, 0.0])
    rand3[1] = torch.tensor([1.0 - 2.0**-24] * 3)
    cams = [export.PinholeCamera(c2w[i], float(fx[i]), float(fy[i]), float(cx[i]), float(cy[i]), w, h, distortion_params=dist[i]) for i in range(n)]
    fimg = images.float() / 255.0
    dm = DeviceTrainBatches(images if storage == "uint8" else fimg, masks, cams, num_rays_per_batch=R, device="cuda:0",
                            rand_fn=lambda shape, dev: rand3.to(dev))
    assert dm._lenses is not None
    bundle, batch = dm.next_train(0)
    torch.cuda.synchronize()
    idx, o, d, area, img, m = lr.next_train_batch(rand3, fimg, masks.float(), c2w, fx, fy, cx, cy, distortion_params=dist)
    idx = torch.minimum(idx, torch.tensor([n - 1, h - 1, w - 1]))
    assert torch.equal(batch["indices"].cpu().long(), idx)
    assert torch.equal(bundle.camera_indices.cpu().long()[:, 0], idx[:, 0])
    assert torch.equal(batch["image"].cpu(), fimg[idx[:, 0], idx[:, 1], idx[:, 2]])
    assert torch.equal(batch["fruit_mask"].cpu()[:, 0], masks.float()[idx[:, 0], idx[:, 1], idx[:, 2]])
    assert torch.equal(bundle.origins.cpu(), c2w[idx[:, 0]][:, :3, 3])
    keep = (idx == ns.pixel_sampler_indices(rand3, n, h, w)).all(-1)
    got_d, got_a = bundle.directions.cpu()[keep], bundle.pixel_area.cpu()[keep]
    d, area = d[keep], area[keep]
    assert (got_d - d).abs().max() <= 2e-6
    assert ((got_a - area).abs() <= 2e-3 * area.abs() + 1e-12).all()
    # the lens is applied to the distorted cameras only
    _, _, d_pin, _, _, _ = ns.next_train_batch(rand3, fimg, masks.float(), c2w, fx, fy, cx, cy)
    moved = (bundle.directions.cpu() - d_pin).abs().amax(-1)[keep]
    lensed = (dist != 0).any(-1)[idx[keep, 0]]
    assert moved[lensed].max() > 1e-2 and moved[~lensed].max() <= 2e-6
    # all-zero lenses: nothing is uploaded and the pinhole kernel runs
    cams0 = [export.PinholeCamera(c.c2w, c.fx, c.fy, c.cx, c.cy, w, h, distortion_params=torch.zeros(6)) for c in cams]
    dm0 = DeviceTrainBatches(images, masks, cams0, num_rays_per_batch=R, device="cuda:0", rand_fn=lambda shape, dev: rand3.to(dev))
    assert dm0._lenses is None


def test_device_batches_refuse_non_perspective_cameras():
    from cropnerf_b200.datamanager import DeviceTrainBatches

    images = torch.zeros((2, 6, 8, 3), dtype=torch.uint8)
    cams = [SimpleNamespace(camera_type=t, **vars(export.PinholeCamera(torch.eye(3, 4), 10.0, 10.0, 4.0, 3.0, 8, 6))) for t in (1, 2)]
    with pytest.raises(ValueError, match="FISHEYE"):
        DeviceTrainBatches(images, None, cams, device="cuda:0")


def test_generate_rays_boxes_lens_equals_one_box_at_a_time(dev):
    c2w = synthetic.make_cameras(2, seed=3)[1]
    lens = torch.tensor([-0.3, 0.08, -0.01, 0.0, 2e-3, -1e-3])
    cam = export.PinholeCamera(c2w=c2w, fx=70.0, fy=65.0, cx=40.0, cy=30.0, width=80, height=60, distortion_params=lens)
    boxes = torch.tensor([[-0.25, -0.2, -0.2, 0.15, 0.2, 0.25], [0.1, 0.1, 0.1, 0.4, 0.35, 0.3], [5.0, 5.0, 5.0, 5.1, 5.1, 5.1], [-0.25, -0.2, -0.2, 0.15, 0.2, 0.25]])
    k, npix = boxes.shape[0], 80 * 60
    cap = k * npix
    o = torch.empty((cap, 3), device=dev); d = torch.empty((cap, 3), device=dev); area = torch.empty((cap,), device=dev)
    nears = torch.empty((cap,), device=dev); fars = torch.empty((cap,), device=dev)
    tags = torch.empty((cap,), device=dev, dtype=torch.int32); count = torch.zeros((1,), device=dev, dtype=torch.int32)
    cs = export._camera_struct(cam)
    ls = export._lens_struct(lens)
    bd = boxes.to(dev)
    L.check(L.lib().cnb_generate_rays_boxes_lens(C.byref(cs), C.byref(ls), bd.data_ptr(), k, cap, o.data_ptr(), d.data_ptr(), area.data_ptr(),
                                                 nears.data_ptr(), fars.data_ptr(), tags.data_ptr(), count.data_ptr(), L.stream_ptr(dev)), "generate_rays_boxes_lens")
    n = int(count)
    order = torch.argsort(tags[:n])
    tg = tags[:n][order].cpu()
    got = {name: t[:n][order].cpu() for name, t in (("o", o), ("d", d), ("area", area), ("near", nears), ("far", fars))}
    expect_tags = []
    moved = False
    for b in range(k):
        rb = export.generate_rays(cam.c2w, cam.fx, cam.fy, cam.cx, cam.cy, cam.width, cam.height, dev, aabb=boxes[b], distortion_params=lens)
        valid = (rb.nears[:, 0] < 1e10).cpu()
        pix = torch.nonzero(valid)[:, 0]
        sel = (tg >= b * npix) & (tg < (b + 1) * npix)
        assert torch.equal(tg[sel] - b * npix, pix.to(torch.int32)), b
        assert torch.equal(got["d"][sel], rb.directions.cpu()[valid]) and torch.equal(got["o"][sel], rb.origins.cpu()[valid])
        assert torch.equal(got["near"][sel], rb.nears.cpu()[valid][:, 0]) and torch.equal(got["far"][sel], rb.fars.cpu()[valid][:, 0])
        assert torch.equal(got["area"][sel], rb.pixel_area.cpu()[valid][:, 0])
        expect_tags.append(pix.numel())
        pin = export.generate_rays(cam.c2w, cam.fx, cam.fy, cam.cx, cam.cy, cam.width, cam.height, dev, aabb=boxes[b])
        moved = moved or not torch.equal(valid, (pin.nears[:, 0] < 1e10).cpu())
    assert n == sum(expect_tags) and expect_tags[2] == 0 and expect_tags[0] == expect_tags[3] > 50
    assert moved, "the lens must change which pixels hit some box"
    # NULL or zero lens: the pinhole entry's output
    for zl in (None, C.byref(export._lens_struct(torch.zeros(6)))):
        count2 = torch.zeros((1,), device=dev, dtype=torch.int32)
        d2 = torch.empty_like(d)
        L.check(L.lib().cnb_generate_rays_boxes_lens(C.byref(cs), zl, bd.data_ptr(), k, cap, o.data_ptr(), d2.data_ptr(), area.data_ptr(),
                                                     nears.data_ptr(), fars.data_ptr(), tags.data_ptr(), count2.data_ptr(), L.stream_ptr(dev)), "boxes")
        n2 = int(count2)
        rb = export.generate_rays(cam.c2w, cam.fx, cam.fy, cam.cx, cam.cy, cam.width, cam.height, dev, aabb=boxes[0])
        hits0 = tags[:n2] < npix
        assert torch.equal(d2[:n2][hits0][torch.argsort(tags[:n2][hits0])], rb.directions[rb.nears[:, 0] < 1e10])


def _oracle_images(oracle, cam, box):
    H, W = cam.height, cam.width
    yy, xx = torch.meshgrid(torch.arange(H), torch.arange(W), indexing="ij")
    coords = torch.stack([yy, xx], -1).reshape(-1, 2).float() + 0.5
    o, d, area = lr.generate_pinhole_rays(cam.c2w, cam.fx, cam.fy, cam.cx, cam.cy, coords, distortion_params=cam.distortion_params)
    tmin, tmax = ns.intersect_aabb(o, d, torch.as_tensor(box, dtype=torch.float32).reshape(-1))
    valid = tmin < 1e10
    wo = torch.zeros((H * W, 3))
    vis = torch.zeros((H * W, 3))
    if int(valid.sum()) >= 10:
        rb = ns.RayBundle(origins=o[valid].contiguous(), directions=d[valid], pixel_area=area[valid], camera_indices=torch.zeros((int(valid.sum()), 1), dtype=torch.long),
                          nears=tmin[valid][:, None], fars=tmax[valid][:, None])
        with torch.no_grad():
            wo[valid] = oracle(rb)["semantics"].expand(-1, 3)
            rb.fars = rb.nears
            rb.nears = torch.zeros_like(rb.nears)
            front = torch.zeros(H * W)
            front[valid] = oracle.get_density_for_ray_bundle(rb)
        vis = wo.clone()
        vis[front >= 0.5] = 0.0
    return export.to_png_bytes(wo.view(H, W, 3)), export.to_png_bytes(vis.view(H, W, 3)), valid.view(H, W)


def test_project_clusters_with_lens_matches_oracle(dev, tmp_path):
    cfg = cases.make_config(dict(log2_hashmap_size=14))
    oracle, state = cases.build_oracle(cfg, 6, 0, 0.5)
    oracle.eval()
    model = product_model(cfg, state, 6, dev, False)
    c2ws = synthetic.make_cameras(3, seed=7)
    lenses = [torch.tensor([-0.3, 0.08, -0.01, 0.0, 2e-3, -1e-3]), torch.zeros(6), torch.tensor([0.25, 0.0, 0.0, 0.0, 0.0, 0.0])]
    # handed over as a nerfstudio Cameras batch (attribute names and shapes of nerfstudio's Cameras)
    ns_cams = SimpleNamespace(camera_to_worlds=c2ws, fx=torch.full((3, 1), 60.0), fy=torch.full((3, 1), 60.0), cx=torch.full((3, 1), 24.0),
                              cy=torch.full((3, 1), 18.0), width=torch.full((3, 1), 48), height=torch.full((3, 1), 36),
                              distortion_params=torch.stack(lenses), camera_type=torch.ones((3, 1), dtype=torch.int64))
    cams = export.cameras_from_nerfstudio(ns_cams)
    clusters = [
        {"aabb": np.array([[[-0.25, -0.2, -0.2], [0.15, 0.2, 0.25]], [[0.1, 0.1, 0.1], [0.4, 0.35, 0.3]]], dtype=np.float32), "pcd": {}},
        {"aabb": np.array([[[5.0, 5.0, 5.0], [5.1, 5.1, 5.1]]], dtype=np.float32), "pcd": {}},
    ]
    out_dir = str(tmp_path / "projection")
    st = export.project_clusters(model, ns_cams, clusters, out_dir)
    assert st["pairs"] == 6 and st["images"] == 2 * (2 * 3 + 1 * 3) and st["rays"] > 0
    n_checked, moved = 0, 0
    for k, cluster in enumerate(clusters):
        for j, cam in enumerate(cams):
            cam_dir = os.path.join(out_dir, f"super_cluster_{k}", f"cam_{j}")
            for i in range(cluster["aabb"].shape[0]):
                wo_ref, vis_ref, valid = _oracle_images(oracle, cam, cluster["aabb"][i])
                wo = cv2.imread(os.path.join(cam_dir, f"wo_occ_cluster_{i}.png"), cv2.IMREAD_COLOR)[..., ::-1]
                vis = cv2.imread(os.path.join(cam_dir, f"visible_cluster_{i}.png"), cv2.IMREAD_COLOR)[..., ::-1]
                assert wo.shape == (36, 48, 3)
                if k == 1:
                    assert not wo.any() and not vis.any() and not valid.any()
                    continue
                assert valid.sum() > 50, "test boxes should be on screen"
                assert (np.abs(wo.astype(int) - wo_ref.astype(int)) <= 1).mean() >= 0.995
                assert (np.abs(vis.astype(int) - vis_ref.astype(int)) <= 1).mean() >= 0.995
                assert not wo[~valid.numpy()].any()
                pin = export.PinholeCamera(cam.c2w, cam.fx, cam.fy, cam.cx, cam.cy, cam.width, cam.height)
                moved += int((valid != _oracle_images(oracle, pin, cluster["aabb"][i])[2]).sum())
                n_checked += 1
    assert n_checked == 6
    assert moved > 0, "the lens must change which pixels see the boxes"


def test_nerfstudio_cameras_feed_a_fused_training_step(dev):
    """End to end: nerfstudio-style Cameras with distortion -> cameras_from_nerfstudio -> DeviceTrainBatches -> one fused training step."""
    from cropnerf_b200.datamanager import DeviceTrainBatches

    n, h, w, R = 6, 45, 60, 1024
    cfg = cases.make_config(dict(log2_hashmap_size=14))
    _, state = cases.build_oracle(cfg, n, 0, 0.5)
    model = product_model(cfg, state, n, dev, True, precision="mixed")
    g = torch.Generator().manual_seed(3)
    ns_cams = SimpleNamespace(camera_to_worlds=synthetic.make_cameras(n, seed=5), fx=torch.full((n, 1), 50.0), fy=torch.full((n, 1), 50.0),
                              cx=torch.full((n, 1), w / 2.0), cy=torch.full((n, 1), h / 2.0), width=torch.full((n, 1), w),
                              height=torch.full((n, 1), h), distortion_params=torch.rand((n, 6), generator=g) * 0.02 - 0.01,
                              camera_type=torch.ones((n, 1), dtype=torch.int64))
    images = torch.randint(0, 256, (n, h, w, 3), generator=g, dtype=torch.uint8)
    masks = (torch.rand((n, h, w), generator=g) < 0.2).to(torch.uint8)
    dm = DeviceTrainBatches(images, masks, export.cameras_from_nerfstudio(ns_cams), num_rays_per_batch=R, device=dev, seed=1)
    assert dm._lenses is not None
    dm_direct = DeviceTrainBatches(images, masks, ns_cams, num_rays_per_batch=R, device=dev, seed=1)   # the Cameras object itself
    bundle, batch = dm.next_train(0)
    bundle2, _ = dm_direct.next_train(0)
    assert torch.equal(bundle.directions, bundle2.directions)
    tr = engine.Trainer(model)
    assert tr._use_fused()
    stats = tr.train_iteration(0, bundle, batch)
    torch.cuda.synchronize()
    for k in ("loss", "rgb_loss", "semantics_loss"):
        assert np.isfinite(float(stats[k])), (k, float(stats[k]))
