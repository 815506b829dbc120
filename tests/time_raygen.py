"""Cost of lens undistortion in the three device ray generators: each timed with the lens off and on, alternately.

    python tests/time_raygen.py [--calls 200] [--out DIR]

* ``cnb_sample_train_batch`` / ``_lens``: 4096 rays drawn from 300 resident 1920x1080 uint8 images with masks (the training batch);
* ``cnb_generate_rays`` / ``_lens``: every pixel of one 1920x1080 image, with pixel areas;
* ``cnb_generate_rays_boxes`` / ``_lens``: one 1080p camera against 4 boxes, and the whole ``project_camera_boxes`` call (ray
  generation, hit-count read-back, two renders of the hits on the base-preset model, scatter) around it.

The kernels are captured in CUDA graphs of 20 back-to-back calls, so the host's launch cost is not in the time; each replay is
bracketed by CUDA events and the per-call time is the median over ``--calls`` replays (then divided by 20).  ``project_camera_boxes``
reads a count back to the host, so it is timed call by call with events.  The lens is nerfstudio's OPENCV model with all six
parameters non-zero.  Prints JSON and, with --out DIR, writes DIR/r3_raygen_lens.json."""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402
from cropnerf_b200 import _lib as L  # noqa: E402
from cropnerf_b200 import export, synthetic  # noqa: E402

LENS = [-0.12, 0.03, -0.004, 0.0005, 1e-3, -5e-4]   # k1, k2, k3, k4, p1, p2
PER_GRAPH = 20


def gpu_info():
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True, timeout=30)
        info["power_limit_and_max_sm_clock"] = q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else None
    except (OSError, subprocess.TimeoutExpired):
        info["power_limit_and_max_sm_clock"] = None
    return info


def graph_of(fn):
    """fn() enqueues one call on the current stream; returns a CUDA graph of PER_GRAPH calls (warmed up first)."""
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for _ in range(3):
            fn()
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for _ in range(PER_GRAPH):
            fn()
    torch.cuda.synchronize()
    return g


def alternate(runs, calls, per_call_divisor=1):
    """runs: {name: callable}; each timed `calls` times between events, names interleaved.  Returns median / min in microseconds."""
    times = {k: [] for k in runs}
    for k, f in runs.items():   # warm-up
        for _ in range(3):
            f()
    torch.cuda.synchronize()
    for _ in range(calls):
        for k, f in runs.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            f()
            e1.record()
            e1.synchronize()
            times[k].append(1e3 * e0.elapsed_time(e1) / per_call_divisor)
    return {k: {"median_us": statistics.median(v), "min_us": min(v), "samples": len(v)} for k, v in times.items()}


def time_train_batch(dev, calls):
    from cropnerf_b200.datamanager import DeviceTrainBatches

    n, h, w, R = bench.NUM_IMAGES, synthetic.IMAGE_H, synthetic.IMAGE_W, 4096
    g = torch.Generator(device=dev).manual_seed(0)
    images = torch.randint(0, 256, (n, h, w, 3), generator=g, device=dev, dtype=torch.uint8)
    masks = (torch.rand((n, h, w), generator=g, device=dev) < 0.1).to(torch.uint8)
    c2w = synthetic.make_cameras(n, seed=1)
    cams = [export.PinholeCamera(c2w[i], synthetic.FOCAL, synthetic.FOCAL, w / 2, h / 2, w, h, distortion_params=torch.tensor(LENS)) for i in range(n)]
    dm = DeviceTrainBatches(images, masks, cams, num_rays_per_batch=R, device=dev)
    rand3 = torch.rand((R, 3), device=dev, generator=g)
    out = [torch.empty((R, 3), device=dev, dtype=torch.int32), torch.empty((R, 3), device=dev), torch.empty((R, 3), device=dev),
           torch.empty((R, 1), device=dev), torch.empty((R, 1), device=dev, dtype=torch.int32), torch.empty((R, 3), device=dev),
           torch.empty((R, 1), device=dev)]
    ptrs = [t.data_ptr() for t in out]
    lib = L.lib()

    def off():
        L.check(lib.cnb_sample_train_batch(C.byref(dm._set), rand3.data_ptr(), R, *ptrs, L.stream_ptr(dev)), "sample_train_batch")

    def on():
        L.check(lib.cnb_sample_train_batch_lens(C.byref(dm._set), dm._lenses.data_ptr(), rand3.data_ptr(), R, *ptrs, L.stream_ptr(dev)), "sample_train_batch_lens")

    res = alternate({"lens_off": graph_of(off).replay, "lens_on": graph_of(on).replay}, calls, PER_GRAPH)
    res["config"] = {"rays": R, "images": n, "height": h, "width": w, "storage": "uint8 images + uint8 masks resident (2.5 GB)"}
    del images, masks, dm
    return res


def time_generate_rays(dev, calls):
    h, w = synthetic.IMAGE_H, synthetic.IMAGE_W
    n = h * w
    cam = export._camera_struct(export.PinholeCamera(synthetic.make_cameras(2, seed=1)[0], synthetic.FOCAL, synthetic.FOCAL, w / 2, h / 2, w, h))
    lens = export._lens_struct(torch.tensor(LENS))
    o, d, area = torch.empty((n, 3), device=dev), torch.empty((n, 3), device=dev), torch.empty((n,), device=dev)
    lib = L.lib()

    def off():
        L.check(lib.cnb_generate_rays(C.byref(cam), None, n, None, o.data_ptr(), d.data_ptr(), area.data_ptr(), None, None, None, L.stream_ptr(dev)), "generate_rays")

    def on():
        L.check(lib.cnb_generate_rays_lens(C.byref(cam), C.byref(lens), None, n, None, o.data_ptr(), d.data_ptr(), area.data_ptr(), None, None, None,
                                           L.stream_ptr(dev)), "generate_rays_lens")

    res = alternate({"lens_off": graph_of(off).replay, "lens_on": graph_of(on).replay}, calls, PER_GRAPH)
    res["config"] = {"rays": n, "height": h, "width": w, "outputs": "origins, directions, pixel_area (no AABB)", "bytes_written": n * 7 * 4}
    return res


def time_projection(dev, calls):
    h, w = synthetic.IMAGE_H, synthetic.IMAGE_W
    model = bench.build_export_model(dev, "mixed")
    c2w = synthetic.make_cameras(2, seed=1)[0]
    cam_off = export.PinholeCamera(c2w, synthetic.FOCAL, synthetic.FOCAL, w / 2, h / 2, w, h)
    cam_on = export.PinholeCamera(c2w, synthetic.FOCAL, synthetic.FOCAL, w / 2, h / 2, w, h, distortion_params=torch.tensor(LENS))
    g = torch.Generator().manual_seed(11)
    c = (torch.rand((4, 3), generator=g) - 0.5) * 0.6
    half = 0.04 + 0.03 * torch.rand((4, 3), generator=g)
    boxes = torch.cat([c - half, c + half], dim=1)
    # the ray-generation kernel alone, graphed
    k, npix = 4, w * h
    cap = k * npix
    bufs = [torch.empty((cap, 3), device=dev), torch.empty((cap, 3), device=dev)] + [torch.empty((cap,), device=dev) for _ in range(3)]
    tags, count = torch.empty((cap,), device=dev, dtype=torch.int32), torch.zeros((1,), device=dev, dtype=torch.int32)
    bd = boxes.to(dev).contiguous()
    cs, ls = export._camera_struct(cam_off), export._lens_struct(torch.tensor(LENS))
    lib = L.lib()

    def kernel(lens):
        def f():
            count.zero_()   # the count accumulates: cleared in every call, so that each one writes all its hits
            L.check(lib.cnb_generate_rays_boxes_lens(C.byref(cs), lens, bd.data_ptr(), k, cap, *[b.data_ptr() for b in bufs], tags.data_ptr(),
                                                     count.data_ptr(), L.stream_ptr(dev)), "generate_rays_boxes_lens")
        return f

    res = {"kernel": alternate({"lens_off": graph_of(kernel(None)).replay, "lens_on": graph_of(kernel(C.byref(ls))).replay}, calls, PER_GRAPH)}
    hits = {}

    def call(cam, name):
        def f():
            hits[name] = export.project_camera_boxes(model, cam, boxes)["hits"]
        return f

    res["project_camera_boxes"] = alternate({"lens_off": call(cam_off, "lens_off"), "lens_on": call(cam_on, "lens_on")}, calls)
    res["config"] = {"height": h, "width": w, "boxes": k, "model": "base preset (FruitNerfModelConfig defaults), mixed precision",
                     "hits": hits}
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--calls", type=int, default=200)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_raygen.py measures GPU kernels and needs a CUDA device")
    dev = torch.device("cuda:0")
    result = {"gpu": gpu_info(), "lens": dict(zip(("k1", "k2", "k3", "k4", "p1", "p2"), LENS)), "calls": args.calls, "calls_per_graph": PER_GRAPH,
              "sample_train_batch": time_train_batch(dev, args.calls), "generate_rays": time_generate_rays(dev, args.calls),
              "generate_rays_boxes": time_projection(dev, args.calls)}
    text = json.dumps(result, indent=1)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "r3_raygen_lens.json"), "w") as f:
            f.write(text + "\n")
    print(text)


if __name__ == "__main__":
    main()
