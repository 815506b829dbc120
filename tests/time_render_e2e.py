import os, sys, time, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench
from cropnerf_b200.rays import RayBundle
dev = torch.device("cuda:0")
model = bench.build_model(dev, "mixed").eval()
R = 32768
rhost = bench.host_batch(R, 5)
hb = RayBundle(rhost["origins"], rhost["directions"], rhost["pixel_area"], rhost["camera_indices"])
for _ in range(3):
    model.get_outputs_for_camera_jagged_ray_bundle(hb)
torch.cuda.synchronize()
t0 = time.perf_counter()
for _ in range(10):
    model.get_outputs_for_camera_jagged_ray_bundle(hb)
t1 = time.perf_counter()
print("e2e ms/call", (t1 - t0) * 100)
# phases
T = {"h2d": 0, "fwd": 0, "d2h": 0}
for _ in range(10):
    a = time.perf_counter()
    rb = hb._map(lambda t: t.to(dev, non_blocking=True)); torch.cuda.synchronize()
    b = time.perf_counter()
    with torch.no_grad():
        out = model(rb)
    torch.cuda.synchronize()
    c = time.perf_counter()
    host = {k: torch.empty(v.shape, dtype=v.dtype, pin_memory=True) for k, v in out.items()}
    c2 = time.perf_counter()
    for k, v in out.items():
        host[k].copy_(v, non_blocking=True)
    torch.cuda.synchronize()
    d = time.perf_counter()
    T["h2d"] += b - a; T["fwd"] += c - b; T["d2h"] += d - c2
print({k: round(v * 100, 3) for k, v in T.items()})
import cProfile, pstats
pr = cProfile.Profile(); pr.enable()
for _ in range(10):
    model.get_outputs_for_camera_jagged_ray_bundle(hb)
pr.disable()
pstats.Stats(pr).sort_stats("tottime").print_stats(12)
