"""Profiling aid: a few eval renders of 32768 rays (the export / projection chunk body) in mixed precision."""
import os, sys, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench
from cropnerf_b200.rays import RayBundle
dev = torch.device("cuda:0")
prec = sys.argv[1] if len(sys.argv) > 1 else "mixed"
R = int(sys.argv[2]) if len(sys.argv) > 2 else 32768
model = bench.build_model(dev, prec).eval()
hb = bench.host_batch(R, 5)
rb, _ = bench.to_bundle(hb, dev, False)
for _ in range(4):
    with torch.no_grad():
        out = model(RayBundle(rb.origins, rb.directions, rb.pixel_area, rb.camera_indices))
torch.cuda.synchronize()
print("ok", float(out["rgb"].mean()))
