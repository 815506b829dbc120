import os, sys, torch, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench
from cropnerf_b200.rays import RayBundle
dev = torch.device("cuda:0")
for prec in ("fp32", "mixed"):
    model = bench.build_model(dev, prec).eval()
    for R in (4096, 32768):
        hb = bench.host_batch(R, 5)
        rb, _ = bench.to_bundle(hb, dev, False)
        def run():
            with torch.no_grad():
                return model(RayBundle(rb.origins, rb.directions, rb.pixel_area, rb.camera_indices))
        for _ in range(3): run()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(10): run()
        e1.record(); torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / 10
        print(prec, R, "ms/render", round(ms, 3), "Mrays/s", round(R / ms / 1e3, 2))
