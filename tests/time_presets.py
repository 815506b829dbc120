"""Training-step, eval-render and field-stage times of the fruit_nerf_big / fruit_nerf_huge presets in exact fp32 and in mixed precision, and
the achieved rate of the tensor-core MLP operator (csrc/mlp_mixed.cu) on the presets' MLP shapes.

    python tests/time_presets.py [--steps 10] [--rounds 3] [--out DIR]

Full table sizes (log2_hashmap_size 21) and the presets' own batches (8192 / 16384 rays).  The two precisions are timed alternately, each
round a window of `steps` training iterations between device events after warm-up.  Prints the result as JSON and, with --out DIR, also
writes it to DIR/time_presets.json."""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402
from cropnerf_b200 import _lib as L  # noqa: E402
from cropnerf_b200 import engine, synthetic  # noqa: E402
from cropnerf_b200.fruit_nerf import FruitModel, FruitNerfModelConfig  # noqa: E402
from cropnerf_b200.rays import RayBundle  # noqa: E402

# fruit_nerf_config.py:66-190 as forwarded to FruitField (method_config.py fruit_nerf_b200_big / _huge)
PRESETS = {
    "big": (8192, dict(num_nerf_samples_per_ray=128, num_proposal_samples_per_ray=(512, 256), geo_feat_dim=30, hidden_dim_semantics=128,
                       num_layers_semantic=3, max_res=4096, proposal_weights_anneal_max_num_iters=5000, log2_hashmap_size=21)),
    "huge": (16384, dict(num_nerf_samples_per_ray=64, num_proposal_samples_per_ray=(512, 512), geo_feat_dim=30, hidden_dim_semantics=128,
                         num_layers_semantic=3, max_res=8192, proposal_weights_anneal_max_num_iters=5000, log2_hashmap_size=21,
                         proposal_net_args_list=[{"hidden_dim": 16, "log2_hashmap_size": 17, "num_levels": 5, "max_res": 512, "use_linear": False},
                                                 {"hidden_dim": 16, "log2_hashmap_size": 17, "num_levels": 7, "max_res": 2048, "use_linear": False}])),
}
# the field MLPs of both presets: base, semantic, RGB
MLP_SHAPES = {"base": ((32, 64, 31), L.ACT_NONE), "semantic": ((30, 128, 128, 64), L.ACT_NONE), "rgb": ((78, 64, 64, 3), L.ACT_SIGMOID)}


def build(dev, preset, precision):
    torch.manual_seed(0)
    model = FruitModel(FruitNerfModelConfig(precision=precision, **PRESETS[preset][1]), num_train_data=bench.NUM_IMAGES)
    model.load_state_dict(synthetic.randomize_state(model.state_dict(), seed=0, table_scale=0.5))
    return model.to(dev)


def gpu_info():
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True, timeout=30)
        info["power_limit_and_max_sm_clock"] = q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else None
    except (OSError, subprocess.TimeoutExpired):
        info["power_limit_and_max_sm_clock"] = None
    return info


def time_training(dev, preset, steps, rounds):
    R = PRESETS[preset][0]
    host = [bench.host_batch(R, seed=i) for i in range(2)]
    res = {}
    runs = {}
    for precision in ("fp32", "mixed"):
        model = build(dev, preset, precision)
        tr = engine.Trainer(model, optimizers=engine.BIG_PRESET_OPTIMIZERS, cuda_graph=True)
        batches = [bench.to_bundle(h, dev, non_blocking=False) for h in host]
        for i in range(3):   # warm-up: eager step, graph capture, replay (past the 5000 anneal iterations, which run eagerly)
            tr.train_iteration(6000 + i, *batches[i % 2])
        runs[precision] = (model, tr, batches)
        res[precision] = {"step_ms": []}
    torch.cuda.synchronize()
    step = 6100
    for _ in range(rounds):
        for precision in ("fp32", "mixed"):   # alternating windows
            model, tr, batches = runs[precision]
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for i in range(steps):
                tr.train_iteration(step + i, *batches[i % 2])
            e1.record()
            torch.cuda.synchronize()
            res[precision]["step_ms"].append(e0.elapsed_time(e1) / steps)
        step += steps
    for precision in ("fp32", "mixed"):
        model, tr, batches = runs[precision]
        # per-stage device times (the stage timers live in the C call: eager steps)
        tr.cuda_graph = False
        tr.force_proposal_update = True
        L.lib().cnb_profile_enable(1)
        n_prof = 3
        for i in range(n_prof):
            tr.train_iteration(step + i, *batches[i % 2])
        stages = L.stage_profile_read()
        L.lib().cnb_profile_enable(0)
        res[precision]["stages_ms"] = {k: round(v["ms"] / n_prof, 4) for k, v in stages.items()}
        res[precision]["field_fwd_bwd_ms"] = round((stages["field_fwd"]["ms"] + stages["field_bwd"]["ms"]) / n_prof, 4)
        # eval render of one 32 768-ray chunk (eval_num_rays_per_chunk)
        model.eval()
        rb, _ = bench.to_bundle(bench.host_batch(32768, seed=999), dev, non_blocking=False)
        with torch.no_grad():
            for _ in range(2):
                model(RayBundle(rb.origins, rb.directions, rb.pixel_area, rb.camera_indices))
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(5):
                model(RayBundle(rb.origins, rb.directions, rb.pixel_area, rb.camera_indices))
            e1.record()
            torch.cuda.synchronize()
        res[precision]["render_32768_rays_ms"] = round(e0.elapsed_time(e1) / 5, 4)
        res[precision]["step_ms_median"] = round(sorted(res[precision]["step_ms"])[len(res[precision]["step_ms"]) // 2], 4)
        res[precision]["step_ms"] = [round(v, 4) for v in res[precision]["step_ms"]]
        del runs[precision]
        torch.cuda.empty_cache()
    res["field_speedup_mixed_vs_fp32"] = round(res["fp32"]["field_fwd_bwd_ms"] / res["mixed"]["field_fwd_bwd_ms"], 3)
    res["step_speedup_mixed_vs_fp32"] = round(res["fp32"]["step_ms_median"] / res["mixed"]["step_ms_median"], 3)
    res["rays_per_step"] = R
    return res


def time_operator(dev, n=1 << 20, reps=10):
    """cnb_mlp_mixed_fwd / _bwd alone at n rows: FLOPs from the shapes (2 * in * out per layer forward; dW and dX twice that backward, no dX of
    layer 0 when not requested -- here it is) over event time."""
    out = {}
    lib = L.lib()
    for name, (dims, act) in MLP_SHAPES.items():
        g = torch.Generator(device=dev).manual_seed(0)
        Ws = [torch.randn((dims[i + 1], dims[i]), device=dev, generator=g) * dims[i] ** -0.5 for i in range(len(dims) - 1)]
        bs = [torch.zeros(dims[i + 1], device=dev) for i in range(len(dims) - 1)]
        dWs, dbs = [torch.zeros_like(w) for w in Ws], [torch.zeros_like(b) for b in bs]
        m = L.make_mlp(Ws, bs, act, dWs, dbs)
        x = torch.rand((n, dims[0]), device=dev, generator=g)
        dy = torch.randn((n, dims[-1]), device=dev, generator=g)
        y = torch.empty((n, dims[-1]), device=dev)
        dx = torch.empty((n, dims[0]), device=dev)
        scratch = torch.empty((lib.cnb_mlp_mixed_scratch_floats(C.byref(m), n, 1),), device=dev)
        st = L.stream_ptr(dev)
        fwd = lambda: L.check(lib.cnb_mlp_mixed_fwd(C.byref(m), x.data_ptr(), dims[0], n, y.data_ptr(), scratch.data_ptr(), 1, st), "fwd")  # noqa: E731
        bwd = lambda: L.check(lib.cnb_mlp_mixed_bwd(C.byref(m), x.data_ptr(), dims[0], y.data_ptr(), dy.data_ptr(), n, dx.data_ptr(), dims[0],  # noqa: E731
                                                    scratch.data_ptr(), st), "bwd")
        flops = sum(2 * dims[i] * dims[i + 1] for i in range(len(dims) - 1)) * n
        t = {}
        for tag, fn in (("fwd", fwd), ("bwd", bwd)):
            fn(); fn()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(reps):
                fn()
            e1.record()
            torch.cuda.synchronize()
            t[tag] = e0.elapsed_time(e1) / reps
        out[name] = {"dims": list(dims), "rows": n, "fwd_ms": round(t["fwd"], 4), "bwd_ms": round(t["bwd"], 4),
                     "fwd_tflops": round(flops / t["fwd"] / 1e9, 2), "bwd_tflops": round(2 * flops / t["bwd"] / 1e9, 2)}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None, help="directory for time_presets.json (default: print only)")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_presets.py measures on a CUDA device; none is visible")
    dev = torch.device("cuda:0")
    result = {"gpu": gpu_info(), "operator": time_operator(dev)}
    for preset in PRESETS:
        result[preset] = time_training(dev, preset, args.steps, args.rounds)
    result["gpu_after"] = gpu_info()
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "time_presets.json"), "w") as f:
            json.dump(result, f, indent=1)
    print(json.dumps(result, indent=1))


if __name__ == "__main__":
    main()
