"""fp32 vs fp16 field tables (FruitField table_precision="fp16") on the fruit_nerf_big / fruit_nerf_huge presets in mixed precision.

    python tests/time_fp16_tables.py [--steps 10] [--rounds 3] [--train-steps 300] [--out DIR]

Per preset, with the two table precisions alternating within one session (`rounds` runs each):
  * cnb_hashgrid_fwd alone at 1 M samples (16 levels x 2^21 rows: 256 MiB fp32 / 128 MiB fp16, twice / once the 126 MB L2);
  * the graphed training step (tests/time_presets.py's method: device events around `steps` iterations after warm-up);
  * the field_fwd / field_bwd / adam_fields stages (stage timers of the C call, eager steps);
  * the eval render of one 32 768-ray chunk;
  * the extra device memory of the fp16 copy.
Then `train-steps` steps of the big preset from the same seed with each table precision: both loss curves (every 10th step).
Writes DIR/r5_fp16_tables.json with --out."""
import argparse
import ctypes as C
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from time_presets import PRESETS, gpu_info  # noqa: E402

import bench  # noqa: E402
from cropnerf_b200 import _lib as L  # noqa: E402
from cropnerf_b200 import engine, synthetic  # noqa: E402
from cropnerf_b200.fruit_nerf import FruitModel, FruitNerfModelConfig  # noqa: E402
from cropnerf_b200.rays import RayBundle  # noqa: E402

TP = ("fp32", "fp16")


def build(dev, preset, table_precision):
    torch.manual_seed(0)
    model = FruitModel(FruitNerfModelConfig(precision="mixed", table_precision=table_precision, **PRESETS[preset][1]), num_train_data=bench.NUM_IMAGES)
    model.load_state_dict(synthetic.randomize_state(model.state_dict(), seed=0, table_scale=0.5))
    return model.to(dev)


def events_ms(fn, reps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def time_gather(dev, preset, rounds, n=1 << 20, reps=20):
    cfg = PRESETS[preset][1]
    model = build(dev, preset, "fp16")
    f = model.field
    table = f.mlp_base_grid.hash_table.detach()
    half = f.table_half_current()
    nl, log2_T, scal = f.mlp_base_grid.grid_cfg()
    g = torch.Generator(device=dev).manual_seed(0)
    pos = torch.rand((n, 3), device=dev, generator=g)
    out = torch.empty((n, 2 * nl), device=dev)
    grid = L.make_grid(table, None, nl, log2_T, scal)
    st = L.stream_ptr(dev)
    lib = L.lib()
    calls = {"fp32": lambda: L.check(lib.cnb_hashgrid_fwd(C.byref(grid), pos.data_ptr(), n, out.data_ptr(), None, st), "fwd"),
             "fp16": lambda: L.check(lib.cnb_hashgrid_fwd_half(C.byref(grid), half.data_ptr(), pos.data_ptr(), n, out.data_ptr(), None, st), "fwd")}
    res = {tp: [] for tp in TP}
    for fn in calls.values():
        fn(); fn()
    for _ in range(rounds):
        for tp in TP:
            res[tp].append(round(events_ms(calls[tp], reps), 4))
    gathers = n * nl * 8
    return {"samples": n, "levels": nl, "rows_per_level": 1 << log2_T, "max_res": cfg["max_res"],
            **{f"{tp}_ms": res[tp] for tp in TP},
            **{f"{tp}_corner_gathers_per_s_G": round(gathers / (min(res[tp]) * 1e-3) / 1e9, 1) for tp in TP}}


def time_model(dev, preset, steps, rounds):
    R = PRESETS[preset][0]
    host = [bench.host_batch(R, seed=i) for i in range(2)]
    runs, res = {}, {}
    for tp in TP:
        model = build(dev, preset, tp)
        tr = engine.Trainer(model, optimizers=engine.BIG_PRESET_OPTIMIZERS, cuda_graph=True)
        batches = [bench.to_bundle(h, dev, non_blocking=False) for h in host]
        for i in range(3):
            tr.train_iteration(6000 + i, *batches[i % 2])
        runs[tp] = (model, tr, batches)
        res[tp] = {"step_ms": [], "extra_device_bytes": int(model.field.table_half.numel() * 2) if tp == "fp16" else 0}
    torch.cuda.synchronize()
    step = 6100
    for _ in range(rounds):
        for tp in TP:
            model, tr, batches = runs[tp]
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for i in range(steps):
                tr.train_iteration(step + i, *batches[i % 2])
            e1.record()
            torch.cuda.synchronize()
            res[tp]["step_ms"].append(round(e0.elapsed_time(e1) / steps, 4))
        step += steps
    # stage times (eager steps: the stage timers live in the C call; the fields group's update is the adam_fields stage there), alternating
    for tp in TP:
        runs[tp][1].cuda_graph = False
        runs[tp][1].force_proposal_update = True
        res[tp]["stages_ms"] = []
    for _ in range(rounds):
        for tp in TP:
            model, tr, batches = runs[tp]
            tr.wait_deferred_update()
            tr.train_iteration(step, *batches[0])
            # in-step update: the eager trainer runs its own Adam; time the fused fields update here directly
            L.lib().cnb_profile_enable(1)
            for i in range(3):
                tr.train_iteration(step + 1 + i, *batches[i % 2])
            stages = L.stage_profile_read()
            L.lib().cnb_profile_enable(0)
            res[tp]["stages_ms"].append({k: round(stages[k]["ms"] / 3, 4) for k in ("field_fwd", "field_bwd") if k in stages})
            step += 4
    # the fields group's update alone (RAdam step scalars, live bitmap; fp16: + the fused copy store)
    for tp in TP:
        res[tp]["fields_update_ms"] = []
    for _ in range(rounds):
        for tp in TP:
            model, tr, _ = runs[tp]
            g = tr.groups["fields"]
            sc = engine.step_scalars(tr.optimizers["fields"], 1e-4, 10000)

            def upd(g=g, sc=sc):
                from cropnerf_b200 import ops
                ops.adam_step_scalars(g.flat, g.grad, g.exp_avg, g.exp_avg_sq, sc, live=g.live, half=g.half)
            upd()
            res[tp]["fields_update_ms"].append(round(events_ms(upd, 20), 4))
    for tp in TP:
        res[tp]["render_32768_rays_ms"] = []
    rb, _ = bench.to_bundle(bench.host_batch(32768, seed=999), dev, non_blocking=False)
    bundle = lambda: RayBundle(rb.origins, rb.directions, rb.pixel_area, rb.camera_indices)  # noqa: E731
    for tp in TP:
        runs[tp][0].eval()
        with torch.no_grad():
            runs[tp][0](bundle()); runs[tp][0](bundle())
    for _ in range(rounds):
        for tp in TP:
            model = runs[tp][0]
            with torch.no_grad():
                res[tp]["render_32768_rays_ms"].append(round(events_ms(lambda: model(bundle()), 5), 4))
    for tp in TP:
        r = res[tp]
        r["step_ms_median"] = sorted(r["step_ms"])[len(r["step_ms"]) // 2]
        r["field_fwd_ms_median"] = sorted(s["field_fwd"] for s in r["stages_ms"])[rounds // 2]
        r["field_bwd_ms_median"] = sorted(s["field_bwd"] for s in r["stages_ms"])[rounds // 2]
        r["render_ms_median"] = sorted(r["render_32768_rays_ms"])[rounds // 2]
        r["fields_update_ms_median"] = sorted(r["fields_update_ms"])[rounds // 2]
    del runs
    torch.cuda.empty_cache()
    res["rays_per_step"] = R
    res["step_ratio_fp16_over_fp32"] = round(res["fp16"]["step_ms_median"] / res["fp32"]["step_ms_median"], 4)
    res["render_ratio_fp16_over_fp32"] = round(res["fp16"]["render_ms_median"] / res["fp32"]["render_ms_median"], 4)
    res["field_fwd_ratio_fp16_over_fp32"] = round(res["fp16"]["field_fwd_ms_median"] / res["fp32"]["field_fwd_ms_median"], 4)
    return res


def loss_curves(dev, train_steps):
    R = PRESETS["big"][0]
    out = {}
    for tp in TP:
        model = build(dev, "big", tp)
        tr = engine.Trainer(model, optimizers=engine.BIG_PRESET_OPTIMIZERS, cuda_graph=True)
        losses = []
        for step in range(train_steps):
            rb, batch = bench.to_bundle(bench.host_batch(R, seed=step), dev, non_blocking=False)
            losses.append(tr.train_iteration(step, rb, batch)["loss"].detach().clone())
        c = torch.stack(losses).cpu()
        out[tp] = {"finite": bool(torch.isfinite(c).all()), "loss_every_10": [round(float(x), 6) for x in c[::10]], "last": round(float(c[-1]), 6)}
        del model, tr
        torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--train-steps", type=int, default=300)
    ap.add_argument("--out", default=None, help="directory for r5_fp16_tables.json (default: print only)")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_fp16_tables.py measures on a CUDA device; none is visible")
    dev = torch.device("cuda:0")
    result = {"gpu": gpu_info()}
    for preset in PRESETS:
        result[preset] = {"hashgrid_fwd": time_gather(dev, preset, args.rounds)}
        result[preset].update(time_model(dev, preset, args.steps, args.rounds))
    result["big_loss_curves"] = loss_curves(dev, args.train_steps)
    result["gpu_after"] = gpu_info()
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "r5_fp16_tables.json"), "w") as f:
            json.dump(result, f, indent=1)
    print(json.dumps(result, indent=1))


if __name__ == "__main__":
    main()
