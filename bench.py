#!/usr/bin/env python
"""Benchmark of the FruitNeRF per-ray rendering hot path (BASELINE.json metric), one JSON line on stdout.

  python bench.py --gpus N --steps K --warmup W [--impl reference] [--precision fp32|mixed] [--dump-outputs DIR]
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Headline `value`: training rays/s (fwd + bwd + gradient all-reduce + Adam) of the `fruit_nerf` preset
(BASELINE.json configs[1]: 4096-ray batch per GPU, proposal 256/96 + 48 NeRF samples, full-size hash tables), inputs
resident in HBM.  `e2e`: the same step through the public API with HOST ray/target buffers (pinned) copied in and the
loss read back every step.  `render`: eval-mode render (the export / projection loop body) in rays/s.
`roofline`: dominant C-ABI call, algorithmic bytes (SURVEY.md section 8d) / CUDA-event time.  `cpu_baseline`: the oracle
(torch CPU restatement of the reference path) on the box's host cores on a bounded sample.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

RAYS_PER_GPU = 4096
PROPOSAL_SAMPLES = (256, 96)
NERF_SAMPLES = 48
NUM_IMAGES = 300
# algorithmic bytes per ray (SURVEY.md section 8d / BASELINE.md section 3), fp32 tables: 8 corners * 2 floats per (sample, level)
FETCH_BYTES = {"prop0": 256 * 5 * 8 * 8, "prop1": 96 * 5 * 8 * 8, "field": 48 * 16 * 8 * 8}
RENDER_BYTES_PER_RAY = sum(FETCH_BYTES.values()) + 40 + 24                    # 161 856
TRAIN_BYTES_PER_RAY = 3 * sum(FETCH_BYTES.values()) + 64 + 16                 # 485 456 (update step: gather + scatter RMW)


WORKLOAD = ("BASELINE configs[1]: fruit_nerf preset training step, 4096 rays/GPU, proposal 256/96 + 48 NeRF samples, "
            "field 16x2^19x2 + 2 proposal 5x2^17x2 fp32 hash tables, 300 synthetic 1080p cameras")


def workload_config():
    """`config` of the JSON line -- the SAME dict in the product arm and in `--impl reference` (the driver compares them)."""
    return {"workload": WORKLOAD, "rays_per_gpu": RAYS_PER_GPU, "samples_per_ray": sum(PROPOSAL_SAMPLES) + NERF_SAMPLES,
            "l2": "inputs larger than L2: one step streams ~0.4 GB (parameters, gradients, Adam moments, workspace) through the 126 MB L2; steps timed back to back"}


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        return float(p["hbm_gbs"]), "measured"
    return 6650.0, "fallback"


class ClockSampler:
    """SM clock / throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe).

    Primary source: NVML (the library nvidia-smi itself reads) polled every 2 ms from a thread, so that a timed region of a few
    milliseconds still gets several samples; fallback: an `nvidia-smi --query-gpu ... -lms 100` child process."""

    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

    def __init__(self, index: int):
        self.index = index
        self.rows = []          # nvidia-smi rows
        self.samples = []       # NVML (sm_mhz, reasons bitmask)
        self.proc = None
        self.nvml = None
        self.handle = None
        self.max_mhz = None
        self.running = False
        self.thread = None
        self.source = None

    def _nvml_open(self):
        import pynvml
        pynvml.nvmlInit()
        try:
            uuid = str(torch.cuda.get_device_properties(self.index).uuid)
            self.handle = pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + uuid) if not uuid.startswith("GPU-") else uuid)
        except Exception:
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(self.index)
        self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
        pynvml.nvmlDeviceGetClockInfo(self.handle, pynvml.NVML_CLOCK_SM)              # probe both queries once
        pynvml.nvmlDeviceGetCurrentClocksEventReasons(self.handle)
        self.nvml = pynvml

    def _poll(self):
        nv, h = self.nvml, self.handle
        while self.running:
            try:
                self.samples.append((float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)), int(nv.nvmlDeviceGetCurrentClocksEventReasons(h))))
            except Exception:
                pass
            time.sleep(0.002)

    def start(self):
        try:
            self._nvml_open()
            self.running = True
            self.source = "nvml"
            self.thread = threading.Thread(target=self._poll, daemon=True)
            self.thread.start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.source = "nvidia-smi"
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.nvml is not None:
            self.running = False
            self.thread.join(timeout=1.0)
            nv = self.nvml
            bits = {"hw_slowdown": nv.nvmlClocksEventReasonHwSlowdown, "hw_thermal_slowdown": nv.nvmlClocksEventReasonHwThermalSlowdown,
                    "sw_thermal_slowdown": nv.nvmlClocksEventReasonSwThermalSlowdown, "sw_power_cap": nv.nvmlClocksEventReasonSwPowerCap}
            sm = sorted(s for s, _ in self.samples)
            reasons = sorted(n for n, b in bits.items() if any(r & b for _, r in self.samples))
            try:
                nv.nvmlShutdown()
            except Exception:
                pass
            return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": self.max_mhz, "reasons": reasons, "samples": len(sm), "source": "nvml"}
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
                for n, v in zip(self.NAMES, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                pass
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons), "samples": len(sm),
                "source": "nvidia-smi"}


def build_model(dev, precision, seed=0):
    from cropnerf_b200 import synthetic
    from cropnerf_b200.fruit_nerf import FruitModel, FruitNerfModelConfig

    torch.manual_seed(seed)
    cfg = FruitNerfModelConfig(precision=precision)
    model = FruitModel(cfg, num_train_data=NUM_IMAGES)
    state = synthetic.randomize_state(model.state_dict(), seed=seed, table_scale=0.5)
    model.load_state_dict(state)
    return model.to(dev)


def host_batch(R, seed):
    from cropnerf_b200 import synthetic

    rays = synthetic.make_rays(R, seed=seed, num_cameras=NUM_IMAGES)
    tgt = synthetic.make_targets(R, seed=seed + 7)
    out = {**rays, **tgt}
    return {k: v.pin_memory() for k, v in out.items()}


def to_bundle(batch, dev, non_blocking=True):
    from cropnerf_b200.rays import RayBundle

    g = {k: v.to(dev, non_blocking=non_blocking) for k, v in batch.items()}
    rb = RayBundle(g["origins"], g["directions"], g["pixel_area"], g["camera_indices"])
    return rb, {"image": g["image"], "fruit_mask": g["fruit_mask"]}


def bytes_of(batch):
    return int(sum(v.numel() * v.element_size() for v in batch.values()))


DUMP_PARAM_FLOATS = 15 << 20   # --dump-outputs: parameter values written, all groups together (60 MiB of float32)


def last_step_outputs(trainer, stats):
    """What the caller of the last timed training step is left with: the loss / metric scalars the step returns and the parameters it
    updated.  A flat group larger than its share of DUMP_PARAM_FLOATS is written as a fixed sample (seeded, sorted indices), so that two
    builds of the project run with the same arguments write the same elements."""
    out = {k: v.detach().float().cpu().numpy() for k, v in stats.items()}
    share = DUMP_PARAM_FLOATS // len(trainer.groups)
    for name, g in trainer.groups.items():
        n = g.flat.numel()
        if n <= share:
            out["params_" + name] = g.flat.cpu().numpy()
        else:
            idx = torch.randperm(n, generator=torch.Generator().manual_seed(0))[:share].sort().values
            out[f"params_{name}_sample"] = g.flat[idx.to(g.flat.device)].cpu().numpy()
    return out


def measure(args, precision, dev, world, rank, local_rank, full=True):
    """One precision mode: training step (resident + end-to-end), per-stage device times, eval render."""
    from cropnerf_b200 import _lib as L
    from cropnerf_b200 import engine
    from cropnerf_b200.rays import RayBundle
    import torch.distributed as dist

    model = build_model(dev, precision)
    # every timed step back-propagates into all three networks (the update step SURVEY.md 8d's 485 456 B/ray describes;
    # in steady state only 1 step in 6 does, ProposalNetworkSampler update_sched) and is replayed as one CUDA graph
    trainer = engine.Trainer(model, world_size=world, cuda_graph=not args.no_graph, force_proposal_update=True, ddp=args.ddp)
    R = RAYS_PER_GPU
    nb = 8  # distinct ray batches cycled through (fresh rays every step, like next_train)
    host = [host_batch(R, seed=100 * rank + i) for i in range(nb)]
    resident = [to_bundle(b, dev, non_blocking=False) for b in host]
    l2_flush = torch.empty((192 << 20,), dtype=torch.uint8, device=dev)  # > 126 MB L2

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def train_step(step, rb, tg):
        rb = RayBundle(rb.origins, rb.directions, rb.pixel_area, rb.camera_indices)  # the collider mutates the bundle
        return trainer.train_iteration(step, rb, tg)

    steps = args.steps if full else max(3, args.steps // 2)
    # ---- warm-up -----------------------------------------------------------------------------------------
    step = 2000  # past proposal_weights_anneal_max_num_iters (1000): anneal == 1 as in 39 000 of the 40 000 training iterations
    for _ in range(max(args.warmup, 3)):
        train_step(step, *resident[step % nb]); step += 1
    barrier()

    # ---- timed: resident inputs ----------------------------------------------------------------------------
    # Headline: EXACTLY `steps` training steps back to back (barrier + synchronize on both sides, one event pair) -- a training loop's
    # throughput.  No flush is needed or wanted there: one step streams ~0.4 GB (parameters, gradients, Adam moments, workspace) through the
    # 126 MB L2, and the optimiser / parameter exchange of step i is allowed to overlap the first stage of step i+1 (it is part of the
    # program, not of a gap between measurements).  The flushed per-step time is measured as well, with each step's own deferred update inside
    # its timed region, so that no work can hide in the untimed flush.
    def settle():
        if getattr(trainer, "wait_deferred_update", None) is not None:
            trainer.wait_deferred_update()

    clocks = ClockSampler(local_rank)
    if rank == 0 and full:
        clocks.start()
    barrier()
    b0, b1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    b0.record()
    h0 = time.perf_counter()
    for i in range(steps):
        stats = train_step(step, *resident[step % nb]); step += 1
    host_enqueue_ms = 1e3 * (time.perf_counter() - h0) / steps   # host time to ENQUEUE one step (no sync inside): must stay below ms_per_step
    settle()
    b1.record()
    barrier()
    clk = clocks.stop() if (rank == 0 and full) else None
    t_local = b0.elapsed_time(b1) / 1e3
    # taken before the legs below train on: they overwrite the returned loss buffer and move the parameters
    outputs = last_step_outputs(trainer, stats) if (args.dump_outputs and full and rank == 0) else None
    barrier()  # rank 0 has just spent ~0.2 s stopping its clock sampler: line the ranks up again
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    for i in range(steps):
        l2_flush.fill_(i & 0xFF)  # 192 MiB fill: cold L2 for every step
        ev[i][0].record()
        train_step(step, *resident[step % nb]); step += 1
        settle()
        ev[i][1].record()
    barrier()
    t_b2b_local = sum(a.elapsed_time(b) for a, b in ev) / 1e3   # (kept name) flushed, serialised per-step time

    # ---- timed: end to end through the public API with host buffers ------------------------------------------
    # the public call takes the pinned HOST rays / targets as they are: train_iteration copies them (H2D, async) into the graphed
    # step's static device buffers, replays the step, runs the optimiser; the loss is read back (D2H + sync) every step
    def host_bundle(b):
        return RayBundle(b["origins"], b["directions"], None, b["camera_indices"]), {"image": b["image"], "fruit_mask": b["fruit_mask"]}

    for i in range(3):
        rb, tg = host_bundle(host[step % nb])
        float(trainer.train_iteration(step, rb, tg)["loss"].item()); step += 1
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    loss_host = 0.0
    for i in range(steps):
        rb, tg = host_bundle(host[step % nb])          # pinned host memory in ...
        stats = trainer.train_iteration(step, rb, tg); step += 1   # ... H2D inside the call, every step
        loss_host = float(stats["loss"].item())        # D2H read of the step's result
    e1.record()
    barrier()
    t_e2e_local = e0.elapsed_time(e1) / 1e3

    # ---- replicas: after all those steps every rank must hold bit-identical parameters (each element is computed once, by its
    # owner, and broadcast; or all-reduced in a fixed order) -- a checksum of every flat group, all-gathered and compared ----------
    replicas_identical = None
    if world > 1:
        settle()
        torch.cuda.synchronize()
        sums = torch.stack([g.flat.view(torch.int32).to(torch.int64).sum() for g in trainer.groups.values()])
        allsums = [torch.empty_like(sums) for _ in range(world)]
        dist.all_gather(allsums, sums)
        replicas_identical = all(bool(torch.equal(a, allsums[0])) for a in allsums)
        assert replicas_identical, f"rank {rank}: parameter checksums differ across replicas: {[a.tolist() for a in allsums]}"

    # ---- where the step spends its time, and what N > 1 adds (rank 0's view, CUDA events around the two graphs of the pipelined step, a separate
    # short pass): graph A = samplers + proposal forward; `wait` = the stream idling for the previous step's `fields` exchange (what the
    # exchange could not hide behind graph A); graph B = field forward + whole backward + the in-graph proposal exchange -------------------
    ddp_breakdown = None
    if not args.no_graph and full:
        trainer._probe = []
        barrier()
        for i in range(12):
            train_step(step, *resident[step % nb]); step += 1
        settle()
        torch.cuda.synchronize()
        evs = trainer._probe[2:]
        trainer._probe = None
        if evs:
            a = sum(e[0].elapsed_time(e[1]) for e in evs) / len(evs)
            w = sum(e[1].elapsed_time(e[2]) for e in evs) / len(evs)
            b = sum(e[2].elapsed_time(e[3]) for e in evs) / len(evs)
            ddp_breakdown = {"graph_a_ms": a, "wait_for_fields_exchange_ms": w, "graph_b_ms": b, "steps": len(evs),
                             "note": "graph_a = samplers + proposal forward (overlaps the previous step's fields exchange); wait = stream idle until that exchange "
                                     "has landed; graph_b = field forward + backward + in-graph proposal exchange; compare graph_a + graph_b with the N = 1 line's ms_per_step"}

    # ---- end to end from DEVICE-resident images (row f1: FruitDataManager.next_train as one kernel, datamanager.DeviceTrainBatches):
    # the pixel sampler + ray generator run on the GPU over uint8 images held in HBM, so no ray / target bytes cross PCIe at all;
    # the loss is still read back every step -----------------------------------------------------------------------------------
    t_dev_batches = None
    if full and not args.no_device_batches:
        from cropnerf_b200 import synthetic
        from cropnerf_b200.datamanager import DeviceTrainBatches
        from cropnerf_b200.export import PinholeCamera
        gen = torch.Generator(device=dev).manual_seed(1234 + rank)
        imgs = torch.randint(0, 256, (NUM_IMAGES, synthetic.IMAGE_H, synthetic.IMAGE_W, 3), device=dev, dtype=torch.uint8, generator=gen)
        msk = (torch.rand((NUM_IMAGES, synthetic.IMAGE_H, synthetic.IMAGE_W), device=dev, generator=gen) < 0.1).to(torch.uint8)
        c2w = synthetic.make_cameras(NUM_IMAGES, seed=1)
        cams = [PinholeCamera(c2w[i], synthetic.FOCAL, synthetic.FOCAL, synthetic.IMAGE_W / 2, synthetic.IMAGE_H / 2, synthetic.IMAGE_W, synthetic.IMAGE_H)
                for i in range(NUM_IMAGES)]
        dm = DeviceTrainBatches(imgs, msk, cams, num_rays_per_batch=R, device=dev, seed=rank)
        for i in range(3):
            rb, tg = dm.next_train(step)
            float(trainer.train_iteration(step, rb, tg)["loss"].item()); step += 1
        barrier()
        d0, d1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        d0.record()
        for i in range(steps):
            rb, tg = dm.next_train(step)
            stats = trainer.train_iteration(step, rb, tg); step += 1
            float(stats["loss"].item())
        d1.record()
        barrier()
        t_dev_batches = d0.elapsed_time(d1) / 1e3
        del dm, imgs, msk

    # ---- per-stage device times (separate pass so the events do not perturb the timed region) ----------------
    stage, adam_ms, n_prof = {}, 0.0, min(steps, 5)
    nonupdate_ms = None
    camopt_ms = None
    if full:
        # the same all-update step with the SO3xR3 camera optimizer on (row a17: nerfacto's default, which fruit_nerf_config.py keeps):
        # pose corrections, dLoss/d rays and the pose gradient all inside cnb_train_step (csrc/camera_opt.cu), replayed as CUDA graphs and
        # timed back to back like the headline; one extra gather pass per network for the hash-grid input gradients
        from cropnerf_b200.fruit_nerf import CameraOptimizer
        cmodel = build_model(dev, precision)
        cmodel.camera_optimizer = CameraOptimizer(NUM_IMAGES, "SO3xR3").to(dev)
        ctr = engine.Trainer(cmodel, world_size=1, cuda_graph=not args.no_graph, force_proposal_update=True)
        for i in range(4):
            rb0, tg0 = resident[(step + i) % nb]
            ctr.train_iteration(2000 + i, RayBundle(rb0.origins, rb0.directions, rb0.pixel_area, rb0.camera_indices), tg0)
        ctr.wait_deferred_update()
        torch.cuda.synchronize()
        c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        c0.record()
        for i in range(steps):
            rb0, tg0 = resident[(step + i) % nb]
            ctr.train_iteration(2004 + i, RayBundle(rb0.origins, rb0.directions, rb0.pixel_area, rb0.camera_indices), tg0)
        ctr.wait_deferred_update()
        c1.record()
        torch.cuda.synchronize()
        camopt_ms = c0.elapsed_time(c1) / steps
        del ctr, cmodel
        # steady-state step kind: proposal networks frozen this step (5 of every 6 steps after proposal_warmup)
        trainer.force_proposal_update = False
        model.proposal_sampler._step = 20000
        def frozen_step():
            nonlocal step
            model.proposal_sampler._steps_since_update = 1   # keeps "updated" false
            train_step(step, *resident[step % nb]); step += 1
            model.proposal_sampler._step = 20000

        for _ in range(3):
            frozen_step()
        settle()
        torch.cuda.synchronize()
        n0, n1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        n0.record()
        for _ in range(steps):   # back to back, like the headline
            frozen_step()
        settle()
        n1.record()
        torch.cuda.synchronize()
        nonupdate_ms = n0.elapsed_time(n1) / steps
        trainer.force_proposal_update = True
        trainer.cuda_graph = False  # the stage timers live in the C call, which a graph replay does not re-enter
        L.lib().cnb_profile_enable(1)
        a_ev = []
        orig_opt = trainer.optimizer_step

        def timed_opt(s, **kw):
            a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a0.record(); orig_opt(s, **kw); a1.record()
            a_ev.append((a0, a1))

        trainer.optimizer_step = timed_opt
        for i in range(n_prof):
            l2_flush.fill_(i & 0xFF)
            train_step(step, *resident[step % nb]); step += 1
        stage = L.stage_profile_read()
        L.lib().cnb_profile_enable(0)
        trainer.optimizer_step = orig_opt
        trainer.cuda_graph = not args.no_graph
        adam_ms = sum(a.elapsed_time(b) for a, b in a_ev) / n_prof

    # ---- render (export / projection loop body), eval mode ----------------------------------------------------
    model.eval()
    Rr = 32768
    rhost = host_batch(Rr, seed=999 + rank)
    rres, _ = to_bundle(rhost, dev, non_blocking=False)

    def render_once(rb):
        with torch.no_grad():
            return model(RayBundle(rb.origins, rb.directions, rb.pixel_area, rb.camera_indices))

    for _ in range(3):
        render_once(rres)
    barrier()
    n_r = max(3, min(steps, 10))
    rev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(n_r)]
    for i in range(n_r):
        l2_flush.fill_(i & 0xFF)
        rev[i][0].record()
        render_once(rres)
        rev[i][1].record()
    barrier()
    t_render_local = sum(a.elapsed_time(b) for a, b in rev) / 1e3
    # end to end through the public chunked-render API (host rays in, host outputs out)
    host_bundle = RayBundle(rhost["origins"], rhost["directions"], rhost["pixel_area"], rhost["camera_indices"])
    for _ in range(2):
        model.get_outputs_for_camera_jagged_ray_bundle(host_bundle)
    barrier()
    h0, h1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    h0.record()
    d2h_render = 0
    for _ in range(n_r):
        host_out = model.get_outputs_for_camera_jagged_ray_bundle(host_bundle)
        d2h_render = sum(v.numel() * v.element_size() for v in host_out.values())
    h1.record()
    barrier()
    t_render_e2e_local = h0.elapsed_time(h1) / 1e3
    render_stage = {}
    if full:
        L.lib().cnb_profile_enable(1)
        for i in range(3):
            l2_flush.fill_(i & 0xFF)
            render_once(rres)
        render_stage = {k: v["ms"] / 3 for k, v in L.stage_profile_read().items()}
        L.lib().cnb_profile_enable(0)
    model.train()

    # ---- reduce over ranks (max time) -----------------------------------------------------------------------
    times = torch.tensor([t_local, t_e2e_local, t_render_local, t_render_e2e_local, t_b2b_local], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(times, op=dist.ReduceOp.MAX)
    t, t_e2e, t_render, t_render_e2e, t_b2b = times.tolist()
    ddp_mode = trainer.ddp if world > 1 else None
    if trainer.comm is not None:
        assert not trainer.comm.timed_out(), "a peer-memory barrier timed out during the benchmark"
    del trainer, model, l2_flush
    torch.cuda.empty_cache()
    return {"outputs": outputs, "ddp": ddp_mode, "host_enqueue_ms": host_enqueue_ms, "ddp_breakdown": ddp_breakdown, "replicas_identical": replicas_identical, "t_dev_batches": t_dev_batches, "t_b2b": t_b2b, "steps": steps, "t": t, "t_e2e": t_e2e, "t_render": t_render, "t_render_e2e": t_render_e2e, "n_r": n_r, "Rr": Rr, "clk": clk,
            "stage": stage, "n_prof": n_prof, "nonupdate_ms": nonupdate_ms, "camopt_ms": camopt_ms, "adam_ms": adam_ms, "render_stage": render_stage, "loss": loss_host,
            "h2d_train": bytes_of({k: host[0][k] for k in ("origins", "directions", "camera_indices", "image", "fruit_mask")}), "h2d_render": bytes_of({k: rhost[k] for k in ("origins", "directions", "pixel_area", "camera_indices")}),
            "d2h_render": int(d2h_render)}


# algorithmic bytes per ray of each pipeline stage (fp32 tables, 8 corners x 8 B per (sample, level); SURVEY.md section 8d):
# forward = one gather; backward (proposals and field alike) = scatter read-modify-write only: the encoded features are kept by
# the forward on update steps (cnb_density_field_fwd_keep / the field ctx), so no backward kernel re-gathers the tables
STAGE_BYTES_PER_RAY = {
    "proposal0_fwd": FETCH_BYTES["prop0"], "proposal1_fwd": FETCH_BYTES["prop1"], "field_fwd": FETCH_BYTES["field"],
    "proposal0_bwd": 2 * FETCH_BYTES["prop0"], "proposal1_bwd": 2 * FETCH_BYTES["prop1"], "field_bwd": 2 * FETCH_BYTES["field"],
}


# DRAM traffic per launch of each stage (dram__bytes_read.sum + dram__bytes_write.sum of its kernels, one `ncu --set full`
# capture of this same command, third training step: profiles/r2c_top_kernels_ncu_full.csv).  field_bwd = k_field_bwd_tc5 + k_tc5_reduce +
# k_hashgrid_bwd<1>.  Far below the algorithmic bytes because the tables live in L2: the forward gathers are bound by the L1TEX data
# pipe, the backward by the SM's red issue rate (DESIGN.md 4).
NCU_DRAM_SOURCE = "profiles/r2c_top_kernels_ncu_full.csv: ncu --set full --clock-control none, round-2 final code state (field backward on tcgen05)"
NCU_DRAM_BYTES_PER_LAUNCH = {
    "field_bwd": (26.26 + 0.63 + 10.06 + 0.0 + 73.31 + 1.19) * 1e6, "field_fwd": (49.70 + 10.00) * 1e6, "proposal0_bwd": (53.41 + 1.78) * 1e6,
    "proposal1_bwd": (4.79 + 0.01) * 1e6, "proposal0_fwd": (7.19 + 1.47) * 1e6, "proposal1_fwd": 5.16e6,
}


def run_product(args):
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    # stdout carries exactly ONE JSON line: anything libraries print there meanwhile (NCCL's version banner) goes to stderr
    sys.stdout.flush()
    saved_stdout = os.dup(1)
    os.dup2(2, 1)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # NCCL_DEBUG is left as the launcher set it (the driver reads the communicator lines); fd 1 already points at stderr here,
        # so whatever NCCL prints cannot land on the JSON line
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    assert args.gpus == world, f"--gpus {args.gpus} but WORLD_SIZE={world} (launch N>1 with torch.distributed.run)"

    m = measure(args, args.precision, dev, world, rank, local_rank, full=True)
    if m["outputs"] is not None:
        import numpy as np

        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, arr in m["outputs"].items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), arr)
    other = "fp32" if args.precision == "mixed" else "mixed"
    m2 = measure(args, other, dev, world, rank, local_rank, full=False) if not args.single_precision else None
    R = RAYS_PER_GPU

    if rank == 0:
        peak, peak_src = load_peaks()
        steps = m["steps"]
        total_rays = world * R * steps
        value = total_rays / m["t"]
        n_prof = m["n_prof"]
        tot = {k: v["ms"] / n_prof for k, v in m["stage"].items()}
        tot["adam (fused Adam + grad clear, 2 flat groups)"] = m["adam_ms"]
        launches = sum(v["kernels"] for v in m["stage"].values()) / n_prof + 3  # + 2 fused Adam passes + the loss finalisation kernel
        cand = {k: v for k, v in tot.items() if k in STAGE_BYTES_PER_RAY}
        dom = max(cand, key=cand.get)
        calls = m["stage"][dom]["calls"] / n_prof
        per_launch_ms = tot[dom] / calls
        per_ray = STAGE_BYTES_PER_RAY[dom]
        ach = per_ray * R / (per_launch_ms * 1e-3) / 1e9
        roofline = {"bound": "hbm", "kernel": dom, "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                    "traffic": NCU_DRAM_BYTES_PER_LAUNCH.get(dom) if args.precision == "mixed" else None,
                    "traffic_source": NCU_DRAM_SOURCE if (args.precision == "mixed" and dom in NCU_DRAM_BYTES_PER_LAUNCH) else None,
                    "peak_source": peak_src, "ms_per_launch": per_launch_ms, "share_of_step": tot[dom] / (sum(tot.values()) + 1e-12),
                    "algorithmic_bytes_per_launch": per_ray * R,
                    "note": "algorithmic bytes = 8-byte corner fetches of SURVEY.md 8d; the 74 MiB of tables are L2-resident, so DRAM traffic is far below this"}
        step_achieved = TRAIN_BYTES_PER_RAY * total_rays / m["t"] / 1e9
        n_r, Rr = m["n_r"], m["Rr"]
        line = {
            "metric": "train_rays_per_s", "value": value, "unit": "rays/s", "n_gpus": world, "steps": steps, "warmup": max(args.warmup, 3),
            "ms_per_step": 1e3 * m["t"] / steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32" if args.precision == "fp32" else "f16 tensor-core MLPs (bf16 gradients), f32 hash tables / accumulation / compositing",
            "data": "synthetic",
            "config": workload_config(),
            "detail": {"precision": args.precision,
                       "ms_per_step_l2_flushed_serialised": 1e3 * m["t_b2b"] / steps, "data_parallel": m["ddp"], "replicas_identical": m["replicas_identical"], "ddp_breakdown": m["ddp_breakdown"],
                       "host_enqueue_ms_per_step": m["host_enqueue_ms"],
                       "note_overlap": "the big 'fields' group is updated on a side stream (one GPU: fused Adam; N>1: reduce-scatter + Adam + all-gather over NVLink) and only gates the "
                                       "NEXT step's field forward; ms_per_step_l2_flushed_serialised flushes L2 (192 MiB fill) before every step and waits for that update inside the step's timed region",
                       "includes": "fwd + losses + bwd (all three networks updated EVERY step) + gradient exchange (N>1) + Adam; "
                                   + ("cnb_train_step eager" if args.no_graph else "cnb_train_step replayed as two CUDA graphs (samplers + proposal forward | rest)"),
                       "non_update_step_ms": m["nonupdate_ms"],
                       "camera_optimizer_step_ms": m["camopt_ms"],
                       "steady_state_rays_per_s": (world * R / ((m["t"] / steps + 5 * m["nonupdate_ms"] * 1e-3) / 6)) if m["nonupdate_ms"] else None},
            "samples_per_s": value * 400,
            "step_roofline": {"algorithmic_bytes_per_ray": TRAIN_BYTES_PER_RAY, "achieved_GBps": step_achieved, "frac": step_achieved / (peak * world),
                              "roofline_rays_per_s_per_gpu": peak * 1e9 / TRAIN_BYTES_PER_RAY},
            "e2e": {"value": total_rays / m["t_e2e"], "unit": "rays/s", "h2d_bytes_per_step": m["h2d_train"], "d2h_bytes_per_step": 4,
                    "last_loss": m["loss"]},
            "e2e_device_batches": ({"value": total_rays / m["t_dev_batches"], "unit": "rays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 4,
                                    "what": "same step fed by DeviceTrainBatches.next_train (cnb_sample_train_batch over 300 uint8 1080p images + masks resident in HBM)"}
                                   if m["t_dev_batches"] else None),
            "render": {"value": world * Rr * n_r / m["t_render"], "unit": "rays/s", "rays_per_call": Rr, "l2": "flushed between calls",
                       "e2e": {"value": world * Rr * n_r / m["t_render_e2e"], "unit": "rays/s", "h2d_bytes_per_step": m["h2d_render"],
                               "d2h_bytes_per_step": m["d2h_render"]},
                       "roofline_frac": (RENDER_BYTES_PER_RAY * world * Rr * n_r / m["t_render"] / 1e9) / (peak * world),
                       "stage_ms_per_call": {k: round(v, 4) for k, v in sorted(m["render_stage"].items(), key=lambda kv: -kv[1])}},
            "roofline": roofline,
            "stage_ms_per_step": {k: round(v, 4) for k, v in sorted(tot.items(), key=lambda kv: -kv[1])},
            "gpu_launches": int(round(launches * steps)),
            "clocks": m["clk"],
        }
        if m2 is not None:
            line["other_precision"] = {"precision": other, "train_rays_per_s": world * R * m2["steps"] / m2["t"], "ms_per_step": 1e3 * m2["t"] / m2["steps"],
                                       "render_rays_per_s": world * m2["Rr"] * m2["n_r"] / m2["t_render"]}
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline(sample_rays=args.cpu_rays, steps=2, warmup=1)
        sys.stdout.flush()
        os.dup2(saved_stdout, 1)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


# ---------------------------------------------------------------------------------------------------------------------
# BASELINE configs[2] / configs[3] as timed workloads: `--workload export` (ns-export pointcloud: render rays until 10 M semantic-filtered
# points inside the crop OBB are collected, rays sharded over the ranks, no communication) and `--workload projection`
# (semantic_projection: for every (super-cluster, view) pair clip the view's rays against the sub-cluster boxes, render the un-occluded
# semantics and the opacity in front of the box at full 1080p resolution, pairs sharded over the ranks).
EXPORT_OBB = ((-0.0571, 0.1105, -0.5401), (0.0, 0.0, 0.0), (1.0, 1.0, 1.0))   # README.md:125 of the reference: centre, rpy, scale


def build_export_model(dev, precision):
    from cropnerf_b200 import synthetic
    from cropnerf_b200.fruit_nerf import FruitModel, FruitNerfModelConfig

    torch.manual_seed(0)
    model = FruitModel(FruitNerfModelConfig(precision=precision), num_train_data=NUM_IMAGES)
    # a scene with fruit in it: the semantic head's bias lifted so that a good share of the rays is labelled (sigmoid > 0.9)
    model.load_state_dict(synthetic.randomize_state(model.state_dict(), seed=0, table_scale=0.5, sem_bias=3.0))
    return model.to(dev).eval()


def synthetic_cameras(n):
    from cropnerf_b200 import synthetic
    from cropnerf_b200.export import PinholeCamera

    c2w = synthetic.make_cameras(n, seed=1)
    return [PinholeCamera(c2w[i], synthetic.FOCAL, synthetic.FOCAL, synthetic.IMAGE_W / 2, synthetic.IMAGE_H / 2, synthetic.IMAGE_W, synthetic.IMAGE_H) for i in range(n)]


def run_workload(args):
    import torch.distributed as dist
    from cropnerf_b200 import export, synthetic
    from cropnerf_b200.rays import RayBundle

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    sys.stdout.flush()
    saved_stdout = os.dup(1)
    os.dup2(2, 1)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    assert args.gpus == world, f"--gpus {args.gpus} but WORLD_SIZE={world}"
    model = build_export_model(dev, args.precision)
    peak, peak_src = load_peaks()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    clocks = ClockSampler(local_rank)
    if args.workload == "export":
        B = args.export_batch
        nb = 16
        gen = torch.Generator().manual_seed(4242 + rank)
        host = [synthetic.make_rays(B, seed=7000 + 100 * rank + i, num_cameras=NUM_IMAGES) for i in range(nb)]
        batches = [RayBundle(h["origins"].to(dev), h["directions"].to(dev), h["pixel_area"].to(dev), h["camera_indices"].to(dev)) for h in host]
        obb = export.OrientedBox.from_params(*EXPORT_OBB)

        def next_rays(i):
            b = batches[i % nb]
            return RayBundle(b.origins, b.directions, b.pixel_area, b.camera_indices)

        export.generate_point_cloud(model, next_rays, 4 * B // 8, crop_obb=obb, rank=0, world_size=1)   # warm-up
        barrier()
        if rank == 0:
            clocks.start()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record()
        got = export.generate_point_cloud(model, next_rays, args.points, crop_obb=obb, rank=rank, world_size=world)
        e1.record()
        barrier()
        wall = time.perf_counter() - t0
        clk = clocks.stop() if rank == 0 else None
        t_local = e0.elapsed_time(e1) / 1e3
        stats = torch.tensor([t_local, wall, float(got["rays_rendered"]), float(got["points"].shape[0]), float(got["rays_needed"])], device=dev, dtype=torch.float64)
        mx = stats.clone()
        if world > 1:
            dist.all_reduce(mx, op=dist.ReduceOp.MAX)
            dist.all_reduce(stats, op=dist.ReduceOp.SUM)
        t, wall_max = float(mx[0]), float(mx[1])
        rays, pts, needed = (float(stats[2]), float(stats[3]), float(stats[4])) if world > 1 else (float(got["rays_rendered"]), float(got["points"].shape[0]), float(got["rays_needed"]))
        line = {"metric": "export_render_rays_per_s", "value": rays / t, "unit": "rays/s", "n_gpus": world, "steps": 1, "warmup": 1, "ms_per_step": 1e3 * t,
                "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32" if args.precision == "fp32" else "f16 tensor-core MLPs, f32 hash tables / compositing",
                "data": "synthetic",
                "config": {"workload": f"BASELINE configs[2]: ns-export pointcloud, render rays until {args.points} semantic-filtered points lie inside the crop OBB, rays sharded over the ranks",
                           "rays_per_batch": B, "num_points": args.points, "precision": args.precision, "obb": EXPORT_OBB,
                           "l2": "inputs larger than L2: every 32768-ray batch streams ~90 MB of workspace besides the 74 MiB of tables"},
                "kept_points": pts, "kept_points_per_s": pts / t, "rays_rendered": rays, "rays_needed_by_reference_loop": needed, "hit_rate": pts / max(needed, 1.0),
                "wall_s": wall_max,
                "roofline": {"bound": "hbm", "kernel": "render (fused eval chain)", "achieved": RENDER_BYTES_PER_RAY * rays / t / 1e9, "peak": peak * world, "unit": "GB/s",
                             "frac": RENDER_BYTES_PER_RAY * rays / t / 1e9 / (peak * world), "traffic": None, "peak_source": peak_src},
                "e2e": {"value": rays / wall_max, "unit": "rays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 4 * int(got["batches"]),
                        "note": "wall clock of generate_point_cloud (host loop + the asynchronous 4-byte count read-backs); the rays come from device-resident batches"},
                "gpu_launches": int(got["batches"]) * 10, "clocks": clk}
    else:
        cams = synthetic_cameras(args.views)
        g = torch.Generator().manual_seed(11)
        clusters = []
        for k in range(args.super_clusters):
            c = (torch.rand((2, 3), generator=g) - 0.5) * 0.6
            half = 0.04 + 0.03 * torch.rand((2, 3), generator=g)
            clusters.append({"aabb": torch.stack([c - half, c + half], dim=1).numpy(), "pcd": {}})
        export.project_clusters(model, cams[:2], clusters[:1], None)   # warm-up
        barrier()
        if rank == 0:
            clocks.start()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record()
        st = export.project_clusters(model, cams, clusters, None, rank=rank, world_size=world)
        e1.record()
        barrier()
        wall = time.perf_counter() - t0
        clk = clocks.stop() if rank == 0 else None
        stats = torch.tensor([e0.elapsed_time(e1) / 1e3, wall, float(st["rays"]), float(st["pairs"])], device=dev, dtype=torch.float64)
        mx = stats.clone()
        if world > 1:
            dist.all_reduce(mx, op=dist.ReduceOp.MAX)
            dist.all_reduce(stats, op=dist.ReduceOp.SUM)
        t, wall_max = float(mx[0]), float(mx[1])
        rays, pairs = float(stats[2]), float(stats[3])
        npix = cams[0].width * cams[0].height
        line = {"metric": "projection_render_rays_per_s", "value": rays / t, "unit": "rays/s", "n_gpus": world, "steps": 1, "warmup": 1, "ms_per_step": 1e3 * t,
                "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32" if args.precision == "fp32" else "f16 tensor-core MLPs, f32 hash tables / compositing",
                "data": "synthetic",
                "config": {"workload": f"BASELINE configs[3]: semantic_projection over {args.views} 1080p views x {args.super_clusters} super-clusters (2 sub-cluster boxes each), "
                                       "(super-cluster, view) pairs sharded over the ranks", "views": args.views, "super_clusters": args.super_clusters, "precision": args.precision,
                           "l2": "inputs larger than L2 (tables 74 MiB + per-chunk workspace)"},
                "pairs": pairs, "pairs_per_s": pairs / t, "pixels_tested_per_s": pairs * npix / t, "rays_rendered": rays, "wall_s": wall_max,
                "roofline": {"bound": "hbm", "kernel": "render (fused eval chain)", "achieved": RENDER_BYTES_PER_RAY * rays / t / 1e9, "peak": peak * world, "unit": "GB/s",
                             "frac": RENDER_BYTES_PER_RAY * rays / t / 1e9 / (peak * world), "traffic": None, "peak_source": peak_src},
                "e2e": {"value": rays / wall_max, "unit": "rays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 4 * int(pairs),
                        "note": "wall clock of project_clusters without the PNG encode (out_dir=None): ray generation, hit-count read-back, two renders and the scatter per pair"},
                "gpu_launches": int(pairs) * 30, "clocks": clk}
    if rank == 0:
        sys.stdout.flush()
        os.dup2(saved_stdout, 1)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def cpu_baseline(sample_rays: int, steps: int, warmup: int):
    """The oracle (port of the reference's torch path) timed on the host cores: one training step (fwd+bwd) of
    `sample_rays` rays of the same workload.  The only place bench.py executes oracle/."""
    from cropnerf_b200 import synthetic
    from oracle import cases

    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    cfg = cases.make_config({}, small=False)
    model, _ = cases.build_oracle(cfg, NUM_IMAGES, 0, 0.5)
    model.train()
    rays = synthetic.make_rays(sample_rays, seed=5, num_cameras=NUM_IMAGES)
    tgt = synthetic.make_targets(sample_rays, seed=6)
    times = []
    opt = torch.optim.Adam(model.parameters(), lr=1e-2, eps=1e-15)  # fruit_nerf_config.py:45-60
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        opt.zero_grad(set_to_none=True)
        out = model(cases.oracle_bundle(rays))
        metrics = model.get_metrics_dict(out, tgt)  # psnr + distortion, computed every step by the Trainer (fruit_nerf.py:639-645)
        loss = sum(model.get_loss_dict(out, tgt).values())
        loss.backward()
        opt.step()
        dt = time.perf_counter() - t0
        if i >= warmup:
            times.append(dt)
    t = sum(times) / len(times)
    # BASELINE configs[0]: the reference's own CPU-runnable case -- field forward + volume render (eval mode, no gradients) of the same rays;
    # the denominator for the `render` numbers of the product line
    model.eval()
    rtimes = []
    with torch.no_grad():
        for i in range(1 + max(1, min(steps, 3))):
            t0 = time.perf_counter()
            model(cases.oracle_bundle(rays))
            if i >= 1:
                rtimes.append(time.perf_counter() - t0)
    tr = sum(rtimes) / len(rtimes)
    return {"value": sample_rays / t, "unit": "rays/s", "cores": cores, "kind": "port",
            "sample": f"{sample_rays}-ray training step (fwd + losses/metrics + bwd + Adam) of the same fruit_nerf preset, torch {torch.__version__} CPU, "
                      f"{warmup} warm-up + mean of {steps}", "seconds_per_step": t,
            "render": {"value": sample_rays / tr, "unit": "rays/s", "seconds_per_call": tr,
                       "sample": f"eval forward + volume render of the same {sample_rays} rays (BASELINE configs[0]), 1 warm-up + mean of {len(rtimes)}"}}


def run_reference(args):
    """`--impl reference`: the reference's CPU implementation of the path = the oracle port (nerfstudio itself cannot be
    installed here), all host threads, bounded sample per step."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    sample = args.cpu_rays
    res = cpu_baseline(sample_rays=sample, steps=args.steps, warmup=max(1, min(args.warmup, 3)))
    line = {
        "impl": "reference", "metric": "train_rays_per_s", "value": res["value"], "unit": "rays/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * res["seconds_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": workload_config(),
        "detail": {"rays_per_step": sample, "precision": "fp32", "cores": res["cores"]},
        "cpu_baseline": res,
        "e2e": {"value": res["value"], "unit": "rays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--precision", default=os.environ.get("CNB_PRECISION", "mixed"), choices=["fp32", "mixed"],
                    help="mixed = fp16 tensor-core MLPs like the reference's autocast training (fruit_nerf_config.py:35); fp32 = exact mode")
    ap.add_argument("--no-graph", action="store_true", help="launch every kernel of the step eagerly instead of replaying a CUDA graph")
    ap.add_argument("--single-precision", action="store_true", help="skip the short pass in the other precision mode")
    ap.add_argument("--cpu-rays", type=int, default=RAYS_PER_GPU, help="rays per CPU-baseline step (default: the full 4096-ray batch of the workload, ~1.1 s per step on 16 cores)")
    ap.add_argument("--no-device-batches", action="store_true", help="skip the leg that trains from DeviceTrainBatches (2.5 GB of synthetic images in HBM)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--ddp", default=os.environ.get("CNB_DDP", "auto"), choices=["auto", "nccl", "p2p", "p2p_multimem"],
                    help="N>1: gradient exchange + Adam = NCCL all-reduce then local Adam, or one reduce-scatter+Adam+all-gather kernel over NVLink peer memory")
    ap.add_argument("--workload", default="train", choices=["train", "export", "projection"],
                    help="train = BASELINE configs[1] (the headline line); export = configs[2] (ns-export pointcloud); projection = configs[3] (semantic_projection)")
    ap.add_argument("--points", type=int, default=10_000_000, help="--workload export: semantic-filtered points to collect (whole job)")
    ap.add_argument("--export-batch", type=int, default=32768, help="--workload export: rays per rendered batch")
    ap.add_argument("--views", type=int, default=300, help="--workload projection: 1080p views")
    ap.add_argument("--super-clusters", type=int, default=2, help="--workload projection: super-clusters (2 sub-cluster boxes each)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last one returned (loss / metric scalars) and the "
                                                          "parameters it updated (a fixed sample of the large groups) as DIR/<name>.npy, float32, under 64 MB")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "b200" or args.workload != "train"):
        ap.error("--dump-outputs writes the outputs of the CUDA training step: it needs --impl b200 --workload train")
    if args.impl == "reference":
        run_reference(args)
    elif args.workload != "train":
        run_workload(args)
    else:
        run_product(args)


if __name__ == "__main__":
    main()
