"""Time the proposal-network density operators alone at the benchmark's shapes.

    python tests/time_proposal_bwd.py [--calls 200] [--out DIR] [--dump DIR]

The fruit_nerf preset has two proposal networks, each a 5-level hash grid of 2^17 rows per level (max resolution 128 and 256),
hidden width 16, evaluated at 256 and 96 samples on each of 4096 rays.  For each network and precision the script times
``cnb_density_field_bwd_kept`` (the training step's proposal backward: MLP recompute from the kept features, MLP parameter
gradients, table-gradient scatter) and ``cnb_density_field_fwd_keep`` (the forward that keeps those features).

Rays start inside the unit box in random directions; samples are spaced like the proposal sampler's first pass (uniform in the
piecewise linear-disparity space between near 0.05 and far 1000, jittered), under the scene contraction.  Parameters and the
upstream gradient are seeded.  Each operator is captured in a CUDA graph of 20 back-to-back calls; a replay is bracketed by
CUDA events, and the per-call time is the median over ``--calls`` replays divided by 20.  The cases are interleaved replay by
replay.  Prints one JSON line with the GPU's name and power limit; with --out DIR also writes DIR/proposal_bwd.json.  With
--dump DIR, writes the gradients of one backward call from zero (table, W1, b1, W2, b2) of each case to DIR/<case>.pt, so two
builds can be compared on the same inputs."""
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

from cropnerf_b200 import _lib as L  # noqa: E402
from cropnerf_b200 import ops  # noqa: E402
from oracle import nerfstudio_torch as ns  # noqa: E402

RAYS, LEVELS, LOG2_T, HIDDEN = 4096, 5, 17, 16
NETS = {"proposal0": (256, 128), "proposal1": (96, 256)}   # samples per ray, max resolution
NEAR, FAR = 0.05, 1000.0
PER_GRAPH = 20
PARAMS = ("table", "W1", "b1", "W2", "b2")


def gpu_info():
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True, timeout=30)
        info["power_limit_and_max_sm_clock"] = q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else None
    except (OSError, subprocess.TimeoutExpired):
        info["power_limit_and_max_sm_clock"] = None
    return info


def lindisp_piecewise(x):
    return torch.where(x < 1.0, x * 0.5, 1.0 - 1.0 / (2.0 * x))


def lindisp_piecewise_inv(x):
    return torch.where(x < 0.5, 2.0 * x, 1.0 / (2.0 - 2.0 * x))


def make_case(S, max_res, precision, dev, seed):
    g = torch.Generator().manual_seed(seed)
    u = lambda *shape: torch.rand(shape, generator=g) * 2 - 1  # noqa: E731
    T = 2**LOG2_T
    origins = u(RAYS, 3) * 0.6
    directions = torch.nn.functional.normalize(torch.randn((RAYS, 3), generator=g), dim=-1)
    bins = torch.linspace(0.0, 1.0, S + 1).expand(RAYS, S + 1).clone()
    bins[:, 1:-1] += (torch.rand((RAYS, S - 1), generator=g) - 0.5) / S
    s_near, s_far = lindisp_piecewise(torch.tensor(NEAR)), lindisp_piecewise(torch.tensor(FAR))
    edges = lindisp_piecewise_inv(bins * s_far + (1.0 - bins) * s_near)
    t = {
        "origins": origins, "directions": directions, "starts": edges[:, :-1].contiguous(), "ends": edges[:, 1:].contiguous(),
        "table": u(LEVELS * T, 2) * 0.5, "W1": u(HIDDEN, 2 * LEVELS) * (6.0 / (2 * LEVELS)) ** 0.5, "b1": u(HIDDEN) * 0.2,
        "W2": u(1, HIDDEN) * (6.0 / HIDDEN) ** 0.5, "b2": u(1) * 0.2,
    }
    dd = torch.rand(RAYS * S, generator=g) * 2.0 - 0.5
    dd[torch.rand(RAYS * S, generator=g) < 0.1] = 0.0
    t = {k: v.to(dev).contiguous() for k, v in t.items()}
    grads = {k: torch.zeros_like(t[k]) for k in PARAMS}
    f = L.DensityField()
    f.grid = L.make_grid(t["table"], grads["table"], LEVELS, LOG2_T, ns.hash_scalings(LEVELS, 16, max_res).tolist())
    f.mlp = L.make_mlp([t["W1"], t["W2"]], [t["b1"], t["b2"]], L.ACT_NONE, [grads["W1"], grads["W2"]], [grads["b1"], grads["b2"]])
    f.warp = L.make_warp(True, [[-1.0] * 3, [1.0] * 3])
    f.average_init_density = 1.0
    f.precision = L.PREC_MIXED if precision == "mixed" else L.PREC_FP32
    sm = ops.make_samples(t["origins"], t["directions"], t["starts"], t["ends"], None, RAYS, S, S)
    case = {"f": f, "sm": sm, "t": t, "grads": grads, "dd": dd.to(dev), "density": torch.empty(RAYS * S, device=dev),
            "feat": torch.empty(LEVELS * RAYS * S * 2, device=dev)}
    fwd(case)()
    torch.cuda.synchronize()
    return case


def fwd(c):
    def call():
        L.check(L.lib().cnb_density_field_fwd_keep(C.byref(c["f"]), C.byref(c["sm"]), c["density"].data_ptr(), c["feat"].data_ptr(), L.stream_ptr()),
                "fwd_keep")
    return call


def bwd(c):
    def call():
        L.check(L.lib().cnb_density_field_bwd_kept(C.byref(c["f"]), C.byref(c["sm"]), c["dd"].data_ptr(), c["feat"].data_ptr(), L.stream_ptr()),
                "bwd_kept")
    return call


def graph_of(fn):
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for _ in range(3):
            fn()
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    gr = torch.cuda.CUDAGraph()
    with torch.cuda.graph(gr):
        for _ in range(PER_GRAPH):
            fn()
    torch.cuda.synchronize()
    return gr


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--calls", type=int, default=200, help="graph replays per operator")
    ap.add_argument("--out", help="directory for proposal_bwd.json")
    ap.add_argument("--dump", help="directory for the gradients of one backward call per case")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "time_proposal_bwd.py needs a CUDA device"
    dev = torch.device("cuda:0")
    L.lib()
    cases = {f"{net}_{prec}": make_case(S, res, prec, dev, seed=i)
             for i, (net, (S, res)) in enumerate(NETS.items()) for prec in ("mixed", "fp32")}
    if args.dump:
        os.makedirs(args.dump, exist_ok=True)
        for name, c in cases.items():
            for gt in c["grads"].values():
                gt.zero_()
            bwd(c)()
            torch.cuda.synchronize()
            torch.save({k: v.cpu() for k, v in c["grads"].items()}, os.path.join(args.dump, name + ".pt"))
    graphs = {}
    for name, c in cases.items():
        graphs[name + "/bwd_kept"] = graph_of(bwd(c))
        graphs[name + "/fwd_keep"] = graph_of(fwd(c))
    times = {k: [] for k in graphs}
    for _ in range(args.calls):
        for k, gr in graphs.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            gr.replay()
            e1.record()
            e1.synchronize()
            times[k].append(1e3 * e0.elapsed_time(e1) / PER_GRAPH)
    res = {
        "what": f"per-call time of the proposal density operators, {RAYS} rays, {LEVELS} levels x 2^{LOG2_T} rows, hidden {HIDDEN}, "
                f"median (min) over {args.calls} replays of a {PER_GRAPH}-call CUDA graph",
        "gpu": gpu_info(),
        "us_per_call": {k: {"median": round(statistics.median(v), 2), "min": round(min(v), 2)} for k, v in times.items()},
    }
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "proposal_bwd.json"), "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
