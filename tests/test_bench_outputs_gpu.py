"""``bench.py --dump-outputs DIR``: after the timed steps the benchmark writes what its last timed training step returned and the parameters
that step left, as float32 ``DIR/<name>.npy`` under 64 MB, so that two builds run with the same arguments can be compared array by array."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
STATS = {"loss", "rgb_loss", "semantics_loss", "interlevel_loss", "distortion", "psnr", "camera_opt_regularizer"}


@pytest.mark.gpu
def test_bench_dumps_the_last_timed_step(tmp_path):
    import torch

    sys.path.insert(0, ROOT)
    import bench

    dump = tmp_path / "out"
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "3", "--warmup", "3", "--single-precision",
           "--no-device-batches", "--no-cpu-baseline", "--dump-outputs", str(dump)]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=1200, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-3000:]
    line = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1])
    assert line["steps"] == 3
    files = sorted(dump.glob("*.npy"))
    arrays = {p.stem: np.load(p) for p in files}
    assert set(arrays) == STATS | {"params_proposal_networks", "params_fields_sample"}
    assert all(a.dtype == np.float32 and np.isfinite(a).all() for a in arrays.values())
    assert sum(p.stat().st_size for p in files) <= 64e6
    assert arrays["loss"] > 0 and arrays["rgb_loss"] > 0
    # the dumped parameters are the benchmark model's flat groups after training: the whole proposal group, which moved from its initial
    # values, and a sample of the field group of its share of the budget
    from cropnerf_b200.engine import FlatGroup

    model = bench.build_model(torch.device("cuda:0"), "mixed")
    groups = {n: FlatGroup(p) for n, p in model.get_param_groups().items() if p}
    init = groups["proposal_networks"].flat.cpu().numpy()
    assert arrays["params_proposal_networks"].shape == init.shape and (arrays["params_proposal_networks"] != init).any()
    assert groups["fields"].flat.numel() > bench.DUMP_PARAM_FLOATS // len(groups) == arrays["params_fields_sample"].size
