"""CPU tests of the measurement contract: the reference arm of bench.py runs without a GPU and prints one well-formed JSON
line, and the committed product-arm line (profiles/r1_final_bench_1gpu.json, produced on a B200) carries every key the
contract names, with self-consistent arithmetic (value = rays / time, roofline.frac = achieved / peak, ...)."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BASE_KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype", "data", "config"}


def test_reference_arm_prints_one_contract_line_on_cpu():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0", "--cpu-rays", "64"],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert BASE_KEYS <= set(d) and d["impl"] == "reference"
    assert d["metric"] == "train_rays_per_s" and d["unit"] == "rays/s" and d["higher_is_better"] is True and d["vs_baseline"] is None
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["cpu_baseline"]["render"]["value"] > 0 and d["cpu_baseline"]["render"]["unit"] == "rays/s"
    assert abs(d["value"] - d["detail"]["rays_per_step"] / (d["ms_per_step"] / 1e3)) < 1e-6 * d["value"]
    assert "workload" in d["config"] and "model" not in d["config"]
    # the reference arm names the product arm's workload: the very same `config` dict (the driver's same_config check)
    sys.path.insert(0, ROOT)
    import bench
    assert d["config"] == bench.workload_config()


def test_reference_arm_defaults_to_the_full_batch_of_the_workload():
    sys.path.insert(0, ROOT)
    import bench
    assert bench.RAYS_PER_GPU == 4096 and bench.workload_config()["rays_per_gpu"] == 4096
    src = open(os.path.join(ROOT, "bench.py")).read()
    assert '"--cpu-rays", type=int, default=RAYS_PER_GPU' in src
    assert 'os.environ["NCCL_DEBUG"]' not in src   # the driver reads NCCL's communicator lines


def test_reference_arm_non_zero_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", LOCAL_RANK="1", WORLD_SIZE="2")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, timeout=600, cwd=ROOT, env=env)
    assert out.returncode == 0 and not [l for l in out.stdout.splitlines() if l.startswith("{")]


def test_steps_sets_the_number_of_timed_steps():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "51", "--warmup", "0", "--cpu-rays", "16"],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    d = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1])
    assert d["steps"] == 51 and d["cpu_baseline"]["sample"].endswith("mean of 51")


def test_bad_arguments_are_refused_before_any_work(tmp_path):
    dump = tmp_path / "out"
    for extra in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", str(dump)], ["--workload", "export", "--dump-outputs", str(dump)]):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *extra], capture_output=True, text=True, timeout=300, cwd=ROOT)
        assert out.returncode == 2 and "error:" in out.stderr, (extra, out.stderr[-2000:])
    assert not dump.exists()


def test_committed_product_line_has_every_contract_key_and_consistent_arithmetic():
    path = os.path.join(ROOT, "profiles", "r2_bench_1gpu.json")
    if not os.path.exists(path):
        path = os.path.join(ROOT, "profiles", "r1_final_bench_1gpu.json")
    if not os.path.exists(path):
        pytest.skip("no committed bench line")
    d = json.loads(open(path).read().strip().splitlines()[-1])
    assert BASE_KEYS <= set(d) and d.get("impl", "b200") != "reference"
    assert d["n_gpus"] == 1 and d["scaling"] == "weak" and d["data"] == "synthetic" and d["vs_baseline"] is None and d["warmup"] >= 3
    rays = d["config"]["rays_per_gpu"] * d["n_gpus"]
    assert abs(d["value"] - rays / (d["ms_per_step"] / 1e3)) < 1e-6 * d["value"]
    assert abs(d["samples_per_s"] - d["value"] * d["config"]["samples_per_ray"]) < 1e-6 * d["samples_per_s"]
    r = d["roofline"]
    assert r["bound"] in ("hbm", "tensor") and r["unit"] in ("GB/s", "TFLOP/s") and r["peak_source"] in ("measured", "fallback")
    assert abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9
    assert abs(r["achieved"] - r["algorithmic_bytes_per_launch"] / (r["ms_per_launch"] * 1e-3) / 1e9) < 1e-6 * r["achieved"]
    assert r["traffic"] is None or r["traffic"] > 0
    # the field backward's algorithmic bytes: 2 x (48 samples x 16 levels x 8 corners x 8 B) per ray (SURVEY.md 8d, DESIGN.md 4)
    assert r["algorithmic_bytes_per_launch"] == 2 * 48 * 16 * 8 * 8 * d["config"]["rays_per_gpu"]
    s = d["step_roofline"]
    assert s["algorithmic_bytes_per_ray"] == 3 * (256 * 5 + 96 * 5 + 48 * 16) * 8 * 8 + 64 + 16
    assert abs(s["frac"] - d["value"] * s["algorithmic_bytes_per_ray"] / 1e9 / r["peak"]) < 1e-6
    c = d["cpu_baseline"]
    assert c["kind"] in ("port", "reference") and c["cores"] >= 1 and c["value"] > 0 and c["sample"]
    e = d["e2e"]
    assert 0 < e["value"] <= d["value"] * 1.001 and e["unit"] == d["unit"]
    # host rays in: origins + directions (2 x 12 B) + int64 camera index + rgb target (12 B) + mask (4 B) = 48 B per ray; loss out: 4 B
    assert e["h2d_bytes_per_step"] == 48 * d["config"]["rays_per_gpu"] and e["d2h_bytes_per_step"] == 4
    assert d["gpu_launches"] > 0 and d["gpu_launches"] % d["steps"] == 0
    k = d["clocks"]
    assert k["sm_mhz"] and k["sm_max_mhz"]
    if "sw_power_cap" not in k["reasons"]:   # a power-capped run is kept and noted; anything else must be near the maximum clock
        assert k["sm_mhz"] >= 0.9 * k["sm_max_mhz"]
    assert not set(k["reasons"]) & {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"}
