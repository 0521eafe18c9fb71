"""bench.py contract: the JSON line both arms print (CPU arm executed here; the GPU arm's committed line checked)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from tests.util import ROOT

BASE = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
        "dtype", "data", "config", "e2e", "cpu_baseline"}


def test_reference_arm_prints_one_json_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1"],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert BASE <= set(d) and d["impl"] == "reference" and d["value"] > 0
    assert d["metric"] == "snake_env_steps_per_sec" and d["unit"] == "env-steps/s" and d["higher_is_better"] is True
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["vs_baseline"] is None and "workload" in d["config"]
    assert d["config"]["envs_per_bench_step"] == 32768 and len(d["config"]["differences_from_the_gpu_arm"]) == 3


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1"],
                         capture_output=True, text=True, timeout=120, cwd=ROOT, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""


@pytest.mark.gpu
def test_dumped_outputs_repeat_from_run_to_run(tmp_path):
    """--dump-outputs writes what the last timed step returned; two runs with the same arguments write the same arrays, on
    the CUDA-graph path (small env counts) and on the one-launch-per-step path, where a seeded sample of envs is written"""
    for envs, steps, written in ((4096, 7, 4096), (400000, 5, 65536)):
        dumps = []
        for run in range(2):
            d = tmp_path / ("%d_%d" % (envs, run))
            out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(steps), "--warmup", "3",
                                  "--envs", str(envs), "--e2e-steps", "2", "--skip-cpu", "--skip-config2", "--skip-config4",
                                  "--skip-gram", "--skip-variants", "--dump-outputs", str(d)],
                                 capture_output=True, text=True, timeout=600, cwd=ROOT)
            assert out.returncode == 0, out.stderr[-2000:]
            line = json.loads(out.stdout.strip().splitlines()[-1])
            assert line["steps"] == steps and line["config"]["env_errors"] == 0
            dumps.append({f.stem: np.load(f) for f in d.iterdir()})
        a, b = dumps
        assert set(a) == {"env_index", "act_idx", "reward", "done", "mask", "obs"}
        assert all(x.dtype in (np.float32, np.float64) for x in a.values()) and sum(x.nbytes for x in a.values()) <= 64 << 20
        assert a["obs"].shape == (written, 2, 10, 10) and a["mask"].shape == (written, 3)
        assert set(np.unique(a["obs"])) <= {-1, 0, 1, 2} and set(np.unique(a["act_idx"])) <= {0, 1, 2}
        for name in a:
            assert np.array_equal(a[name], b[name]), name


def test_committed_gpu_line_has_the_contract_keys():
    for name in ("r01_bench_n1.json", "r02_bench_n1.json"):
        _check_gpu_line(os.path.join(ROOT, "profiles", name), round2=name.startswith("r02"))


def _check_gpu_line(p, round2):
    d = json.loads(open(p).read().strip().splitlines()[-1])
    assert BASE | {"roofline", "gpu_launches", "clocks"} <= set(d)
    if round2:
        assert d["clocks"]["samples"] >= 8 and d["clocks"]["sm_mhz"] is not None          # the sampler starts before the warm-up
        assert ("bits" in d["e2e"]["obs_format"] or "packed2" in d["e2e"]["obs_format"]) and "full_f32_obs_variant" in d["e2e"]
        c4 = d["config4_65536_envs"]
        assert c4["native_f32"]["max_err_vs_float64_of_maxQ"] < 2e-5 < c4["native_bf16"]["max_err_vs_float64_of_maxQ"]
        for t in ("terms3", "terms1"):
            r = d["gram_5a"][t]["roofline"]
            assert r["frac"] <= r["frac_executed"] + 1e-9 and r["traffic"] is not None      # frac = algorithmic FLOP, as the spec asks
        assert d["cpu_baseline"]["sample"].startswith("32768 envs")
    r = d["roofline"]
    assert r["bound"] == "hbm" and r["unit"] == "GB/s" and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9
    assert r["traffic"] is None or 0.5 < r["traffic"] / (876 * d["config"]["envs_per_gpu"]) < 1.5
    assert d["e2e"]["h2d_bytes_per_step"] > 0 and d["e2e"]["d2h_bytes_per_step"] > 0
    assert d["gpu_launches"] == d["steps"] * d["n_gpus"] and d["scaling"] == "weak"
    assert not set(d["clocks"]["reasons"]) & {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"}
