"""The driver-facing contract of bench.py: one JSON line with the agreed keys, for the reference arm (CPU, any box)
and for the GPU arm (tiny run, -m gpu)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from tests.conftest import ROOT

BASE_KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
             "vs_baseline", "dtype", "data", "config", "e2e", "cpu_baseline", "gpu_launches"}


def _run(args, timeout=600):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, capture_output=True, text=True, timeout=timeout, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.strip().splitlines() if l.startswith("{")]
    assert len(lines) == 1, out.stdout[-2000:]
    return json.loads(lines[0])


def test_reference_arm_line():
    d = _run(["--impl", "reference", "--steps", "1", "--warmup", "1"])
    assert d["impl"] == "reference" and BASE_KEYS <= set(d)
    assert d["metric"].startswith("env-steps/sec") and d["unit"] == "env-steps/s" and d["higher_is_better"] is True
    assert d["vs_baseline"] is None and d["steps"] == 1 and d["value"] > 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and "model" not in d["config"]


@pytest.mark.gpu
def test_gpu_arm_line():
    # exactly --steps launches are timed, inside one event pair: 8000 of them (~4 us each) make a region of > 15 ms
    d = _run(["--steps", "8000", "--warmup", "3", "--no-vecenv", "--no-ppo", "--no-configs", "--sweep", "--rotating-handles", "8",
              "--cpu-budget", "2"])
    assert BASE_KEYS | {"roofline", "clocks"} <= set(d)
    assert d["n_gpus"] == 1 and d["steps"] == 8000 and d["gpu_launches"] == 8000 and d["timing"]["launches_in_timed_region"] == 8000
    assert d["scaling"] == "weak" and d["dtype"] == "f32" and d["timed_region_s"] >= 0.015
    assert d["pybullet_cpu"].startswith("n/a") and d["e2e_alternative"]["value"] > 0
    assert d["value"] > 1e8 and abs(d["ms_per_step"] * 1e-3 * d["value"] - 4096) < 1e-3 * 4096        # value = envs / time per step
    r = d["roofline"]
    assert r["bound"] == "hbm" and r["unit"] == "GB/s" and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9 and r["traffic"] is not None
    e = d["e2e"]
    assert e["h2d_bytes_per_step"] == 4096 * 16 and e["d2h_bytes_per_step"] == 4096 * (13 * 4 + 4 + 1 + 4) and 0 < e["value"] < d["value"]
    c = d["cpu_baseline"]
    assert c["kind"] == "port" and c["cores"] >= 1 and c["value"] > 0 and "sample" in c
    assert "workload" in d["config"] and "l2" in d["config"] and "model" not in d["config"]
    assert set(d["clocks"]) >= {"sm_mhz", "sm_max_mhz", "reasons"}


def _load_bench():
    import importlib.util
    spec = importlib.util.spec_from_file_location("_bench", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    return bench


@pytest.mark.gpu
def test_dump_outputs_depend_on_the_arguments_only(tmp_path):
    """--dump-outputs: the last timed step's obs / reward / done / found_targets, bit-identical for identical arguments;
    one more timed step changes them (--steps is the number of steps the timed path runs)."""
    quick = ["--warmup", "3", "--no-vecenv", "--no-ppo", "--no-configs", "--no-cpu", "--sweep", "--rotating-handles", "8"]
    dumps = {}
    for name, steps in (("a", 40), ("b", 40), ("c", 41)):
        d = _run(["--steps", str(steps), "--dump-outputs", str(tmp_path / name)] + quick)
        assert d["steps"] == steps and d["gpu_launches"] == steps
        dumps[name] = {f[:-4]: np.load(tmp_path / name / f) for f in sorted(os.listdir(tmp_path / name))}
    a, b, c = dumps["a"], dumps["b"], dumps["c"]
    assert sorted(a) == ["done", "found_targets", "obs", "reward"]
    assert a["obs"].shape == (4096, 13) and a["obs"].dtype == np.float32 and a["reward"].shape == (4096,)
    assert a["done"].dtype == np.float64 and set(np.unique(a["done"])) <= {0.0, 1.0, 2.0, 3.0}
    assert np.isfinite(a["obs"]).all() and np.isfinite(a["reward"]).all()
    for k in a:
        np.testing.assert_array_equal(a[k], b[k], err_msg=k)
    assert any(not np.array_equal(a[k], c[k]) for k in a)
    # what the last timed launch computed: 8 handles, K = 40 >= 8 so two graphs (untimed, timed), the last launch steps handle
    # 79 % 8 = 7; it has been stepped 24 times (warm-up rotations) + 5 (untimed graph) + 5 (timed graph), always with actions[7]
    import argparse
    import torch
    bench = _load_bench()
    env = bench.make_env(4096, argparse.Namespace(track="circle", substeps=8), torch.device("cuda", 0))
    env.reset()
    acts = bench.make_actions(8, 4096, "saturating", env.device, seed=4321)
    for _ in range(24 + 5 + 5):
        obs, reward, done, found = env.step(acts[7])
    for k, v in (("obs", obs), ("reward", reward), ("done", done), ("found_targets", found)):
        np.testing.assert_array_equal(a[k], v.cpu().numpy().astype(a[k].dtype), err_msg=k)
    env.close()


def test_dump_outputs_keep_a_fixed_sample_of_large_outputs(tmp_path):
    bench = _load_bench()
    n = 1 << 16
    rng = np.random.default_rng(3)
    arrays = {"obs": rng.standard_normal((n, 13)).astype(np.float32), "done": rng.integers(0, 4, n).astype(np.uint8),
              "found_targets": rng.integers(0, 1 << 20, n).astype(np.int32)}
    bench.dump_outputs(str(tmp_path / "all"), arrays)
    for k, v in arrays.items():
        got = np.load(tmp_path / "all" / (k + ".npy"))
        assert got.dtype == (np.float32 if v.dtype == np.float32 else np.float64)
        np.testing.assert_array_equal(got, v.astype(got.dtype))
    assert not (tmp_path / "all" / "env_index.npy").exists()
    limit = 1 << 20                                     # 1 MiB: the 65 536 rows of 68 bytes do not fit
    for name in ("s1", "s2"):
        bench.dump_outputs(str(tmp_path / name), arrays, limit=limit)
    files = sorted(os.listdir(tmp_path / "s1"))
    assert files == ["done.npy", "env_index.npy", "found_targets.npy", "obs.npy"]
    assert sum(os.path.getsize(tmp_path / "s1" / f) for f in files) <= limit
    idx = np.load(tmp_path / "s1" / "env_index.npy").astype(np.int64)
    assert (np.diff(idx) > 0).all() and idx[0] >= 0 and idx[-1] < n and len(idx) > n // 8
    for k, v in arrays.items():
        got = np.load(tmp_path / "s1" / (k + ".npy"))
        np.testing.assert_array_equal(got, v[idx].astype(got.dtype))
        np.testing.assert_array_equal(got, np.load(tmp_path / "s2" / (k + ".npy")))


def test_roofline_rows_find_the_committed_ncu_captures():
    """bench.py's per-variant roofline rows quote the ncu DRAM bytes of the SAME configuration from profiles/ncu_summary_r*.json:
    the lookup keys (envs, substeps, variant prefix) must match what tools/summarize_profiles*.py wrote."""
    bench = _load_bench()
    assert bench.ncu_traffic(4096, 8) == 560640.0                      # headline kernel, 4096 envs
    assert bench.ncu_traffic(4194304, 8) > 1.2e9 and bench.ncu_traffic(4194304, 1) > 1.1e9
    for envs, sub, variant in ((12, 1, "norm_"), (4096, 8, "norm_"), (16384, 8, "phys3_"), (131072, 8, "full_rw3_"),
                               (131072, 8, "full_rw8_"), (131072, 8, "full_rw9_")):
        assert bench.ncu_traffic(envs, sub, variant) is not None, (envs, sub, variant)
    assert bench.ncu_traffic(777, 8) is None and bench.ncu_traffic(4096, 8, "no_such_") is None
    r = bench.roofline(4096, 4e-6, substeps=8)
    assert r["bound"] == "hbm" and r["traffic"] == 560640.0 and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-12
    assert r["algorithmic_bytes_per_launch"] == 4096 * bench.BYTES_PER_ENV_STEP
