"""The bench contract on the CPU arm: `bench.py --impl reference` prints exactly ONE stdout line, valid JSON, with the
keys the driver reads (metric, value, unit, n_gpus, steps, warmup, ms_per_step, higher_is_better, scaling, vs_baseline,
dtype, data, config.workload, impl, cpu_baseline, e2e).  Runs the oracle on a scene small enough for a few seconds."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                        "--gaussians", "4000", "--width", "160", "--height", "96"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, r.stdout
    d = json.loads(lines[0])
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
              "dtype", "data", "config", "impl", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["impl"] == "reference" and d["unit"] == "views/s" and d["higher_is_better"] is True
    assert d["value"] > 0 and d["cpu_baseline"]["kind"] in ("port", "reference") and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert "workload" in d["config"]


def test_metric_matches_baseline_json():
    base = json.load(open(os.path.join(ROOT, "BASELINE.json")))
    src = open(os.path.join(ROOT, "bench.py")).read()
    assert base["metric"].split()[0] in src or "views" in src


def _bench_module():
    import importlib.util
    spec = importlib.util.spec_from_file_location("bench_under_test", os.path.join(ROOT, "bench.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


def test_clock_sampler_keeps_the_samples_stamped_inside_the_timed_region(tmp_path, monkeypatch):
    """ClockSampler against a stand-in nvidia-smi that prints stamped CSV lines in nvidia-smi's format: only samples whose
    timestamp lies between mark_begin() and mark_end() are reported; with none inside, the warm-up samples are and it says so;
    a throttle reason seen inside the region is listed."""
    import time
    fake = tmp_path / "nvidia-smi"
    fake.write_text("#!" + sys.executable + "\n"
                    "import datetime, time\n"
                    "n = 0\n"
                    "while True:\n"
                    "    t = datetime.datetime.now().strftime('%Y/%m/%d %H:%M:%S.%f')[:-3]\n"
                    "    cap = 'Active' if n >= 12 else 'Not Active'\n"
                    "    print(f'{t}, 0, 1965, 1965, 700.1, 0x0000000000000004, Not Active, Not Active, Not Active, {cap}', flush=True)\n"
                    "    n += 1\n"
                    "    time.sleep(0.02)\n")
    fake.chmod(0o755)
    monkeypatch.setenv("PATH", str(tmp_path) + os.pathsep + os.environ.get("PATH", ""))
    bench = _bench_module()
    s = bench.ClockSampler(0)
    s.start()
    time.sleep(0.6)
    s.mark_begin()
    time.sleep(0.3)
    s.mark_end()
    out = s.stop()
    assert out["window"] == "timed region" and 5 <= out["samples"] < out["samples_total"]
    assert out["sm_mhz"] == 1965.0 and out["sm_max_mhz"] == 1965.0 and out["reasons"] == ["sw_power_cap"]
    s = bench.ClockSampler(0)
    s.start()
    time.sleep(0.4)
    s.mark_begin(); s.mark_end()
    out = s.stop()
    assert out["samples"] == out["samples_total"] > 0 and out["window"].startswith("warm-up")
    assert bench.ClockSampler._stamp("2026/09/24 00:53:12.345") is not None and bench.ClockSampler._stamp("N/A") is None


def test_path_bytes_count_only_the_launched_stages():
    """stage_bytes lists every variant (16- and 32-bit tile keys, level A's scatter); the whole-path figure must be the sum over
    the stages a run launched, and project_backward is charged on the Gaussians that carry a gradient."""
    bench = _bench_module()
    st = {"Nv": 984960, "Nmax": 1000064, "D": 10897674, "P": 2073600, "N_visible": 923397, "tiles": 16200, "tile_sort_passes": 2,
          "N_grad": 108250}
    b = bench.stage_bytes(st, 128, 16)
    assert b["lgs_project_backward"] == 48 * st["Nv"] + (44 + 2 * 236) * st["N_grad"]
    st2 = dict(st); del st2["N_grad"]
    assert bench.stage_bytes(st2, 128, 16)["lgs_project_backward"] == 48 * st["Nv"] + (44 + 2 * 236) * st["Nv"]
    src = open(os.path.join(ROOT, "bench.py")).read()
    assert "sum(v for k, v in bytes_per.items())" not in src


def test_dump_outputs_writes_the_step_results_at_a_fixed_sample(tmp_path):
    """--dump-outputs: float32 .npy per returned array, gradients at the same seeded Gaussian sample on every call."""
    import numpy as np
    import torch
    bench = _bench_module()
    C, S = 600, 128
    n = C * S
    g = torch.Generator().manual_seed(0)
    shapes = {"xyz": (3,), "scale": (3,), "rot": (4,), "sh_0": (1, 3), "sh_rest": (15, 3), "opacity": (1,)}
    grads = {k: torch.randn((*s, C, S), generator=g) for k, s in shapes.items()}
    grads["_touched"] = torch.ones(C)
    losses = [torch.tensor(1.5), torch.tensor(-2.0)]
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), losses, grads)
    names = sorted(f for f in os.listdir(tmp_path / "a"))
    assert names == sorted(["losses.npy", "touched.npy"] + [f"grad_{k}.npy" for k in shapes])
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in names) <= 64 << 20
    for f in names:
        a, b = np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f)
        assert a.dtype == np.float32 and np.array_equal(a, b), f
    assert np.array_equal(np.load(tmp_path / "a" / "losses.npy"), [1.5, -2.0])
    x = np.load(tmp_path / "a" / "grad_sh_rest.npy")
    assert x.shape == (15, 3, bench.DUMP_SAMPLE)
    idx = np.sort(np.random.default_rng(0).choice(n, bench.DUMP_SAMPLE, replace=False))
    assert np.array_equal(x, grads["sh_rest"].reshape(15, 3, n).numpy()[..., idx])
