"""bench.py contract checks that need no GPU: the reference (CPU) arm prints ONE well-formed JSON line, non-zero
ranks of a torchrun launch stay silent, and the product arm refuses to run without a CUDA device."""
import json
import os
import subprocess
import sys

import torch

from conftest import ROOT

BENCH = os.path.join(ROOT, "bench.py")


def run(args, env_extra=None, timeout=900):
    env = dict(os.environ)
    env.update(env_extra or {})
    return subprocess.run([sys.executable, BENCH] + args, capture_output=True, text=True, env=env, cwd=ROOT,
                          timeout=timeout)


def test_reference_arm_prints_one_contract_line():
    r = run(["--impl", "reference", "--gpus", "1", "--steps", "1", "--warmup", "1"])
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, lines
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "rays/s" and d["higher_is_better"] is True
    assert d["metric"].startswith("rays/sec @ 128 samples") and d["n_gpus"] == 1 and d["steps"] == 1 and d["warmup"] == 1
    assert d["value"] > 0 and abs(d["value"] - 2048 / (d["ms_per_step"] * 1e-3)) < 1e-6 * d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "rays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["value"] == d["value"] and 1 <= cb["cores"] <= (os.cpu_count() or 1)
    assert "2048" in cb["sample"] and d["vs_baseline"] is None and d["data"] == "synthetic"


def test_reference_arm_non_zero_ranks_are_silent():
    r = run(["--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0"],
            {"RANK": "1", "LOCAL_RANK": "1", "WORLD_SIZE": "2"}, timeout=120)
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_product_arm_has_no_cpu_fallback():
    if torch.cuda.is_available():
        return
    r = run(["--gpus", "1", "--steps", "1", "--warmup", "1"], timeout=300)
    assert r.returncode != 0
    assert "no CUDA device" in (r.stderr + r.stdout)
    assert not any(l.lstrip().startswith("{") for l in r.stdout.splitlines())


def test_steps_and_dump_outputs_arguments_are_checked():
    for args, msg in ((["--steps", "0"], "--steps must be at least 1"),
                      (["--gpus", "2", "--dump-outputs", "dump"], "--dump-outputs"),
                      (["--impl", "reference", "--dump-outputs", "dump"], "--dump-outputs")):
        r = run(args, timeout=300)
        assert r.returncode == 2 and msg in r.stderr, (args, r.stderr[-2000:])
        assert r.stdout.strip() == ""
    assert not os.path.exists(os.path.join(ROOT, "dump"))


def test_clock_sampler_uses_only_lines_that_arrived_inside_the_window(tmp_path, monkeypatch):
    """The `clocks` object of the bench line: a stand-in nvidia-smi that needs 0.2 s to come up and then streams a line
    every 25 ms; only lines stamped inside [begin(), end()] count, a window that closes before the first line reports
    'no samples' (bench.py keeps the load running to 0.4 s so that this cannot happen in a real run)."""
    import importlib.util
    import time
    fake = tmp_path / "nvidia-smi"
    fake.write_text("#!/bin/bash\nsleep 0.2\nwhile true; do echo '0, 1965, 1980, 700.0, Not Active, Not Active, Not Active, Active'; "
                    "sleep 0.025; done\n")
    fake.chmod(0o755)
    monkeypatch.setenv("PATH", str(tmp_path) + os.pathsep + os.environ["PATH"])
    monkeypatch.setattr(sys, "argv", ["bench.py"])
    spec = importlib.util.spec_from_file_location("bench_under_test", BENCH)
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    s = bench.ClockSampler(0)
    s.start()
    time.sleep(0.6)
    s.begin(); time.sleep(0.2); s.end()
    out = s.stop()
    assert out["sm_mhz"] == 1965.0 and out["sm_max_mhz"] == 1980.0 and out["reasons"] == ["sw_power_cap"]
    assert 2 <= out["samples"] <= 12                               # ~8 lines in 0.2 s, none of the ~16 earlier ones
    s = bench.ClockSampler(0)
    s.start(); s.begin(); time.sleep(0.05); s.end()
    assert s.stop()["reasons"] == ["no samples"]
