"""bench.py contract (CPU part): the reference arm prints exactly one JSON line on stdout with the keys the driver reads."""
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..")


def test_reference_arm_prints_one_json_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "1", "--steps", "1",
                        "--warmup", "0", "--batch", "4"], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, r.stdout
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "MIQP plans/sec at 1e-4 gap" and d["unit"] == "plans/s"
    assert d["higher_is_better"] is True and d["value"] > 0 and d["n_gpus"] == 1 and d["steps"] == 1
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "plans/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"]


def test_device_arm_refuses_to_run_without_a_gpu():
    import torch
    if torch.cuda.is_available():
        return
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "0", "--batch", "2"],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode != 0 and "no CPU fallback" in (r.stderr + r.stdout)


def test_both_arms_share_one_config_object_and_every_workload_refuses_without_gpu():
    """`config` must be identical in the GPU arm and the reference arm (the driver compares them); what differs per run lives in
    `run`.  The multi-agent workloads have no CPU fallback either."""
    import importlib.util
    import torch
    spec = importlib.util.spec_from_file_location("_bench_mod", os.path.join(ROOT, "bench.py"))
    # bench.py redirects fd 1 at import: load it in a child process instead and ask for the config there
    code = ("import json, os, sys, importlib.util; "
            f"spec = importlib.util.spec_from_file_location('b', {os.path.join(ROOT, 'bench.py')!r}); "
            "b = importlib.util.module_from_spec(spec); spec.loader.exec_module(b); "
            "h = b.gap_histogram([type('I', (), dict(status=0, gap=g))() for g in (0.0, 5e-5, 5e-4, 0.05, 0.5, 3.0)] + "
            "[type('I', (), dict(status=1, gap=float('nan')))()], 1e-4); "
            "b.emit({'config': b.bench_config(2048), 'hist': h, 'workloads': sorted(b.WORKLOADS)})")
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads(r.stdout.strip().splitlines()[-1])
    assert set(d["config"]) == {"workload", "plans_per_gpu_per_step", "gap", "seeds", "cache"} and d["config"]["plans_per_gpu_per_step"] == 2048
    assert d["hist"] == {"<=0.0001": 2, "<=1e-3": 1, "<=1e-2": 0, "<=1e-1": 1, "<=1": 1, ">1": 1, "no incumbent": 1}
    assert d["workloads"] == ["config3", "config4", "config5"]
    if not torch.cuda.is_available():
        for wl in ("config3", "config4", "config5"):
            rr = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", wl, "--steps", "1", "--warmup", "0"],
                                capture_output=True, text=True, timeout=600)
            assert rr.returncode != 0 and "no CPU fallback" in (rr.stderr + rr.stdout), wl


def test_dump_outputs_writes_float_arrays_of_a_fixed_sample_within_64_mb(tmp_path):
    """--dump-outputs: one row per plan in every array, float32/64 only, at most 64 MB in all; a batch too large for that is
    sampled, and the sample is the same on every run (outputs of two builds are compared row for row)."""
    code = ("import importlib.util, sys, types; import numpy as np; "
            f"spec = importlib.util.spec_from_file_location('b', {os.path.join(ROOT, 'bench.py')!r}); "
            "b = importlib.util.module_from_spec(spec); spec.loader.exec_module(b); "
            "n, ncols = int(sys.argv[1]), 4160; "
            "info = lambda k: types.SimpleNamespace(status=0, proven=True, objective=1.0 + k, best_bound=1.0 + k, gap=0.0, max_violation=1e-9); "
            "s = types.SimpleNamespace(fetch=lambda: ([k + np.arange(ncols) / ncols for k in range(n)], [info(k) for k in range(n)])); "
            "[b.dump_outputs(d, s, [100 + k for k in range(n)]) for d in sys.argv[2:]]")
    for n in (4, 2048):
        dirs = [tmp_path / f"{n}_a", tmp_path / f"{n}_b"]
        r = subprocess.run([sys.executable, "-c", code, str(n)] + [str(d) for d in dirs], capture_output=True, text=True, timeout=300)
        assert r.returncode == 0, r.stderr[-2000:]
        files = sorted(p.name for p in dirs[0].iterdir())
        assert files == sorted(["x.npy", "plan_seed.npy", "status.npy", "proven.npy", "objective.npy", "best_bound.npy", "gap.npy",
                                "max_violation.npy"])
        assert sum(p.stat().st_size for p in dirs[0].iterdir()) <= 64_000_000
        a = {f: np.load(dirs[0] / f) for f in files}
        assert all(v.dtype in (np.float32, np.float64) for v in a.values())
        seeds = a["plan_seed.npy"]
        assert (len(seeds) == n) if n == 4 else (1800 < len(seeds) < n)
        assert np.array_equal(seeds, np.unique(seeds)) and a["x.npy"].shape == (len(seeds), 4160)
        assert np.array_equal(a["x.npy"][:, 0], seeds - 100) and np.array_equal(a["objective.npy"], seeds - 99)
        assert all(np.array_equal(v, np.load(dirs[1] / f)) for f, v in a.items())


def test_bench_rejects_zero_steps():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "0"],
                       capture_output=True, text=True, timeout=300)
    assert r.returncode != 0 and "--steps" in r.stderr
