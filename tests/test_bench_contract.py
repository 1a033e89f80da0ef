"""bench.py's reference arm runs on the CPU, so the JSON contract of a bench line can be checked without a GPU:
one JSON line on stdout, the keys every bench line carries, the reference-arm additions, and a loud failure of the native arm.
The --dump-outputs files are checked here too, and against the native arm's on the GPU."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FIELDS = ("pose", "score", "grad", "hessian", "iterations", "status", "count")


def _run(*args):
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True, timeout=600, cwd=ROOT)


def _bench_module():
    import importlib.util
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    return bench


def test_reference_arm_prints_one_contract_line():
    r = _run("--impl", "reference", "--steps", "2", "--warmup", "1", "--ref-scans", "48")
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype",
              "data", "config", "e2e", "cpu_baseline", "impl"):
        assert k in d, k
    assert d["impl"] == "reference" and d["steps"] == 2 and d["warmup"] == 1 and d["higher_is_better"] is True
    assert d["metric"].startswith("NDT scan-matches/sec") and d["unit"] == "matches/s" and d["vs_baseline"] is None
    assert d["value"] > 0 and d["e2e"]["value"] == d["value"] and d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert "workload" in d["config"] and "model" not in d["config"]


def test_native_arm_fails_loudly_without_a_gpu():
    import torch
    if torch.cuda.is_available():
        import pytest
        pytest.skip("GPU present")
    r = _run("--steps", "1", "--warmup", "1")
    assert r.returncode != 0 and "no CPU fallback" in (r.stderr + r.stdout)


def test_upload_relay_plan_pairs_slow_ranks_with_fast_ones():
    """bench.plan_upload_relay / refine_upload_relay on the copy rates measured on the 8-GPU box (host logic only): the four
    23 GB/s ranks are paired with the four 35 GB/s ranks at x = (fast - slow) / (fast + slow), equal rates plan nothing, and
    the calibration step moves x towards equal step times."""
    bench = _bench_module()

    class Ctx:
        def __init__(self, rank, world):
            self.rank, self.world = rank, world

        def gather_floats(self, v):
            return [float(v)] * self.world

    class M:
        def __init__(self):
            self.calls = []

        def set_upload_relay(self, dev, frac=0.5):
            self.calls.append((dev, frac))

    gbs = [23.4, 23.5, 23.4, 23.5, 34.9, 35.3, 35.2, 35.3]
    m = M()
    plan = bench.plan_upload_relay(Ctx(0, 8), m, gbs)
    assert sorted(plan["pairs"]) == ["0", "1", "2", "3"]
    assert sorted(v["via_rank"] for v in plan["pairs"].values()) == [4, 5, 6, 7]
    assert all(0.19 < v["fraction"] < 0.21 for v in plan["pairs"].values())
    assert len(m.calls) == 1 and m.calls[0][0] == plan["pairs"]["0"]["via_rank"]
    m5 = M()
    assert bench.plan_upload_relay(Ctx(5, 8), m5, gbs) == plan and m5.calls == []      # a fast rank sets nothing
    assert bench.plan_upload_relay(Ctx(0, 2), M(), [55.3, 55.4]) is None
    assert bench.plan_upload_relay(Ctx(0, 1), M(), [50.0]) is None
    t = [11.6, 11.6, 11.6, 11.6, 10.0, 10.0, 10.0, 10.0]
    before = {k: v["fraction"] for k, v in plan["pairs"].items()}
    plan2 = bench.refine_upload_relay(Ctx(0, 8), m, plan, t)
    assert all(before[k] + 0.04 < v["fraction"] < before[k] + 0.10 for k, v in plan2["pairs"].items())
    assert len(m.calls) == 2 and abs(m.calls[1][1] - plan2["pairs"]["0"]["fraction"]) < 1e-3


def test_reference_arm_dumps_the_last_steps_records(tmp_path):
    """--dump-outputs: one float64 .npy per field of the result records, one row per scan, the same bytes on every run."""
    dirs = [tmp_path / "a", tmp_path / "b"]
    for d in dirs:
        r = _run("--impl", "reference", "--steps", "1", "--warmup", "0", "--ref-scans", "48", "--dump-outputs", str(d))
        assert r.returncode == 0, r.stderr[-2000:]
    assert sorted(os.listdir(dirs[0])) == sorted(f + ".npy" for f in FIELDS)
    for f in FIELDS:
        a, b = np.load(dirs[0] / (f + ".npy")), np.load(dirs[1] / (f + ".npy"))
        assert a.dtype == np.float64 and len(a) == 48 and a.tobytes() == b.tobytes(), f
    assert np.load(dirs[0] / "hessian.npy").shape == (48, 3, 3) and (np.load(dirs[0] / "iterations.npy") >= 1).all()


def test_dump_keeps_a_seeded_sample_within_the_budget(tmp_path, monkeypatch):
    from gtsam_ndt_b200 import RESULT_DTYPE
    bench = _bench_module()
    monkeypatch.setattr(bench, "DUMP_BUDGET", 64 << 10)
    res = np.zeros(1000, RESULT_DTYPE)
    res["score"] = np.arange(1000)
    for d in ("a", "b"):
        bench.dump_records(str(tmp_path / d), res)
    names = sorted(os.listdir(tmp_path / "a"))
    assert names == sorted(f + ".npy" for f in FIELDS + ("index",))
    assert sum(os.path.getsize(tmp_path / "a" / n) for n in names) <= 64 << 10
    idx = np.load(tmp_path / "a" / "index.npy")
    assert 100 < len(idx) < 1000 and (np.diff(idx) > 0).all() and np.array_equal(np.load(tmp_path / "a" / "score.npy"), idx)
    assert all((tmp_path / "a" / n).read_bytes() == (tmp_path / "b" / n).read_bytes() for n in names)
    bench.dump_records(str(tmp_path / "r"), res, rank=1, world=2)       # each rank writes its own files within its share
    names = sorted(os.listdir(tmp_path / "r"))
    assert names == sorted(f + "_rank1.npy" for f in FIELDS + ("index",))
    assert sum(os.path.getsize(tmp_path / "r" / n) for n in names) <= 32 << 10


def test_steps_and_dump_arguments_are_checked():
    assert _run("--impl", "reference", "--steps", "0").returncode == 2
    r = _run("--workload", "sweep", "--dump-outputs", "unused")
    assert r.returncode == 2 and "--dump-outputs" in r.stderr


@pytest.mark.gpu
def test_native_dump_equals_the_reference_arms(tmp_path):
    """The GPU's result records on the bench batch are the CPU spec oracle's, so the two arms dump the same arrays."""
    common = ("--scans", "256", "--steps", "2", "--warmup", "1", "--legs", "none", "--no-cpu-baseline")
    for impl in ("native", "reference"):
        r = _run("--impl", impl, *common, "--dump-outputs", str(tmp_path / impl))
        assert r.returncode == 0, r.stderr[-2000:]
        assert json.loads(r.stdout.strip().splitlines()[-1])["steps"] == 2
    for f in FIELDS:
        a, b = np.load(tmp_path / "native" / (f + ".npy")), np.load(tmp_path / "reference" / (f + ".npy"))
        assert len(a) == 256 and a.tobytes() == b.tobytes(), f
