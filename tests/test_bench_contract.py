"""bench.py contract checks that need no GPU: the reference arm (the oracle port timed on the
host cores) prints one well-formed JSON line, and the product arm refuses to run without CUDA."""
import json
import os
import subprocess
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(*argv, timeout=300):
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *argv], cwd=ROOT,
                          capture_output=True, text=True, timeout=timeout)


def test_reference_arm_line():
    r = _run("--impl", "reference", "--steps", "2", "--warmup", "1")
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference"
    assert d["metric"] == "constraint+Jacobian evals/sec" and d["unit"] == "evals/s"
    assert d["higher_is_better"] is True and d["n_gpus"] == 1 and d["steps"] == 2 and d["warmup"] == 1
    assert d["dtype"] == "f64" and d["vs_baseline"] is None
    assert "C4" in d["config"]["workload"]
    assert d["value"] > 0 and d["ms_per_step"] > 0
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("port", "reference") and cb["cores"] >= 1 and cb["sample"]
    assert cb["value"] == pytest.approx(d["value"])
    e = d["e2e"]
    assert e["value"] == pytest.approx(d["value"]) and e["unit"] == d["unit"]
    assert e["h2d_bytes_per_step"] == 0 and e["d2h_bytes_per_step"] == 0


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU behaviour")
def test_product_arm_needs_cuda():
    r = _run("--steps", "1", "--warmup", "1", "--no-cpu", "--no-sweep")
    assert r.returncode != 0
    assert not [ln for ln in r.stdout.splitlines() if ln.startswith("{")]     # no number without a GPU


def test_clock_sampler_reports_missing_nvml():
    sys.path.insert(0, ROOT)
    import bench
    s = bench.ClockSampler(0)
    s.open()
    s.start()
    out = s.stop()
    assert set(out) >= {"sm_mhz", "sm_max_mhz", "reasons", "samples"}
    if out["samples"] == 0:
        assert out["sm_mhz"] is None


def test_both_arms_share_one_config_dict():
    """The driver compares `config` of the two arms: per-arm details live outside it."""
    sys.path.insert(0, ROOT)
    import bench
    cfg = bench.workload_config()
    assert set(cfg) == {"workload", "sharding", "l2_policy"}
    r = _run("--impl", "reference", "--steps", "1", "--warmup", "0")
    d = json.loads([ln for ln in r.stdout.splitlines() if ln.startswith("{")][0])
    assert d["config"] == cfg


def test_dump_outputs_layout_and_budget(tmp_path, monkeypatch):
    """--dump-outputs: float64 arrays; the separation rows of the same seeded pair sample on every
    call, in pair order; whole leading evaluations of the batch within the size budget."""
    import numpy as np
    sys.path.insert(0, ROOT)
    import bench
    B, P, N, L = 3, 20000, 50, 7
    pm = torch.randn((B, P), dtype=torch.float64)
    spd = torch.randn((B, N, L), dtype=torch.float64)
    sep = torch.arange(P, dtype=torch.float64)[None, :, None] + torch.zeros((B, 1, L), dtype=torch.float64)
    sep[1] += 0.5
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), pm, sep, spd)
    out = {f: np.load(str(tmp_path / "a" / f)) for f in os.listdir(str(tmp_path / "a"))}
    assert set(out) == {"pair_min.npy", "max_speed.npy", "separation.npy"}
    assert all(a.dtype == np.float64 for a in out.values())
    assert sum(a.nbytes for a in out.values()) <= bench.DUMP_BYTES
    assert np.array_equal(out["pair_min.npy"], pm.numpy()) and np.array_equal(out["max_speed.npy"], spd.numpy())
    s = out["separation.npy"]
    assert s.shape == (B, bench.DUMP_PAIRS, L)
    pairs = s[0, :, 0]
    assert np.all(np.diff(pairs) > 0) and pairs[0] >= 0 and pairs[-1] < P
    assert np.array_equal(s[1], s[0] + 0.5) and np.array_equal(s[2], s[0])
    for f, a in out.items():
        assert np.array_equal(np.load(str(tmp_path / "b" / f)), a)
    monkeypatch.setattr(bench, "DUMP_BYTES", 2 * 8 * (P + N * L + bench.DUMP_PAIRS * L))
    bench.dump_outputs(str(tmp_path / "c"), pm, sep, spd)
    assert np.load(str(tmp_path / "c" / "separation.npy")).shape[0] == 2
    assert np.array_equal(np.load(str(tmp_path / "c" / "pair_min.npy")), pm[:2].numpy())


def test_bench_rejects_unsupported_arguments(tmp_path):
    for argv in (("--steps", "0"), ("--impl", "reference", "--dump-outputs", str(tmp_path / "d")),
                 ("--workload", "c5", "--dump-outputs", str(tmp_path / "d"))):
        r = _run(*argv, timeout=60)
        assert r.returncode != 0 and "usage" in r.stderr
    assert not os.path.exists(str(tmp_path / "d"))


def test_python_reference_leg_when_staged():
    """cpu_baseline_python times the unmodified reference from baseline/_ref (staged by
    __graft_entry__.build() where /root/reference exists); absent copy -> None."""
    sys.path.insert(0, ROOT)
    import bench
    args, x = bench.synthetic_swarm(64, 10)
    out = bench.cpu_baseline_python(args, x, 100, npairs=256)
    if not os.path.isfile(os.path.join(ROOT, "baseline", "_ref", "bezier.py")):
        assert out is None
        return
    assert out["kind"] == "reference" and out["cores"] == 1 and out["value"] > 0
    assert 1.0 < out["us_per_pair"] < 5000.0
