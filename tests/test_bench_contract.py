"""bench.py's JSON-line contract, checked on CPU through the reference arm (the CPU restatement timed on host cores) and
the failure behaviour of the native arm without a GPU (no silent fallback)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(*args):
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True, timeout=600, cwd=ROOT)


def test_reference_arm_prints_one_json_line_with_the_contract_keys():
    r = _run("--impl", "reference", "--steps", "1", "--warmup", "1", "--ref-n", "16")
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.strip().splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["higher_is_better"] is True and d["unit"] == "particle-steps/s"
    for key in ("metric", "value", "n_gpus", "steps", "warmup", "ms_per_step", "scaling", "vs_baseline", "dtype", "data", "config",
                "cpu_baseline", "e2e"):
        assert key in d, key
    assert d["value"] > 0 and d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["value"] == d["value"] and d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert d["vs_baseline"] is None          # BASELINE.md publishes no number for this metric
    assert "workload" in d["config"]


def test_native_arm_fails_loudly_without_a_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("CUDA present")
    r = _run("--steps", "1", "--warmup", "0", "--no-cpu", "--n", "8")
    assert r.returncode != 0
    assert not [ln for ln in r.stdout.splitlines() if ln.startswith("{") and '"value"' in ln]


class _FakeWorld:
    """num_particles / read_fluid of LiquidWorld over host arrays: particle i of fluid k sits at (k, i, -i)."""

    def __init__(self, counts):
        self.data = [np.stack([np.full(n, k), np.arange(n), -np.arange(n)], axis=1).astype(np.float32) for k, n in enumerate(counts)]

    def num_particles(self, f):
        return len(self.data[f])

    def read_fluid(self, f):
        return self.data[f].copy(), 2 * self.data[f]


@pytest.mark.parametrize("counts", [(1000,), (3_000_000, 1_500_000)], ids=["whole", "sampled"])
def test_dump_outputs_is_a_fixed_f32_sample_within_64_mb(tmp_path, counts):
    sys.path.insert(0, ROOT)
    import bench
    for d in ("a", "b"):
        bench.dump_outputs(_FakeWorld(counts), list(range(len(counts))), str(tmp_path / d))
    names = sorted(os.listdir(tmp_path / "a"))
    assert names == sorted("fluid%d_%s.npy" % (k, q) for k in range(len(counts)) for q in ("positions", "velocities"))
    assert sum(os.path.getsize(tmp_path / "a" / n) for n in names) <= 64 << 20
    for k, n in enumerate(counts):
        p = np.load(tmp_path / "a" / ("fluid%d_positions.npy" % k))
        v = np.load(tmp_path / "a" / ("fluid%d_velocities.npy" % k))
        assert p.dtype == v.dtype == np.float32 and p.shape == v.shape and p.shape[1] == 3
        assert (p[:, 0] == k).all() and np.array_equal(v, 2 * p)                 # rows stay whole, velocities match positions
        idx = p[:, 1].astype(np.int64)
        assert (np.diff(idx) > 0).all() and idx[-1] < n                          # distinct particles in original order
        assert len(idx) == (n if sum(counts) <= bench.DUMP_MAX_PARTICLES else bench.DUMP_MAX_PARTICLES * n // sum(counts))
        assert np.array_equal(p, np.load(tmp_path / "b" / ("fluid%d_positions.npy" % k)))   # same sample on every run


def test_dump_outputs_is_refused_where_it_cannot_apply():
    r = _run("--impl", "reference", "--steps", "1", "--dump-outputs", "unused")
    assert r.returncode == 2 and "--dump-outputs" in r.stderr
    r = _run("--steps", "0")
    assert r.returncode == 2 and "--steps" in r.stderr


class _Args:
    grid_order = "auto"
    backend = 0
    probe = False
    parity_n = 64
    n = 0
    no_settled = False


def _probe_line(ms, parity=True, settled=25.0, settled_error=None):
    st = {"error": settled_error} if settled_error else {"ms_per_step": settled}
    return json.dumps({"ms_per_step": ms, "parity": {"ok": parity}, "roofline": {"ms_per_launch_pair": 1.0},
                       "phases": {"neighbors_ms": 1.6, "grid_ms": 0.4}, "settled": st})


@pytest.mark.parametrize("h,rows,expect", [
    ((8.5, True, 25.0, None), (6.0, True, 20.0, None), "rows"),      # faster, parity green, settled not slower
    ((8.5, True, 25.0, None), (8.4, True, 25.0, None), "h"),         # within noise (< 3 %)
    ((8.5, True, 25.0, None), (6.0, False, 20.0, None), "h"),        # parity failed in the new order
    ((8.5, True, 25.0, None), (6.0, True, 27.0, None), "h"),         # slower in the settled block
    ((8.5, True, 25.0, None), (6.0, True, None, "boom"), "h"),       # settled block raised
])
def test_grid_order_selection_is_parity_gated(monkeypatch, h, rows, expect):
    """bench.py keeps the 'rows' particle order only when its probe passed parity AND was faster; everything else => default."""
    sys.path.insert(0, ROOT)
    import bench

    class R:
        def __init__(self, out, rc=0):
            self.stdout, self.stderr, self.returncode = out, "", rc

    def fake_run(cmd, **kw):
        name = cmd[cmd.index("--grid-order") + 1]
        ms, par, st, err = h if name == "h" else rows
        assert "--probe" in cmd and "--no-cpu" in cmd
        return R(_probe_line(ms, par, st, err))

    monkeypatch.setattr(subprocess, "run", fake_run)
    info = bench.pick_grid_order(_Args(), "c3", 1)
    assert info["chosen"] == expect and set(info["probes"]) == {"h", "rows"}


def test_grid_order_falls_back_when_a_probe_dies(monkeypatch):
    sys.path.insert(0, ROOT)
    import bench

    def fake_run(cmd, **kw):
        if cmd[cmd.index("--grid-order") + 1] == "rows":
            raise subprocess.TimeoutExpired(cmd, 150)
        return type("R", (), {"stdout": _probe_line(8.5), "stderr": "", "returncode": 0})()

    monkeypatch.setattr(subprocess, "run", fake_run)
    info = bench.pick_grid_order(_Args(), "c3", 1)
    assert info["chosen"] == "h" and "error" in info["probes"]["rows"]
    # never probed: multi-GPU, other configs, explicit choices
    assert bench.pick_grid_order(_Args(), "c4", 8)["chosen"] == "h"
    assert bench.pick_grid_order(_Args(), "c5", 1)["chosen"] == "h"
    a = _Args()
    a.grid_order = "rows"
    assert bench.pick_grid_order(a, "c3", 1)["chosen"] == "rows"
