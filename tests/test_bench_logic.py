"""CPU tests of the measurement harness helpers (bench.py): no GPU, no timing claims."""
import importlib.util
import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def bench():
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    mod = importlib.util.module_from_spec(spec)
    sys.path.insert(0, ROOT)
    spec.loader.exec_module(mod)
    return mod


def test_usable_cores_is_bounded_by_affinity(bench):
    n = bench.usable_cores()
    assert 1 <= n <= (os.cpu_count() or 1)
    assert n <= len(os.sched_getaffinity(0))


def test_cpu_samples_are_fractions_of_the_baseline_workload(bench):
    full = bench.LAT_H * bench.LAT_W
    for frames, h, w, eq in bench.CPU_SAMPLES:
        assert abs(frames * h * w / full - eq) < 1e-9      # frame-equivalents = pixels processed / pixels of one frame
        assert h % 8 == 0 and w % 8 == 0                   # three stride-2 levels must divide evenly
    eqs = [s[3] for s in bench.CPU_SAMPLES]
    assert eqs == sorted(eqs, reverse=True)                # largest first: pick_cpu_sample takes the first that fits


def test_pick_cpu_sample_respects_the_time_budget(bench, monkeypatch):
    calls = []

    def fake_step(model, frames, seed=1234, h=bench.LAT_H, w=bench.LAT_W):
        calls.append((frames, h, w))
        return 2.0                                          # the quarter-frame probe "takes" 2 s

    monkeypatch.setattr(bench, "cpu_step", fake_step)
    s, tq = bench.pick_cpu_sample(None, n_steps=4, budget_s=150.0)     # 2 frames would need 2*8*4 = 64 s -> fits
    assert s == bench.CPU_SAMPLES[0] and tq == 2.0
    s, _ = bench.pick_cpu_sample(None, n_steps=8, budget_s=100.0)      # 2 frames: 128 s no; 1 frame: 64 s yes
    assert s == bench.CPU_SAMPLES[1]
    s, _ = bench.pick_cpu_sample(None, n_steps=8, budget_s=10.0)       # nothing fits: smallest sample
    assert s == bench.CPU_SAMPLES[-1]
    assert all(c == bench.CPU_SAMPLES[-1][:3] for c in calls)          # only the probe shape was ever executed


def test_clock_sampler_brackets_the_timed_region(bench, tmp_path, monkeypatch):
    rows = ["1965, 1965, 700.0, Not Active, Not Active, Not Active, Not Active",
            "1950, 1965, 900.0, Not Active, Not Active, Not Active, Active",
            "1200, 1965, 300.0, Active, Not Active, Not Active, Not Active"]

    class FakeProc:
        def terminate(self): pass
        def wait(self, timeout=None): return 0
        def kill(self): pass

    def make():
        cs = bench.ClockSampler.__new__(bench.ClockSampler)
        f = tmp_path / f"s{len(list(tmp_path.iterdir()))}.csv"
        f.write_text("\n".join(rows) + "\n")
        cs.f = open(f, "r+")
        cs.p = FakeProc()
        return cs

    cs = make()
    assert cs.count() == 3
    out = cs.stop(0, 2)                                    # the third sample (idle, hw slowdown) is outside the region
    assert out["sm_mhz"] == 1957.5 and out["reasons"] == ["sw_power_cap"] and out["samples"] == 2
    out = make().stop(1, 1)                                # region shorter than a sampling period: both neighbours
    assert out["samples"] == 2 and out["sm_mhz"] == 1957.5
    out = make().stop()                                    # no bracket: everything
    assert out["samples"] == 3 and "hw_slowdown" in out["reasons"]


def test_dump_outputs_writes_a_fixed_sample(bench, tmp_path, monkeypatch):
    import numpy as np
    import torch
    monkeypatch.setattr(bench, "DUMP_SAMPLE", 100)
    params = [torch.nn.Parameter(torch.arange(60, dtype=torch.float32).reshape(6, 10)), torch.nn.Parameter(-torch.arange(90.0))]
    for p in params:
        p.grad = 2 * p.detach()
    pred, loss = torch.randn(1, 2, 4, 8, 8, dtype=torch.bfloat16), torch.tensor(0.25)
    runs = []
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), pred, loss, params)
        runs.append({f.stem: np.load(f) for f in (tmp_path / d).iterdir()})
    a, b = runs
    assert sorted(a) == ["grads_sample", "loss", "pred", "sample_index", "weights_sample"]
    for k in a:
        assert a[k].dtype in (np.float32, np.float64) and np.array_equal(a[k], b[k]), k
    idx = a["sample_index"].astype(np.int64)
    flat = np.concatenate([p.detach().numpy().reshape(-1) for p in params])
    assert 0 < len(idx) <= 100 and np.all(np.diff(idx) > 0) and idx[-1] < flat.size
    assert np.array_equal(a["weights_sample"], flat[idx]) and np.array_equal(a["grads_sample"], 2 * flat[idx])
    assert a["pred"].shape == (1, 2, 4, 8, 8) and np.array_equal(a["pred"], pred.float().numpy()) and a["loss"] == 0.25


def test_splitk_workspace_is_cached_per_shape():
    from svd_xtend_b200 import raw
    import torch
    a = raw._splitk_workspace(8, 16, torch.device("cpu"))
    b = raw._splitk_workspace(8, 16, torch.device("cpu"))
    c = raw._splitk_workspace(8, 32, torch.device("cpu"))
    assert a is b and c is not a and a.dtype == torch.float32 and float(a.abs().sum()) == 0.0
