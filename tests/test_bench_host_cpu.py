"""Host-side pieces of bench.py that run without a GPU: the clock sampler's helper-process protocol (with a stand-in for
NVML), the workload table (every BASELINE.json config selectable, identical `config` object in both arms) and the
algorithmic-flop count the step-level roofline divides by."""
import json
import os
import sys
import time

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


@pytest.fixture()
def bench(monkeypatch):
    monkeypatch.setattr(sys, "argv", ["bench.py"])
    import bench as B
    yield B
    B.select_workload("cfg2")


def test_clock_sampler_helper_process_samples_only_between_begin_and_stop(bench, monkeypatch):
    monkeypatch.setenv("DVAE_FAKE_NVML", "1")
    c = bench.ClockSampler(0, period_s=0.002)
    assert c.child is not None and c.source == "nvml helper process"
    time.sleep(0.05)                     # before begin(): nothing may be recorded
    c.begin()
    time.sleep(0.05)
    c.sample_now()                       # a no-op now: the launch loop never calls NVML
    out = c.stop()
    assert 5 <= out["samples"] <= 40, out
    assert out["sm_mhz"] == out["sm_max_mhz"] == 1965.0 and out["reasons"] == [] and out["source"] == "nvml helper process"
    assert c.child.poll() is not None    # the helper has exited


def test_clock_sampler_reports_throttle_reasons(bench):
    c = bench.ClockSampler.__new__(bench.ClockSampler)
    c.samples, c.live, c._stop, c.h, c.child, c.source, c.max_mhz = [(1500.0, 0x4 | 0x40, 700.0), (1965.0, 0, 500.0)], False, False, object(), None, "test", 1965.0
    out = c.stop()
    assert set(out["reasons"]) == {"sw_power_cap", "hw_thermal_slowdown"} and out["sm_min_mhz"] == 1500.0 and out["power_w_max"] == 700.0


def test_clock_sampler_without_nvml_degrades_to_null_clocks(bench, monkeypatch):
    monkeypatch.delenv("DVAE_FAKE_NVML", raising=False)
    c = bench.ClockSampler(0)            # no GPU / driver in the CPU container: neither the helper nor the thread can sample
    c.begin()
    out = c.stop()
    if out["samples"] == 0:
        assert out["sm_mhz"] is None and out["reasons"] == []


@pytest.mark.parametrize("name", ["cfg1", "cfg2", "cfg3", "cfg4", "cfg5"])
def test_every_baseline_config_is_a_selectable_workload(bench, name):
    base = json.load(open(os.path.join(ROOT, "BASELINE.json")))
    assert len(base["configs"]) == 5
    bench.select_workload(name)
    cfg = bench.workload_config(1)
    assert cfg["workload"].startswith(name) and cfg["global_batch"] == bench.BATCH and cfg["seq_len"] == bench.SEQ_T
    assert bench.workload_config(8)["global_batch"] == 8 * bench.BATCH and bench.workload_config(8)["parallelism"] == "dp8"
    assert "model" not in cfg            # the tier's contract: config names the workload, no model keys


def test_dump_outputs_stays_under_64_mb_and_samples_the_same_elements_every_time(bench, tmp_path):
    rng = np.random.default_rng(0)
    arrays = {"losses": torch.arange(32, dtype=torch.float32), "lengths": torch.arange(7, dtype=torch.int64) * 3,
              "param.w": torch.from_numpy(rng.standard_normal((6000, 5000)).astype(np.float32)),       # 120 MB alone
              "param.b": np.linspace(-1, 1, 999)}
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), arrays)
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == ["lengths.npy", "losses.npy", "param.b.npy", "param.w.npy"]
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in files) <= 64 * 10 ** 6
    got = {f[:-4]: np.load(tmp_path / "a" / f) for f in files}
    assert got["losses"].dtype == np.float32 and np.array_equal(got["losses"], np.arange(32))      # small arrays whole
    assert got["lengths"].dtype == np.float64 and np.array_equal(got["lengths"], np.arange(7) * 3)
    assert got["param.b"].dtype == np.float32 and got["param.b"].shape == (999,)
    w = got["param.w"]
    assert w.dtype == np.float32 and w.ndim == 1 and 10 ** 7 < w.size < arrays["param.w"].numel()
    assert np.isin(w, arrays["param.w"].numpy()).all()                                             # elements, not noise
    assert np.array_equal(w, np.load(tmp_path / "b" / "param.w.npy"))                              # the same sample


def test_algorithmic_flops_match_the_survey_accounting(bench):
    """SURVEY.md 8a / DESIGN.md 6: 102.6 GFLOP algorithmic per cfg-2 train step, forward + backward = 3 x forward, the
    vocabulary projection the largest single class."""
    bench.select_workload("cfg2")
    f = bench.algorithmic_flops(bench.BATCH, bench.SEQ_T)
    n = (bench.SEQ_T - 1) * bench.BATCH
    assert f["vocab"] == 3.0 * 2 * n * bench.CFG2["hidden_dim"] * bench.VOCAB
    assert abs(f["total"] - 102.64e9) < 0.05e9
    assert f["total"] == f["vocab"] + f["lstm_input_projections"] + f["recurrence"] + f["heads"]
    assert f["vocab"] > max(f["lstm_input_projections"], f["recurrence"], f["heads"])
    bench.select_workload("cfg4")
    f4 = bench.algorithmic_flops(bench.BATCH, bench.SEQ_T)
    assert f4["vocab"] == 3.0 * 2 * (bench.SEQ_T - 1) * bench.BATCH * 1024 * 50000
