"""bench.py helpers that run without a GPU: the nvidia-smi clock sampler keeps only the samples that
arrived inside the timed region (it is started before the warm-up because nvidia-smi needs ~0.1 s to
come up) and falls back to the whole run when the region is shorter than one sample period; the
--dump-outputs writer; argument checks."""

import importlib.util
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def load_bench():
    spec = importlib.util.spec_from_file_location("bench_module", os.path.join(ROOT, "bench.py"))
    mod = importlib.util.module_from_spec(spec)
    argv, sys.argv = sys.argv, ["bench.py"]
    try:
        spec.loader.exec_module(mod)
    finally:
        sys.argv = argv
    return mod


class _Proc:
    def terminate(self): pass
    def wait(self, timeout=None): pass
    def kill(self): pass


LINE = "0, {sm}, 1965, {p}, 0x0, Not Active, Not Active, Not Active, {cap}"


def test_clock_sampler_windows_samples():
    b = load_bench()
    s = b.ClockSampler(0)
    s.proc = _Proc()
    t = time.perf_counter()
    s.lines = [(t - 1.0, LINE.format(sm=1200, p=150.0, cap="Not Active")),        # warm-up sample
               (t + 0.1, LINE.format(sm=1950, p=400.0, cap="Active")),
               (t + 0.2, LINE.format(sm=1965, p=410.0, cap="Not Active"))]
    s.window = (t, t + 0.5)
    r = s.stop()
    assert r["samples"] == 2 and r["scope"] == "timed region"
    assert r["sm_mhz"] == 1957.5 and r["sm_max_mhz"] == 1965.0 and r["reasons"] == ["sw_power_cap"]
    s.window = (t + 5, t + 6)  # nothing inside: fall back to every sample and say so
    r = s.stop()
    assert r["samples"] == 3 and r["scope"] == "warm-up + timed region"


def test_clock_sampler_without_nvidia_smi():
    b = load_bench()
    s = b.ClockSampler(0)
    assert s.stop()["reasons"] == ["nvidia-smi unavailable"]


def test_dump_outputs_writes_every_array(tmp_path):
    import numpy as np
    b = load_bench()
    val = np.arange(10, dtype=np.float64)
    flags = (val > 4).astype(np.float32)
    b.dump_outputs(str(tmp_path), {"content_val": val, "above_threshold": flags})
    assert sorted(os.listdir(tmp_path)) == ["above_threshold.npy", "content_val.npy"]
    assert np.array_equal(np.load(tmp_path / "content_val.npy"), val)
    assert np.load(tmp_path / "above_threshold.npy").dtype == np.float32


def test_dump_outputs_samples_large_outputs_the_same_way(tmp_path, monkeypatch):
    import numpy as np
    b = load_bench()
    monkeypatch.setattr(b, "DUMP_BYTES", 4000)
    val = np.arange(1000, dtype=np.float64)
    comp = np.stack([val] * 4, axis=1)
    for sub in ("a", "b"):
        b.dump_outputs(str(tmp_path / sub), {"content_val": val, "components": comp}, "_rank1")
    idx = np.load(tmp_path / "a" / "frame_index_rank1.npy")
    assert np.array_equal(idx, np.load(tmp_path / "b" / "frame_index_rank1.npy"))
    assert sum(f.stat().st_size for f in (tmp_path / "a").iterdir()) < 4000 + 3 * 256
    assert np.array_equal(np.load(tmp_path / "a" / "content_val_rank1.npy"), idx)
    assert np.array_equal(np.load(tmp_path / "a" / "components_rank1.npy")[:, 3], idx)


def test_steps_must_be_positive(monkeypatch):
    import pytest
    b = load_bench()
    monkeypatch.setattr(sys, "argv", ["bench.py", "--steps", "3"])
    assert b.parse_args().steps == 3
    for bad in (["--steps", "0"], ["--dump-outputs", "x", "--sweep"], ["--dump-outputs", "x", "--impl", "reference"]):
        monkeypatch.setattr(sys, "argv", ["bench.py"] + bad)
        with pytest.raises(SystemExit):
            b.parse_args()
