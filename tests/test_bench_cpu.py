"""Host-side pieces of bench.py that can be checked without a GPU: the clock sampler's parsing / time-window filter and
the --dump-outputs writer."""
import datetime
import importlib.util
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench():
    argv = sys.argv
    sys.argv = ["bench.py"]
    try:
        spec = importlib.util.spec_from_file_location("bench_under_test", os.path.join(ROOT, "bench.py"))
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
    finally:
        sys.argv = argv
    return mod


class _Proc:
    def terminate(self):
        pass


class _Thread:
    def join(self, timeout=None):
        pass


def _row(now, dt, mhz, power_cap="Not Active"):
    ts = datetime.datetime.fromtimestamp(now + dt).strftime("%Y/%m/%d %H:%M:%S.%f")[:-3]
    return [ts, str(mhz), "1965", "500.0", "Not Active", "Not Active", "Not Active", power_cap]


def test_clock_sampler_filters_to_the_timed_region():
    b = _bench()
    now = time.time()
    s = b.ClockSampler(0)
    s.proc, s.thread = _Proc(), _Thread()
    s.rows = [_row(now, -1.0, 1000), _row(now, 0.01, 1965), _row(now, 0.05, 1960, "Active"), _row(now, 0.3, 900)]
    out = s.stop(now, now + 0.1)
    assert out["samples"] == 2 and out["in_timed_region"] and out["sm_mhz"] == 1962.5
    assert out["reasons"] == ["sw_power_cap"] and out["sm_max_mhz"] == 1965.0


def test_clock_sampler_survives_garbage():
    b = _bench()
    now = time.time()
    s = b.ClockSampler(0)
    s.proc, s.thread = _Proc(), _Thread()
    s.rows = [["garbage"], ["x", "y"]]
    assert s.stop(now, now + 0.1) is None
    s.proc = _Proc()
    s.rows = [["not a timestamp", "1950", "1965", "1", "Not Active", "Not Active", "Not Active", "Not Active"]]
    out = s.stop(now, now + 0.1)
    assert out["samples"] == 1 and out["in_timed_region"] is False


def test_write_outputs_keeps_small_arrays_whole(tmp_path):
    b = _bench()
    arrays = dict(losses=np.arange(4, dtype=np.float32), vs=np.ones((3, 2), np.float64), act=np.arange(6).reshape(2, 3))
    b.write_outputs(arrays, str(tmp_path / "out"))
    got = {f[:-4]: np.load(str(tmp_path / "out" / f)) for f in os.listdir(str(tmp_path / "out"))}
    assert sorted(got) == ["act", "losses", "vs"]
    assert got["vs"].dtype == np.float64 and got["losses"].dtype == np.float32 and got["act"].dtype == np.float32
    for k, a in arrays.items():
        np.testing.assert_array_equal(got[k], a)


def test_write_outputs_samples_to_the_limit_at_fixed_positions(tmp_path):
    b = _bench()
    rs = np.random.RandomState(1)
    arrays = dict(params=rs.randn(300000).astype(np.float32), grads=rs.randn(50, 40, 30).astype(np.float32),
                  losses=np.arange(4, dtype=np.float32))
    limit = 3 * 4096 + 3 * 100000
    for d in ("a", "b"):
        b.write_outputs(arrays, str(tmp_path / d), limit=limit)
    files = sorted(os.listdir(str(tmp_path / "a")))
    assert sum(os.path.getsize(str(tmp_path / "a" / f)) for f in files) <= limit
    for f in files:
        np.testing.assert_array_equal(np.load(str(tmp_path / "a" / f)), np.load(str(tmp_path / "b" / f)))
    np.testing.assert_array_equal(np.load(str(tmp_path / "a" / "losses.npy")), arrays["losses"])
    p = np.load(str(tmp_path / "a" / "params.npy"))
    assert p.size == 100000 // 4 and np.isin(p, arrays["params"]).all()
