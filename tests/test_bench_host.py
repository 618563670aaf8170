"""Host-side logic of bench.py that needs no GPU: the clock sampler keeps only the nvidia-smi lines that arrived while
the GPU was under the workload's load, and summarises them (median SM clock, max clock, active throttle reasons);
--dump-outputs writes every instance's outputs, or a fixed sample of them, as float64 within its byte budget."""
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench  # noqa: E402


class _Proc:
    def terminate(self):
        pass

    def wait(self, timeout=None):
        return 0

    def kill(self):
        pass


def _sampler(rows):
    s = bench.ClockSampler(0)
    s.proc = _Proc()
    s.rows = rows
    return s


def test_clock_sampler_window_and_reasons():
    line = "0, {sm}, 1965, 700.0, 0x0, Not Active, Not Active, Not Active, {cap}"
    rows = [(0.5, line.format(sm=210, cap="Not Active")),          # idle clock before the timed region: ignored
            (1.1, line.format(sm=1965, cap="Not Active")),
            (1.2, line.format(sm=1950, cap="Active")),
            (1.3, line.format(sm=1965, cap="Not Active")),
            (2.5, line.format(sm=300, cap="Not Active")),          # after the load: ignored
            (1.25, "garbage line")]
    s = _sampler(rows)
    assert s.count(1.0, 2.0) == 4                                  # three samples + the malformed line
    out = s.stop(1.0, 2.0)
    assert out["samples"] == 3 and out["sm_mhz"] == 1965.0 and out["sm_max_mhz"] == 1965.0
    assert out["reasons"] == ["sw_power_cap"]
    assert _sampler(rows).stop()["samples"] == 5                   # no window: everything that parses


def test_clock_sampler_without_nvidia_smi():
    s = bench.ClockSampler(0)
    assert s.stop(0.0, 1.0)["reasons"] == ["nvidia-smi unavailable"]


def test_workload_registry_matches_the_documented_names():
    assert sorted(bench.WORKLOADS) == sorted(["ukfom", "usckf", "msckf", "fusion", "ekf", "msckf_ekf", "safefusion", "deadreckon"])
    for name, cls in bench.WORKLOADS.items():
        assert cls.name == name and cls.unit and cls.metric
        assert callable(getattr(cls, "outputs", None))


class _Outputs:
    """Stands in for a workload after its timed steps: host arrays and (CPU) torch tensors, one row per instance."""

    def __init__(self, n):
        import torch
        rng = np.random.default_rng(3)
        self.n = n
        self.arrays = {"mu": rng.normal(size=(n, 5)), "P": torch.from_numpy(rng.normal(size=(n, 4, 4))),
                       "status": np.arange(n, dtype=np.int32) % 3}

    def units_per_step(self):
        return self.n

    def outputs(self, k):
        return dict(self.arrays)


def _load(d):
    return {f[:-4]: np.load(os.path.join(d, f)) for f in sorted(os.listdir(d))}


def test_dump_outputs_writes_every_instance_when_they_fit(tmp_path):
    wl = _Outputs(100)
    bench.dump_outputs(wl, 7, str(tmp_path))
    got = _load(str(tmp_path))
    assert sorted(got) == ["P", "instance", "mu", "status"]
    assert all(a.dtype == np.float64 for a in got.values())
    np.testing.assert_array_equal(got["instance"], np.arange(100))
    np.testing.assert_array_equal(got["mu"], wl.arrays["mu"])
    np.testing.assert_array_equal(got["P"], wl.arrays["P"].numpy())
    np.testing.assert_array_equal(got["status"], wl.arrays["status"])


def test_dump_outputs_samples_a_fixed_subset_within_the_budget(tmp_path, monkeypatch):
    wl = _Outputs(5000)
    per = 8 * (1 + 5 + 16 + 1)
    monkeypatch.setattr(bench, "DUMP_BYTES", 300 * per + 7)
    a, b = tmp_path / "a", tmp_path / "b"
    bench.dump_outputs(wl, 0, str(a))
    bench.dump_outputs(wl, 0, str(b))
    ga, gb = _load(str(a)), _load(str(b))
    idx = ga["instance"].astype(np.int64)
    assert len(idx) == 300 and np.all(np.diff(idx) > 0) and idx[-1] < 5000 and idx[-1] > 2500
    assert sum(v.nbytes for v in ga.values()) <= bench.DUMP_BYTES
    np.testing.assert_array_equal(ga["mu"], wl.arrays["mu"][idx])
    np.testing.assert_array_equal(ga["P"], wl.arrays["P"].numpy()[idx])
    np.testing.assert_array_equal(ga["status"], wl.arrays["status"][idx])
    for k in ga:
        np.testing.assert_array_equal(ga[k], gb[k])
