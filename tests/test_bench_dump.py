"""bench.py --dump-outputs: what it writes stays within its budget, is finite, keeps the float precision of each output
(its NaN entries marked in <name>_nonfinite.npy), writes flags and states as float32, samples the same rows of every
array and is identical from run to run.  CPU tensors stand in for the device outputs of a workload."""
import importlib.util
import os
import sys

import numpy as np
import torch

from parity import REPO


def _bench():
    keep = sys.dont_write_bytecode          # bench.py turns the bytecode cache off for its own process
    spec = importlib.util.spec_from_file_location("bench_under_test", os.path.join(REPO, "bench.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    sys.dont_write_bytecode = keep
    return mod


class _Workload:
    """Row i of every output is a function of i, so a dumped row can be traced back to the row it came from.  Like the
    solver's outputs for an unreachable pose, the float rows with i % 5 == 3 are NaN."""

    def __init__(self, n):
        i = torch.arange(n, dtype=torch.float64)
        unreachable = (i % 5 == 3)[:, None]
        joints = torch.stack([i + k / 8 for k in range(7)], dim=1).masked_fill(unreachable, float("nan"))
        elbow = (i % 1000).float()[:, None].repeat(1, 3).masked_fill(unreachable, float("nan"))
        self.out = {"joints": joints, "elbow32": elbow, "state": (i % 9).to(torch.uint8), "reachable": i % 2 == 0}

    def outputs(self):
        return self.out


def _load(d):
    return {f[:-4]: np.load(os.path.join(d, f)) for f in sorted(os.listdir(d))}


def _restore(a, name):
    """The array the caller received: the dumped values with the marked entries put back to NaN."""
    return np.where(a[name + "_nonfinite"] == 1, np.nan, a[name]).astype(a[name].dtype)


def test_dump_outputs_samples_rows_within_budget(tmp_path):
    bench = _bench()
    n = 1_000_000                            # 108 MB with the masks: above the budget, so a sample is written
    wl = _Workload(n)
    rec = bench.dump_outputs(wl, str(tmp_path / "a"))
    bench.dump_outputs(wl, str(tmp_path / "b"))
    a, b = _load(tmp_path / "a"), _load(tmp_path / "b")
    assert sorted(a) == ["elbow32", "elbow32_nonfinite", "joints", "joints_nonfinite", "reachable", "state"]
    assert sum(os.path.getsize(tmp_path / "a" / f"{name}.npy") for name in a) <= 64_000_000
    assert {k: v.dtype for k, v in a.items()} == {"joints": np.float64, "elbow32": np.float32, "state": np.float32, "reachable": np.float32,
                                                  "joints_nonfinite": np.float32, "elbow32_nonfinite": np.float32}
    for name in a:
        assert np.isfinite(a[name]).all(), name
        assert np.array_equal(a[name], b[name]), name
    k = len(a["state"])
    joints, elbow = _restore(a, "joints"), _restore(a, "elbow32")
    ok = ~np.isnan(joints[:, 0])
    idx = joints[ok, 0]                      # the source row of every reachable row, from its first joint
    assert 0 < k < n and np.all(np.diff(idx) > 0) and np.array_equal(idx, np.round(idx))
    assert rec["rows_written_of_total"]["joints"] == [k, n] and rec["sample_seed"] is not None
    assert np.all(idx % 5 != 3) and 0.15 < (~ok).mean() < 0.25
    np.testing.assert_array_equal(joints[ok], idx[:, None] + np.arange(7) / 8)
    np.testing.assert_array_equal(np.isnan(elbow), np.repeat(~ok[:, None], 3, axis=1))
    np.testing.assert_array_equal(elbow[ok, 0], idx % 1000)
    np.testing.assert_array_equal(a["state"][ok], idx % 9)
    np.testing.assert_array_equal(a["reachable"][ok], (idx % 2 == 0).astype(np.float32))


def test_dump_outputs_small_outputs_whole(tmp_path):
    bench = _bench()
    wl = _Workload(1000)
    rec = bench.dump_outputs(wl, str(tmp_path))
    a = _load(tmp_path)
    assert rec["sample_seed"] is None
    np.testing.assert_array_equal(_restore(a, "joints"), wl.out["joints"].numpy())
    np.testing.assert_array_equal(_restore(a, "elbow32"), wl.out["elbow32"].numpy())
    np.testing.assert_array_equal(a["state"], np.arange(1000) % 9)


def test_continuous_outputs_decode_the_trajectory_state_record():
    """Continuous.outputs reads previous_theta / previous_sol / emergency_stop / emergency_bits out of the raw (T, 80)
    bytes of _abi.TRAJ_STATE_DTYPE that the continuous entry updates in place."""
    from reachy2_symbolic_ik_b200 import _abi

    bench = _bench()
    T = 5
    st = np.zeros(T, dtype=_abi.TRAJ_STATE_DTYPE)
    st["previous_theta"] = np.arange(T) * 0.5 - 1.0
    st["previous_sol"] = np.arange(T * 7).reshape(T, 7) / 10.0
    st["has_previous_sol"], st["init"] = 1, 0
    st["emergency_stop"] = np.arange(T) % 2
    st["emergency_bits"] = np.arange(T) * 3 + 1
    raw = torch.from_numpy(st.view(np.uint8).reshape(T, -1).copy())
    wl = bench.Continuous.__new__(bench.Continuous)
    joints, reach, state = torch.zeros(T, 2, 7, dtype=torch.float64), torch.ones(T, 2, dtype=torch.bool), torch.zeros(T, 2, dtype=torch.uint8)
    wl.out = (joints, reach, state, raw)
    o = wl.outputs()
    assert o["joints"] is joints and o["reachable"] is reach and o["state"] is state
    np.testing.assert_array_equal(o["final_previous_theta"].numpy(), st["previous_theta"])
    np.testing.assert_array_equal(o["final_previous_sol"].numpy(), st["previous_sol"])
    np.testing.assert_array_equal(o["final_emergency_stop"].numpy(), st["emergency_stop"])
    np.testing.assert_array_equal(o["final_emergency_bits"].numpy(), st["emergency_bits"])


def test_symik_and_discrete_outputs_name_what_the_caller_receives():
    bench = _bench()
    wl = bench.Symik.__new__(bench.Symik)
    wl.outs = {arm: {k: torch.zeros(3) for k in ("reach", "state", "interval", "joints", "elbow")} for arm in bench.ARMS}
    assert sorted(wl.outputs()) == sorted(f"{arm}_{f}" for arm in bench.ARMS
                                          for f in ("reachable", "state", "theta_interval", "joints", "elbow"))
    d = bench.Discrete.__new__(bench.Discrete)
    d.out = tuple(torch.full((3,), float(i)) for i in range(4))
    assert {k: float(v[0]) for k, v in d.outputs().items()} == {"joints": 0.0, "reachable": 1.0, "state": 2.0, "emergency_bits": 3.0}
