"""Continuous mode on the GPU (r2ik_ctl_continuous_phased_f64 and r2ik_ctl_continuous_f64 through
ControlIK.symbolic_inverse_kinematics_batch) on the trajectory families of continuous_edge_inputs.py: against the CPU oracle,
phased against serial kernel, and against the host build of the same source (test_continuous_edges_host.py).  The device
runs arithmetic the host build never runs (MUFU seeds, sincos_any, FMA contraction in cont_wind_code, rint on the winding
quotient) and the block / tile structure of the phased kernels, which the host build walks one trajectory at a time."""
import numpy as np
import pytest

import continuous_edge_inputs as CE
from test_hostsim_parity import ARMS, cfg_for, ctl_params, hs, hs_continuous, urdf_params  # noqa: F401 (hs: fixture)

pytestmark = pytest.mark.gpu
FAMILIES = [*CE.live_families("r_arm", 1, 2), "events"]


@pytest.fixture(scope="module")
def ctl():
    from reachy2_symbolic_ik_b200 import ControlIK

    return ControlIK(urdf_path="../config_files/reachy2.urdf")


def _gpu(ctl, oracle, arm):
    cj, cp = np.array(oracle.DEFAULT_PREV_JOINTS[arm]), oracle.DEFAULT_CURRENT_POSE[arm]
    return lambda M, states=None, **kw: ctl.symbolic_inverse_kinematics_batch(  # noqa: E731
        arm, M, "continuous", current_joints=cj, current_pose=cp, states=states, **kw)


@pytest.mark.parametrize("arm", ARMS)
@pytest.mark.parametrize("name", FAMILIES)
def test_family_vs_oracle(ctl, hs, oracle, arm, name):
    """At every shape: phased and serial kernels against the oracle; phased against serial (1e-12, integer state
    identical), also with every 1st / 7th / 97th waypoint sent down the serial get_joints route; flags, states and the
    controller's integer state identical to the host build's."""
    M, want, ill = CE.reference(oracle, arm, name)
    ocfg, opar = CE.oracle_config(oracle, arm)
    run = _gpu(ctl, oracle, arm)
    cfg, par = cfg_for(arm, urdf_params(), -1.01), ctl_params(oracle, arm)
    worst = 0.0
    for T, W in CE.SHAPES:
        X = np.ascontiguousarray(M[:T, :W])
        w = oracle.ctl_continuous_batch(ocfg, opar, X)
        phased, serial = run(X, phased=True), run(X, phased=False)
        for form, got in (("phased", phased), ("serial", serial)):
            worst = max(worst, CE.compare_with_oracle(f"gpu {name} {arm} {T}x{W} {form}", got, w, ill[:T, :W]))
        CE.assert_same_trajectories(phased, serial, f"gpu {name} {arm} {T}x{W} phased vs serial")
        for m in (1, 7, 97):
            CE.assert_same_trajectories(run(X, _test_force_serial_mod=m), serial, f"gpu {name} {arm} {T}x{W} force serial {m}")
        host = hs_continuous(hs, oracle, cfg, par, arm, X, phased=True)
        CE.assert_same_trajectories(phased, host, f"gpu vs host {name} {arm} {T}x{W}", atol=np.inf)
    cuts = [c for c in CE.SPLITS if c < M.shape[1]]
    for phased in (False, True):
        one = run(M, phased=phased)
        split = CE.split_run(lambda m, st: run(m, st, phased=phased), M, cuts)
        CE.assert_same_trajectories(split, one, f"gpu {name} {arm} split phased={phased}", atol=1e-12 if phased else 0)
    latched = want[3]["emergency_stop"].astype(bool)
    print(f"[gpu continuous edges {name} {arm}] {M.shape[0]} x {M.shape[1]} waypoints: latched {int(latched.sum())}/{len(M)} "
          f"trajectories, ill-conditioned {ill.mean():.4f}, max|err| well-conditioned {worst:.2e}")
    if name != "events":
        assert latched.mean() <= CE.LIVE_MAX_LATCHED.get(name, 0.0), f"{name}: {latched.mean():.3f} of the trajectories latched"
    assert ill.mean() <= CE.MAX_ILL.get(name, CE.MAX_ILL_DEFAULT)


@pytest.mark.parametrize("arm", ARMS)
def test_events_unfreeze(ctl, oracle, arm):
    """Each trajectory of the event family resumed with "unfreeze" right after its event, both kernels, against the
    oracle's segments."""
    M, _, _ = CE.reference(oracle, arm, "events")
    at = CE.event_families(arm)[1]
    run = _gpu(ctl, oracle, arm)
    for t, want, ill in CE.unfreeze_references(oracle, arm):
        for phased in (False, True):
            got = CE.unfreeze_run(lambda m, st: run(m, st, phased=phased), oracle, M[t], at[t])
            CE.compare_with_oracle(f"gpu events {arm} traj {t} ({CE.event_kind(t)}) unfreeze phased={phased}", got, want, ill)


@pytest.mark.parametrize("arm", ARMS)
def test_host_pipeline_chunks(ctl, oracle, arm):
    """symbolic_inverse_kinematics_batch_host cuts the waypoint axis into chunks resumed from R2ikTrajState: for chunks of
    1, 7, 127, 128 and 129 waypoints it equals the device-resident call (flags, states identical; joints 1e-12), on a live
    family and on the event family."""
    import torch

    run = _gpu(ctl, oracle, arm)
    for name in ("slow_far", "events"):
        M = np.ascontiguousarray(CE.reference(oracle, arm, name)[0][:65])
        want = run(M)
        for chunk in (1, 7, 127, 128, 129):
            got = ctl.symbolic_inverse_kinematics_batch_host(arm, torch.from_numpy(M).pin_memory(), "continuous", chunk=chunk,
                                                             current_joints=np.array(oracle.DEFAULT_PREV_JOINTS[arm]),
                                                             current_pose=oracle.DEFAULT_CURRENT_POSE[arm])
            got = (got[0].numpy(), got[1].numpy().astype(bool), got[2].numpy(), got[3].numpy().reshape(-1).view(want[3].dtype))
            CE.assert_same_trajectories(got, want, f"host pipeline {name} {arm} chunk={chunk}")


@pytest.mark.parametrize("arm", ARMS)
def test_live_families_large(ctl, arm):
    """4 096 x 1 000 waypoints of the live families (the grid arithmetic blockIdx.x / nblk and (size_t) t * W at a
    realistic size): phased equals serial, and no trajectory of a family that must stay live latches beyond its cap."""
    for name in CE.live_families(arm, 1, 2):
        M = CE.live_families(arm, 4096, 1000, only=(name,))[name]
        a = ctl.symbolic_inverse_kinematics_batch(arm, M, "continuous", phased=True)
        b = ctl.symbolic_inverse_kinematics_batch(arm, M, "continuous", phased=False)
        CE.assert_same_trajectories(a, b, f"gpu large {name} {arm}")
        latched = a[3]["emergency_stop"].astype(bool).mean()
        print(f"[gpu continuous edges large {name} {arm}] 4096 x 1000: latched {latched:.4f}")
        assert latched <= CE.LIVE_MAX_LATCHED.get(name, 0.0) + 0.01, f"{name}: {latched:.3f} latched"


@pytest.mark.parametrize("arm", ARMS)
def test_elbow_circle_normal_in_isclose_band(oracle, arm):
    """Regression (the device twin of test_continuous_edges_host.py's): the FP64 solve of poses whose elbow-circle normal
    lies within the isclose band of +-e_x, against the oracle."""
    from parity import Report
    from reachy2_symbolic_ik_b200 import SymbolicIK

    M = CE.live_families(arm, only=("slow_rmfv",))["slow_rmfv"][::2].reshape(-1, 4, 4)
    res = SymbolicIK(arm=arm).is_reachable_batch(M)
    want = oracle.symik_batch(oracle.arm_config(arm), M)
    rep = Report(f"gpu rmfv band {arm}", len(M))
    rep.exact("reachable", res.reachable, want[0])
    rep.exact("state", res.state, want[2])
    rep.close("interval", res.theta_interval, want[1])
    rep.close("joints", res.joints, want[3])
    rep.check(max_ill_fraction=0.0)
