"""GPU parity of the per-call overrides of ControlIK.symbolic_inverse_kinematics (d_theta_max, preferred_theta,
constrained_mode; control_ik.py:162-172) and of the "unfreeze" control type (:198-212) through the facade / C ABI,
against the reference's golden outputs (tests/golden/ctl_overrides_*.npz, gen_golden.py: gen_ctl_overrides).
The same fixtures pin the oracle (test_oracle_golden.py) and the kernel source on the host (test_hostsim_parity.py)."""
import numpy as np
import pytest

from parity import CTOR_VARIANTS, OVERRIDE_DISCRETE, OVERRIDE_VARIANTS, Report, ill_conditioned_mask, load, run_with_unfreeze
from reachy2_symbolic_ik_b200 import _abi

pytestmark = pytest.mark.gpu
ARMS = ("r_arm", "l_arm")


def urdf_params():
    u = load("symik_urdf.npz")
    return {k[len("param_"):]: u[k] for k in u.files if k.startswith("param_")}


@pytest.fixture(scope="module")
def ctl():
    from reachy2_symbolic_ik_b200 import ControlIK

    return ControlIK(urdf_path="../config_files/reachy2.urdf")


class FakeTime:
    """The clock of the fixture generator: 1/120 s per call, first call far from 0 (the time-out of
    control_ik.py:296-304 fires on the first call and never again)."""

    def __init__(self):
        self.t = 1000.0

    def time(self):
        self.t += 1.0 / 120.0
        return self.t


@pytest.mark.parametrize("arm", ARMS)
@pytest.mark.parametrize("phased", [True, False])
@pytest.mark.parametrize("variant", sorted(OVERRIDE_VARIANTS))
def test_continuous_overrides(ctl, arm, variant, phased):
    g = load(f"ctl_overrides_{arm}.npz")
    pre = f"con_{variant}_"
    M = np.ascontiguousarray(g["M"])
    T, W = M.shape[:2]
    joints, reach, state, st = ctl.symbolic_inverse_kinematics_batch(arm, M, "continuous", phased=phased,
                                                                     **OVERRIDE_VARIANTS[variant])
    for t in range(T):
        rep = Report(f"gpu ctl continuous override {variant} {arm} phased={phased} traj {t}", W)
        rep.exact("reachable", reach[t], g[pre + "reachable"][t])
        rep.exact("state", state[t], g[pre + "state"][t])
        rep.close("joints", joints[t], g[pre + "joints"][t])
        rep.check()
    np.testing.assert_array_equal(st["emergency_stop"].astype(bool), g[pre + "emergency"])
    np.testing.assert_allclose(st["previous_theta"], g[pre + "final_theta"], atol=1e-9)


@pytest.mark.parametrize("arm", ARMS)
@pytest.mark.parametrize("variant", sorted(OVERRIDE_DISCRETE))
def test_discrete_overrides(ctl, oracle, arm, variant):
    g = load(f"ctl_overrides_{arm}.npz")
    M = np.ascontiguousarray(g["dis_M"])
    ocfg = oracle.arm_config(arm, ik_parameters=urdf_params(), singularity_offset=-1.01)
    opar = oracle.ControlParams(arm=arm, **OVERRIDE_DISCRETE[variant])
    ill = ill_conditioned_mask(lambda p: oracle.ctl_discrete_batch(ocfg, opar, p.reshape(M.shape))[:3], M.reshape(len(M), -1))
    for exhaustive in (False, True):
        joints, reach, state, emg = ctl.symbolic_inverse_kinematics_batch(arm, M, "discrete", exhaustive=exhaustive,
                                                                          **OVERRIDE_DISCRETE[variant])
        rep = Report(f"gpu ctl discrete override {variant} {arm} exhaustive={exhaustive}", len(M), ill)
        rep.exact("reachable", reach, g[f"dis_{variant}_reachable"])
        rep.exact("state", state, g[f"dis_{variant}_state"])
        rep.close("joints", joints, g[f"dis_{variant}_joints"])
        rep.check(max_ill_fraction=0.02)
        assert not emg.any()


@pytest.mark.parametrize("arm", ARMS)
@pytest.mark.parametrize("phased", [True, False])
def test_unfreeze_batched(ctl, arm, phased):
    """The trajectory is cut at the "unfreeze" waypoints; the returned controller states are reset as the reference
    resets its own (emergency_stop, emergency_state, init) and passed back to resume."""
    g = load(f"ctl_overrides_{arm}.npz")
    M = g["unf_M"]
    st0 = np.zeros(1, dtype=_abi.TRAJ_STATE_DTYPE)
    st0["init"] = 1
    seg = lambda m, st: ctl.symbolic_inverse_kinematics_batch(arm, m, "continuous", states=st, phased=phased)  # noqa: E731
    joints, reach, state, st = run_with_unfreeze(seg, M, g["unf_at"], st0)
    rep = Report(f"gpu ctl unfreeze {arm} phased={phased}", len(M))
    rep.exact("reachable", reach, g["unf_reachable"])
    rep.exact("state", state, g["unf_state"])
    rep.close("joints", joints, g["unf_joints"])
    rep.check()
    assert bool(st["emergency_stop"][0]) == bool(g["unf_emergency_after"][-1])
    np.testing.assert_allclose(st["previous_theta"][0], g["unf_final_theta"], atol=1e-9)


@pytest.mark.parametrize("arm", ARMS)
def test_unfreeze_scalar_api(arm, monkeypatch):
    """The drop-in scalar call, one waypoint at a time, with control_type="unfreeze" where the fixture sent it:
    joints, flags, state strings and the emergency latch follow the reference call by call."""
    import reachy2_symbolic_ik_b200.control_ik as facade
    from reachy2_symbolic_ik_b200 import ControlIK

    g = load(f"ctl_overrides_{arm}.npz")
    M, unf = g["unf_M"], set(int(u) for u in g["unf_at"])
    monkeypatch.setattr(facade, "time", FakeTime())
    c = ControlIK(urdf_path="../config_files/reachy2.urdf")
    for w in range(len(M)):
        j, ok, s = c.symbolic_inverse_kinematics(arm, M[w], "unfreeze" if w in unf else "continuous")
        assert ok == bool(g["unf_reachable"][w]), w
        assert ("EMERGENCY" in s) == (g["unf_state"][w] == 8), (w, s)
        if g["unf_state"][w] != 8:
            assert s == "", (w, s)
        assert c.emergency_stop == bool(g["unf_emergency_after"][w]), w
        np.testing.assert_allclose(np.asarray(j, dtype=np.float64), g["unf_joints"][w], rtol=0, atol=1e-9, err_msg=f"waypoint {w}")
    np.testing.assert_allclose(c.previous_theta[arm], g["unf_final_theta"], atol=1e-9)


@pytest.mark.parametrize("arm", ARMS)
@pytest.mark.parametrize("phased", [True, False])
def test_continuous_multiturn(ctl, arm, phased):
    """Joint-space ramps through several turns: wrist yaw unwraps up to the +-6 pi clamp of multiturn_safety_check, which
    latches the emergency (utils.py:493-568)."""
    g = load(f"ctl_overrides_{arm}.npz")
    M = np.ascontiguousarray(g["mt_M"])
    T, W = M.shape[:2]
    joints, reach, state, st = ctl.symbolic_inverse_kinematics_batch(arm, M, "continuous", phased=phased)
    for t in range(T):
        rep = Report(f"gpu ctl continuous multi-turn {arm} phased={phased} traj {t}", W)
        rep.exact("reachable", reach[t], g["mt_reachable"][t])
        rep.exact("state", state[t], g["mt_state"][t])
        rep.close("joints", joints[t], g["mt_joints"][t])
        rep.check()
    np.testing.assert_array_equal(st["emergency_stop"].astype(bool), g["mt_emergency"])
    np.testing.assert_allclose(st["previous_theta"], g["mt_final_theta"], atol=1e-9)


@pytest.mark.parametrize("arm", ARMS)
def test_discrete_multiturn_previous_solution(ctl, oracle, arm):
    """Discrete mode from a multi-turn previous solution (allow_multiturn, the +-6 pi clamp and the emergency bits of
    multiturn_safety_check, utils.py:493-568) with explicit current_joints."""
    g = load(f"ctl_overrides_{arm}.npz")
    ocfg = oracle.arm_config(arm, ik_parameters=urdf_params(), singularity_offset=-1.01)
    opar = oracle.ControlParams(arm=arm)
    n = g["dis_mt_joints"].shape[1]
    M = np.ascontiguousarray(g["dis_M"][:n])
    cur = g["dis_mt_current"]
    for k in range(len(g["dis_mt_prev"])):
        prev = g["dis_mt_prev"][k]
        ill = ill_conditioned_mask(lambda p: oracle.ctl_discrete_batch(ocfg, opar, p.reshape(M.shape), prev_joints=prev,
                                                                       current_joints=cur)[:3], M.reshape(len(M), -1))
        for exhaustive in (False, True):
            joints, reach, state, emg = ctl.symbolic_inverse_kinematics_batch(
                arm, M, "discrete", previous_joints=prev, current_joints=cur, exhaustive=exhaustive)
            rep = Report(f"gpu ctl discrete multiturn {arm} prev {k} exhaustive={exhaustive}", n, ill)
            rep.exact("reachable", reach, g["dis_mt_reachable"][k])
            rep.exact("state", state, g["dis_mt_state"][k])
            rep.exact("emergency bits", emg, g["dis_mt_bits"][k])
            rep.close("joints", joints, g["dis_mt_joints"][k])
            rep.check(max_ill_fraction=0.03)


@pytest.mark.parametrize("arm", ARMS)
def test_big_euler_angles(oracle, arm):
    """Goal orientations as euler angles far outside [-pi, pi] (tests/golden/symik_big_euler.npz)."""
    from reachy2_symbolic_ik_b200 import SymbolicIK

    g = load("symik_big_euler.npz")
    P = g[f"{arm}_goal_pose"]
    ocfg = oracle.arm_config(arm)
    ill = ill_conditioned_mask(lambda p: oracle.symik_batch(ocfg, p.reshape(P.shape))[:4], P.reshape(len(P), -1))
    res = SymbolicIK(arm=arm).is_reachable_batch(P)
    rep = Report(f"gpu big euler {arm}", len(P), ill)
    rep.exact("reachable", res.reachable, g[f"{arm}_reachable"])
    rep.exact("state", res.state, g[f"{arm}_state"])
    rep.close("interval", res.theta_interval, g[f"{arm}_interval"])
    rep.close("joints@interval[0]", res.joints, g[f"{arm}_joints"])
    rep.close("elbow", res.elbow, g[f"{arm}_elbow"])
    rep.check(max_ill_fraction=0.03)


@pytest.mark.parametrize("arm", ARMS)
@pytest.mark.parametrize("variant", sorted(CTOR_VARIANTS))
def test_constructor_variants(oracle, arm, variant):
    """SymbolicIK with non-default elbow / wrist limits, margins and singularity plane (symbolic_ik.py:26-37):
    tests/golden/symik_ctor.npz through the facade."""
    from reachy2_symbolic_ik_b200 import SymbolicIK

    g = load("symik_ctor.npz")
    ik = SymbolicIK(arm=arm, **CTOR_VARIANTS[variant])
    ocfg = oracle.arm_config(arm, **CTOR_VARIANTS[variant])
    pre = f"{arm}_{variant}_"
    for layout in ("euler", "mat4"):
        P = g[f"{arm}_goal_pose"] if layout == "euler" else g[f"{arm}_M"]
        ill = ill_conditioned_mask(lambda p: oracle.symik_batch(ocfg, p.reshape(P.shape))[:4], P.reshape(len(P), -1))
        res = ik.is_reachable_batch(P)
        rep = Report(f"gpu ctor {variant} {arm} {layout}", len(P), ill)
        rep.exact("reachable", res.reachable, g[pre + "reachable"])
        rep.exact("state", res.state, g[pre + "state"])
        rep.close("interval", res.theta_interval, g[pre + "interval"])
        rep.close("joints@interval[0]", res.joints, g[pre + "joints"])
        rep.close("elbow", res.elbow, g[pre + "elbow"])
        res2 = ik.is_reachable_batch(P, theta=g[pre + "theta2"])
        rep.close("joints@theta2", res2.joints, g[pre + "joints_theta2"])
        rep.close("elbow@theta2", res2.elbow, g[pre + "elbow_theta2"])
        rep.check(max_ill_fraction=0.03)
    # is_reachable_no_limits (symbolic_ik.py:85-119) on the first / last h poses
    M = g[f"{arm}_M"]
    h = len(g[pre + "nl_theta"]) // 2
    sel = np.r_[0:h, len(M) - h:len(M)]
    Mc, th = np.ascontiguousarray(M[sel]), g[pre + "nl_theta"]
    ill = ill_conditioned_mask(lambda p: oracle.symik_no_limits_batch(ocfg, p.reshape(Mc.shape), th), Mc.reshape(len(sel), -1))
    nj, ne = ik.is_reachable_no_limits_batch(Mc, th)
    rep = Report(f"gpu ctor {variant} {arm} no_limits", len(sel), ill)
    rep.close("no_limits joints", nj, g[pre + "nl_joints"])
    rep.close("no_limits elbow", ne, g[pre + "nl_elbow"])
    rep.check(max_ill_fraction=0.03)


def test_facade_attributes_match_the_reference():
    """Every public attribute an instance of the reference's classes carries (tests/golden/api_surface.json) exists on
    the drop-in classes (examples read them: src/example/test_continuous_ik.py:60, 235-238)."""
    import json
    import os

    from parity import GOLDEN
    from reachy2_symbolic_ik_b200 import ControlIK, SymbolicIK

    ref = json.load(open(os.path.join(GOLDEN, "api_surface.json")))
    ik = SymbolicIK()
    missing = [a for a in ref["SymbolicIK_attributes"] if not hasattr(ik, a)]
    assert not missing, f"SymbolicIK lacks {missing}"
    c = ControlIK(urdf_path="../config_files/reachy2.urdf")
    missing = [a for a in ref["ControlIK_attributes"] if not hasattr(c, a)]
    assert not missing, f"ControlIK lacks {missing}"
