"""CPU check of the *kernel source logic*: tests/hostsim compiles the device solver headers
(r2ik_device.cuh, r2ik_control.cuh) for the host and this file compares them with the
reference's golden outputs.  It exists so that logic regressions are caught in the GPU-less
CI; the GPU parity tests proper (``-m gpu``, tests/test_gpu_*.py) go through libr2ik.so.
The harness is test infrastructure: the package never loads it."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from parity import (CTOR_VARIANTS, OVERRIDE_DISCRETE, OVERRIDE_VARIANTS, REPO, Report, check_f32, ill_conditioned_mask, load,
                    run_with_unfreeze)
from reachy2_symbolic_ik_b200 import _abi

HS_DIR = os.path.join(REPO, "tests", "hostsim")
ARMS = ("r_arm", "l_arm")


@pytest.fixture(scope="module")
def hs():
    subprocess.run(["make", "-C", HS_DIR], check=True, capture_output=True)
    L = C.CDLL(os.path.join(HS_DIR, "_build", "libr2ik_hostsim.so"))
    return L


def dp(a):
    return a.ctypes.data_as(C.POINTER(C.c_double))


def u8(a):
    return a.ctypes.data_as(C.POINTER(C.c_uint8))


def cfg_for(arm, params=None, singularity_offset=0.03):
    return _abi.make_arm_config(arm, params or _abi.DEFAULT_IK_PARAMETERS, 127, 42.5, 1e-8, 0.02, 1e-7,
                                singularity_offset, 1.0)


def hs_symik(hs, cfg, P, theta=None):
    P = np.ascontiguousarray(P, dtype=np.float64)
    n = len(P)
    kind = _abi.POSE_MAT4 if P.shape[1:] == (4, 4) else _abi.POSE_EULER6
    reach = np.zeros(n, np.uint8); state = np.zeros(n, np.uint8)
    itv = np.empty((n, 2)); j = np.empty((n, 7)); e = np.empty((n, 3))
    th = None if theta is None else np.ascontiguousarray(theta, dtype=np.float64)
    hs.hs_symik_batch(C.byref(cfg), kind, dp(P), dp(th) if th is not None else None, C.c_int64(n), u8(reach), u8(state),
                      dp(itv), dp(j), dp(e))
    return reach.astype(bool), itv, state, j, e


def urdf_params():
    u = load("symik_urdf.npz")
    return {k[len("param_"):]: u[k] for k in u.files if k.startswith("param_")}


@pytest.mark.parametrize("arm", ARMS)
@pytest.mark.parametrize("layout", ["euler", "mat4"])
def test_symik_random(hs, oracle, arm, layout):
    g = load(f"symik_random_{arm}.npz")
    P = g["goal_pose"] if layout == "euler" else g["M"]
    ocfg = oracle.arm_config(arm)
    ill = ill_conditioned_mask(lambda p: oracle.symik_batch(ocfg, p.reshape(P.shape))[:4], P.reshape(len(P), -1))
    cfg = cfg_for(arm)
    reach, itv, state, joints, elbow = hs_symik(hs, cfg, P)
    rep = Report(f"hostsim random {arm} {layout}", len(P), ill)
    rep.exact("reachable", reach, g["reachable"])
    rep.exact("state", state, g["state"])
    rep.close("interval", itv, g["interval"])
    rep.close("joints", joints, g["joints"])
    rep.close("elbow", elbow, g["elbow"])
    _, _, _, j2, e2 = hs_symik(hs, cfg, P, g["theta2"])
    rep.close("joints@theta2", j2, g["joints_theta2"])
    rep.close("elbow@theta2", e2, g["elbow_theta2"])
    rep.check()


@pytest.mark.parametrize("arm", ARMS)
@pytest.mark.parametrize("variant", sorted(CTOR_VARIANTS))
def test_constructor_variants(hs, oracle, arm, variant):
    """Non-default elbow / wrist limits, margins and singularity plane (symbolic_ik.py:26-37) on the kernel source."""
    g = load("symik_ctor.npz")
    kw = dict(elbow_limit=127, wrist_limit=42.5, projection_margin=1e-8, backward_limit=0.02, normal_vector_margin=1e-7,
              singularity_offset=0.03, singularity_limit_coeff=1.0)
    kw.update(CTOR_VARIANTS[variant])
    cfg = _abi.make_arm_config(arm, kw.get("ik_parameters", _abi.DEFAULT_IK_PARAMETERS), kw["elbow_limit"], kw["wrist_limit"], kw["projection_margin"],
                               kw["backward_limit"], kw["normal_vector_margin"], kw["singularity_offset"],
                               kw["singularity_limit_coeff"])
    ocfg = oracle.arm_config(arm, **CTOR_VARIANTS[variant])
    pre = f"{arm}_{variant}_"
    for layout in ("euler", "mat4"):
        P = g[f"{arm}_goal_pose"] if layout == "euler" else g[f"{arm}_M"]
        ill = ill_conditioned_mask(lambda p: oracle.symik_batch(ocfg, p.reshape(P.shape))[:4], P.reshape(len(P), -1))
        reach, itv, state, joints, elbow = hs_symik(hs, cfg, P)
        rep = Report(f"hostsim ctor {variant} {arm} {layout}", len(P), ill)
        rep.exact("reachable", reach, g[pre + "reachable"])
        rep.exact("state", state, g[pre + "state"])
        rep.close("interval", itv, g[pre + "interval"])
        rep.close("joints", joints, g[pre + "joints"])
        rep.close("elbow", elbow, g[pre + "elbow"])
        _, _, _, j2, e2 = hs_symik(hs, cfg, P, g[pre + "theta2"])
        rep.close("joints@theta2", j2, g[pre + "joints_theta2"])
        rep.close("elbow@theta2", e2, g[pre + "elbow_theta2"])
        rep.check(max_ill_fraction=0.03)
    # is_reachable_no_limits (symbolic_ik.py:85-119) on the first / last h poses (FK-sampled / task space)
    Mn = g[f"{arm}_M"]
    h = len(g[pre + "nl_theta"]) // 2
    sel = np.r_[0:h, len(Mn) - h:len(Mn)]
    Mc = np.ascontiguousarray(Mn[sel])
    th = np.ascontiguousarray(g[pre + "nl_theta"])
    nj = np.empty((len(sel), 7)); ne = np.empty((len(sel), 3))
    hs.hs_no_limits_batch(C.byref(cfg), _abi.POSE_MAT4, dp(Mc), dp(th), C.c_int64(len(sel)), dp(nj), dp(ne))
    ill_nl = ill_conditioned_mask(lambda p: oracle.symik_no_limits_batch(ocfg, p.reshape(Mc.shape), th), Mc.reshape(len(sel), -1))
    rep = Report(f"hostsim ctor {variant} {arm} no_limits", len(sel), ill_nl)
    rep.close("no_limits joints", nj, g[pre + "nl_joints"])
    rep.close("no_limits elbow", ne, g[pre + "nl_elbow"])
    rep.check(max_ill_fraction=0.03)


@pytest.mark.parametrize("arm", ARMS)
def test_big_euler_angles(hs, oracle, arm):
    """Goal orientations as euler angles far outside [-pi, pi]: the argument reduction of the kernels' sincos (fast
    route for ordinary magnitudes, literal route beyond) against scipy's from_euler in the reference."""
    g = load("symik_big_euler.npz")
    P = g[f"{arm}_goal_pose"]
    ocfg = oracle.arm_config(arm)
    ill = ill_conditioned_mask(lambda p: oracle.symik_batch(ocfg, p.reshape(P.shape))[:4], P.reshape(len(P), -1))
    reach, itv, state, joints, elbow = hs_symik(hs, cfg_for(arm), P)
    rep = Report(f"hostsim big euler {arm}", len(P), ill)
    rep.exact("reachable", reach, g[f"{arm}_reachable"])
    rep.exact("state", state, g[f"{arm}_state"])
    rep.close("interval", itv, g[f"{arm}_interval"])
    rep.close("joints", joints, g[f"{arm}_joints"])
    rep.close("elbow", elbow, g[f"{arm}_elbow"])
    rep.check(max_ill_fraction=0.03)
    P32 = P.astype(np.float32)
    check_f32(f"hostsim f32 big euler {arm}", oracle, arm, P32, hs_symik_f32(hs, cfg_for(arm), P32), max_ill=0.04)


@pytest.mark.parametrize("arm", ARMS)
def test_fk_round_trip(hs, arm):
    """Reference-independent property: forward kinematics of the returned joints reproduces the goal pose whenever no
    goal-shifting branch fired (singularity_offset = -1.01 disables the elbow projection).  Host twin of
    tests/test_gpu_workspace.py::test_fk_round_trip_full_size; the URDF's truncated rpy literals bound the agreement
    at ~1e-6 (SURVEY.md section 4)."""
    from reachy2_symbolic_ik_b200 import fk

    q = fk.sample_fk_joints(40_000, np.random.default_rng(21))
    M = fk.forward_kinematics(q, arm)
    reach, itv, state, joints, elbow = hs_symik(hs, cfg_for(arm, None, -1.01), M)
    assert 0.3 < reach.mean() < 0.7
    M2 = fk.forward_kinematics(joints[reach], arm)
    rot_err = np.abs(M2[:, :3, :3] - M[reach][:, :3, :3]).max(axis=(1, 2))
    pos_err = np.linalg.norm(M2[:, :3, 3] - M[reach][:, :3, 3], axis=1)
    assert np.quantile(rot_err, 0.999) < 1e-5
    assert np.median(pos_err) < 1e-6 and (pos_err < 1e-5).mean() > 0.9
    # every theta of the interval is a solution of the same pose: the round trip holds at a second theta too
    width = np.where(itv[:, 0] <= itv[:, 1], itv[:, 1] - itv[:, 0], itv[:, 1] + 2 * np.pi - itv[:, 0])
    theta2 = np.where(reach, itv[:, 0] + 0.37 * width, 0.0)
    _, _, _, j2, _ = hs_symik(hs, cfg_for(arm, None, -1.01), M, theta2)
    M3 = fk.forward_kinematics(j2[reach], arm)
    assert np.quantile(np.abs(M3[:, :3, :3] - M[reach][:, :3, :3]).max(axis=(1, 2)), 0.999) < 1e-5
    p3 = np.linalg.norm(M3[:, :3, 3] - M[reach][:, :3, 3], axis=1)
    assert np.median(p3) < 1e-6 and (p3 < 1e-5).mean() > 0.9


@pytest.mark.parametrize("arm", ARMS)
def test_named(hs, oracle, arm):
    g = load("symik_named.npz")
    P = g[f"{arm}_poses"]
    ocfg = oracle.arm_config(arm)
    ill = ill_conditioned_mask(lambda p: oracle.symik_batch(ocfg, p.reshape(P.shape))[:4], P.reshape(len(P), -1))
    reach, itv, state, joints, elbow = hs_symik(hs, cfg_for(arm), P)
    rep = Report(f"hostsim named {arm}", len(P), ill)
    rep.exact("reachable", reach, g[f"{arm}_reachable"])
    rep.exact("state", state, g[f"{arm}_state"])
    rep.close("interval", itv, g[f"{arm}_interval"])
    rep.close("joints", joints, g[f"{arm}_joints"])
    rep.check(max_ill_fraction=0.1)


@pytest.mark.parametrize("arm", ARMS)
def test_urdf_and_no_limits(hs, oracle, arm):
    g = load("symik_urdf.npz")
    params = urdf_params()
    M = g[f"{arm}_M"]
    ocfg = oracle.arm_config(arm, ik_parameters=params, singularity_offset=-1.01)
    th = g[f"{arm}_nl_theta"]
    run = lambda p: oracle.symik_batch(ocfg, p.reshape(M.shape))[:4] + oracle.symik_no_limits_batch(  # noqa: E731
        ocfg, p.reshape(M.shape), th)
    ill = ill_conditioned_mask(run, M.reshape(len(M), -1))
    cfg = cfg_for(arm, params, -1.01)
    reach, itv, state, joints, elbow = hs_symik(hs, cfg, M)
    rep = Report(f"hostsim urdf {arm}", len(M), ill)
    rep.exact("reachable", reach, g[f"{arm}_reachable"])
    rep.exact("state", state, g[f"{arm}_state"])
    rep.close("interval", itv, g[f"{arm}_interval"])
    rep.close("joints", joints, g[f"{arm}_joints"])
    n = len(M)
    nj = np.empty((n, 7)); ne = np.empty((n, 3))
    Mc = np.ascontiguousarray(M)
    hs.hs_no_limits_batch(C.byref(cfg), _abi.POSE_MAT4, dp(Mc), dp(np.ascontiguousarray(th)), C.c_int64(n), dp(nj), dp(ne))
    rep.close("no_limits joints", nj, g[f"{arm}_nl_joints"])
    rep.close("no_limits elbow", ne, g[f"{arm}_nl_elbow"])
    rep.check()


def ctl_params(oracle, arm, **kw):
    """R2ikCtlParams has the oracle's field layout; fill it from the oracle's ControlParams."""
    op = oracle.ControlParams(arm=arm, **kw)._c
    p = _abi.CtlParams()
    C.memmove(C.byref(p), C.byref(op), C.sizeof(p))
    return p


@pytest.mark.parametrize("arm", ARMS)
@pytest.mark.parametrize("variant", ["k20", "k360", "low", "dvt"])
def test_ctl_discrete(hs, oracle, arm, variant):
    g = load(f"ctl_discrete_{arm}.npz")
    params = urdf_params()
    off = 0.03 if variant == "dvt" else -1.01
    want_j, want_f, want_s = g[f"joints_{variant}"], g[f"reachable_{variant}"], g[f"state_{variant}"]
    M = np.ascontiguousarray(g["M"][: len(want_j)])
    kw = dict(nb_search_points=360 if variant == "k360" else 20,
              constrained_mode="low_elbow" if variant == "low" else "unconstrained")
    ocfg = oracle.arm_config(arm, ik_parameters=params, singularity_offset=off)
    opar = oracle.ControlParams(arm=arm, **kw)
    ill = ill_conditioned_mask(lambda p: oracle.ctl_discrete_batch(ocfg, opar, p.reshape(M.shape))[:3], M.reshape(len(M), -1))
    cfg = cfg_for(arm, params, off)
    par = ctl_params(oracle, arm, **kw)
    n = len(M)
    prev = np.array(oracle.DEFAULT_PREV_JOINTS[arm])
    joints = np.empty((n, 7)); reach = np.zeros(n, np.uint8); state = np.zeros(n, np.uint8); emg = np.zeros(n, np.uint8)
    hs.hs_ctl_discrete_batch(C.byref(cfg), C.byref(par), dp(M), C.c_int64(n), dp(prev), dp(prev), dp(joints), u8(reach),
                             u8(state), u8(emg))
    rep = Report(f"hostsim ctl discrete {arm} {variant}", n, ill)
    rep.exact("reachable", reach.astype(bool), want_f)
    rep.exact("state", state, want_s)
    rep.close("joints", joints, want_j)
    rep.check(max_ill_fraction=0.02)


@pytest.mark.parametrize("arm", ARMS)
@pytest.mark.parametrize("variant", ["default", "cj", "dvt"])
def test_ctl_continuous(hs, oracle, arm, variant):
    g = load(f"ctl_continuous_{arm}.npz")
    params = urdf_params()
    off = 0.03 if variant == "dvt" else -1.01
    pre = {"default": "", "cj": "cj_", "dvt": "dvt_"}[variant]
    want_j, want_f, want_s = g[pre + "joints"], g[pre + "reachable"], g[pre + "state"]
    T, W = want_j.shape[:2]
    M = np.ascontiguousarray(g["M"][:T])
    cj = np.empty((T, 7)); cp = np.empty((T, 4, 4))
    cj[:] = g["cj_current_joints"] if variant == "cj" else oracle.DEFAULT_PREV_JOINTS[arm]
    cp[:] = g["cj_current_pose"] if variant == "cj" else oracle.DEFAULT_CURRENT_POSE[arm]
    st = np.zeros(T, dtype=_abi.TRAJ_STATE_DTYPE)
    st["init"] = 1
    joints = np.empty((T, W, 7)); reach = np.zeros((T, W), np.uint8); state = np.zeros((T, W), np.uint8)
    cfg = cfg_for(arm, params, off)
    par = ctl_params(oracle, arm)
    hs.hs_ctl_continuous_batch(C.byref(cfg), C.byref(par), dp(M), C.c_int64(T), C.c_int32(W), dp(cj), dp(cp),
                               st.ctypes.data_as(C.c_void_p), dp(joints), u8(reach), u8(state))
    for t in range(T):
        rep = Report(f"hostsim ctl continuous {arm} {variant} traj {t}", W)
        rep.exact("reachable", reach[t].astype(bool), want_f[t])
        rep.exact("state", state[t], want_s[t])
        rep.close("joints", joints[t], want_j[t])
        rep.check()
    np.testing.assert_array_equal(st["emergency_stop"].astype(bool), g[pre + "emergency"])
    np.testing.assert_allclose(st["previous_theta"], g[pre + "final_theta"], atol=1e-9)
    # the phased form (per-waypoint phases + per-trajectory scans on winding codes)
    st2 = np.zeros(T, dtype=_abi.TRAJ_STATE_DTYPE)
    st2["init"] = 1
    j2 = np.empty((T, W, 7)); r2 = np.zeros((T, W), np.uint8); s2 = np.zeros((T, W), np.uint8); ws = np.empty((T, W))
    cd = np.zeros((T, W), np.uint16)
    hs.hs_ctl_continuous_phased_batch(C.byref(cfg), C.byref(par), dp(M), C.c_int64(T), C.c_int32(W), dp(cj), dp(cp),
                                      st2.ctypes.data_as(C.c_void_p), dp(j2), u8(r2), u8(s2), dp(ws), cd.ctypes.data_as(C.c_void_p), C.c_int(0))
    assert_phased_equals_serial((j2, r2, s2, st2), (joints, reach, state, st), f"{arm} {variant}")


def assert_phased_equals_serial(phased, serial, what=""):
    """The phased form against the serial recursion: flags, states and the integer controller state identical, joints /
    previous_sol equal to rounding (an ordinary waypoint's joints are its raw joints plus whole turns in the phased form,
    prev + angle_diff(j, prev) in the serial one), previous_theta identical."""
    np.testing.assert_allclose(phased[0], serial[0], rtol=0, atol=1e-12, err_msg=f"{what} joints")
    np.testing.assert_array_equal(phased[1], serial[1], err_msg=f"{what} flags")
    np.testing.assert_array_equal(phased[2], serial[2], err_msg=f"{what} states")
    for f in ("has_previous_sol", "init", "emergency_stop", "emergency_bits"):
        np.testing.assert_array_equal(phased[3][f], serial[3][f], err_msg=f"{what} controller {f}")
    np.testing.assert_allclose(phased[3]["previous_sol"], serial[3]["previous_sol"], rtol=0, atol=1e-12, err_msg=f"{what} previous_sol")
    np.testing.assert_array_equal(phased[3]["previous_theta"], serial[3]["previous_theta"], err_msg=f"{what} previous_theta")


def hs_continuous(hs, oracle, cfg, par, arm, M, states=None, phased=False, force_serial=0):
    M = np.ascontiguousarray(M, dtype=np.float64)
    T, W = M.shape[:2]
    cj = np.empty((T, 7)); cp = np.empty((T, 4, 4))
    cj[:] = oracle.DEFAULT_PREV_JOINTS[arm]
    cp[:] = oracle.DEFAULT_CURRENT_POSE[arm]
    if states is None:
        states = np.zeros(T, dtype=_abi.TRAJ_STATE_DTYPE)
        states["init"] = 1
    st = np.ascontiguousarray(states).copy()
    joints = np.empty((T, W, 7)); reach = np.zeros((T, W), np.uint8); state = np.zeros((T, W), np.uint8)
    if phased:   # phases 1-2, the joints kernel with winding codes, the scan on codes (csrc/r2ik_cont_codes.cuh)
        ws = np.empty((T, W)); cd = np.zeros((T, W), np.uint16)
        hs.hs_ctl_continuous_phased_batch(C.byref(cfg), C.byref(par), dp(M), C.c_int64(T), C.c_int32(W), dp(cj), dp(cp),
                                          st.ctypes.data_as(C.c_void_p), dp(joints), u8(reach), u8(state), dp(ws),
                                          cd.ctypes.data_as(C.c_void_p), C.c_int(force_serial))
    else:
        hs.hs_ctl_continuous_batch(C.byref(cfg), C.byref(par), dp(M), C.c_int64(T), C.c_int32(W), dp(cj), dp(cp),
                                   st.ctypes.data_as(C.c_void_p), dp(joints), u8(reach), u8(state))
    return joints, reach.astype(bool), state, st


@pytest.mark.parametrize("arm", ARMS)
@pytest.mark.parametrize("variant", sorted(OVERRIDE_VARIANTS))
def test_ctl_continuous_overrides(hs, oracle, arm, variant):
    """Per-call d_theta_max / preferred_theta / constrained_mode (control_ik.py:162-172), serial and phased forms."""
    g = load(f"ctl_overrides_{arm}.npz")
    cfg = cfg_for(arm, urdf_params(), -1.01)
    par = ctl_params(oracle, arm, **OVERRIDE_VARIANTS[variant])
    pre = f"con_{variant}_"
    M = g["M"]
    T, W = M.shape[:2]
    joints, reach, state, st = hs_continuous(hs, oracle, cfg, par, arm, M)
    for t in range(T):
        rep = Report(f"hostsim ctl continuous override {variant} {arm} traj {t}", W)
        rep.exact("reachable", reach[t], g[pre + "reachable"][t])
        rep.exact("state", state[t], g[pre + "state"][t])
        rep.close("joints", joints[t], g[pre + "joints"][t])
        rep.check()
    np.testing.assert_array_equal(st["emergency_stop"].astype(bool), g[pre + "emergency"])
    np.testing.assert_allclose(st["previous_theta"], g[pre + "final_theta"], atol=1e-9)
    assert_phased_equals_serial(hs_continuous(hs, oracle, cfg, par, arm, M, phased=True), (joints, reach, state, st))


@pytest.mark.parametrize("arm", ARMS)
@pytest.mark.parametrize("variant", sorted(OVERRIDE_DISCRETE))
def test_ctl_discrete_overrides(hs, oracle, arm, variant):
    g = load(f"ctl_overrides_{arm}.npz")
    params = urdf_params()
    M = np.ascontiguousarray(g["dis_M"])
    ocfg = oracle.arm_config(arm, ik_parameters=params, singularity_offset=-1.01)
    opar = oracle.ControlParams(arm=arm, **OVERRIDE_DISCRETE[variant])
    ill = ill_conditioned_mask(lambda p: oracle.ctl_discrete_batch(ocfg, opar, p.reshape(M.shape))[:3], M.reshape(len(M), -1))
    cfg = cfg_for(arm, params, -1.01)
    par = ctl_params(oracle, arm, **OVERRIDE_DISCRETE[variant])
    n = len(M)
    prev = np.array(oracle.DEFAULT_PREV_JOINTS[arm])
    joints = np.empty((n, 7)); reach = np.zeros(n, np.uint8); state = np.zeros(n, np.uint8); emg = np.zeros(n, np.uint8)
    hs.hs_ctl_discrete_batch(C.byref(cfg), C.byref(par), dp(M), C.c_int64(n), dp(prev), dp(prev), dp(joints), u8(reach),
                             u8(state), u8(emg))
    rep = Report(f"hostsim ctl discrete override {variant} {arm}", n, ill)
    rep.exact("reachable", reach.astype(bool), g[f"dis_{variant}_reachable"])
    rep.exact("state", state, g[f"dis_{variant}_state"])
    rep.close("joints", joints, g[f"dis_{variant}_joints"])
    rep.check(max_ill_fraction=0.02)


@pytest.mark.parametrize("arm", ARMS)
def test_ctl_discrete_multiturn_previous_solution(hs, oracle, arm):
    """Discrete mode from a multi-turn previous solution (allow_multiturn, +-6 pi clamp, emergency bits;
    utils.py:493-568) and explicit current_joints, on the kernel source."""
    g = load(f"ctl_overrides_{arm}.npz")
    params = urdf_params()
    ocfg = oracle.arm_config(arm, ik_parameters=params, singularity_offset=-1.01)
    opar = oracle.ControlParams(arm=arm)
    cfg = cfg_for(arm, params, -1.01)
    par = ctl_params(oracle, arm)
    n = g["dis_mt_joints"].shape[1]
    M = np.ascontiguousarray(g["dis_M"][:n])
    cur = np.ascontiguousarray(g["dis_mt_current"])
    for k in range(len(g["dis_mt_prev"])):
        prev = np.ascontiguousarray(g["dis_mt_prev"][k])
        ill = ill_conditioned_mask(lambda p: oracle.ctl_discrete_batch(ocfg, opar, p.reshape(M.shape), prev_joints=prev,
                                                                       current_joints=cur)[:3], M.reshape(len(M), -1))
        joints = np.empty((n, 7)); reach = np.zeros(n, np.uint8); state = np.zeros(n, np.uint8); emg = np.zeros(n, np.uint8)
        hs.hs_ctl_discrete_batch(C.byref(cfg), C.byref(par), dp(M), C.c_int64(n), dp(prev), dp(cur), dp(joints), u8(reach),
                                 u8(state), u8(emg))
        rep = Report(f"hostsim ctl discrete multiturn {arm} prev {k}", n, ill)
        rep.exact("reachable", reach.astype(bool), g["dis_mt_reachable"][k])
        rep.exact("state", state, g["dis_mt_state"][k])
        rep.exact("emergency bits", emg, g["dis_mt_bits"][k])
        rep.close("joints", joints, g["dis_mt_joints"][k])
        rep.check(max_ill_fraction=0.03)


@pytest.mark.parametrize("arm", ARMS)
def test_ctl_continuous_multiturn(hs, oracle, arm):
    """Multi-turn wrist yaw up to the +-6 pi clamp and its emergency latch, serial and phased forms of the kernel source."""
    g = load(f"ctl_overrides_{arm}.npz")
    cfg = cfg_for(arm, urdf_params(), -1.01)
    par = ctl_params(oracle, arm)
    M = g["mt_M"]
    T, W = M.shape[:2]
    joints, reach, state, st = hs_continuous(hs, oracle, cfg, par, arm, M)
    for t in range(T):
        rep = Report(f"hostsim ctl continuous multi-turn {arm} traj {t}", W)
        rep.exact("reachable", reach[t], g["mt_reachable"][t])
        rep.exact("state", state[t], g["mt_state"][t])
        rep.close("joints", joints[t], g["mt_joints"][t])
        rep.check()
    np.testing.assert_array_equal(st["emergency_stop"].astype(bool), g["mt_emergency"])
    np.testing.assert_allclose(st["previous_theta"], g["mt_final_theta"], atol=1e-9)
    assert_phased_equals_serial(hs_continuous(hs, oracle, cfg, par, arm, M, phased=True), (joints, reach, state, st))


@pytest.mark.parametrize("arm", ARMS)
def test_ctl_continuous_winding_codes(hs, oracle, arm):
    """The phased K3 with its finish pass on winding codes (csrc/r2ik_cont_codes.cuh: cont_wind_code +
    cont_finish_codes_trajectory, the functions the kernels call) against the serial recursion: flags, states and controller flags identical, joints and
    previous_sol equal to rounding (nj = j + 2 pi k instead of prev + angle_diff(j, prev)) -- on the golden trajectories
    (continuity latch, unreachable stretches), the multi-turn ramps (windings past +-pi, the +-6 pi clamp and its
    emergency bits), trajectories longer than a 128-waypoint block, resumed states, invalid rotations, and with the test
    hook sending every m-th waypoint down the serial get_joints route."""
    from reachy2_symbolic_ik_b200 import fk

    cfg = cfg_for(arm, urdf_params(), -1.01)
    par = ctl_params(oracle, arm)
    g, go = load(f"ctl_continuous_{arm}.npz"), load(f"ctl_overrides_{arm}.npz")
    long = fk.sinusoidal_trajectories(5, 300, arm, seed=77)[0].copy()
    long[1, 140:, :3, :3] = long[1, 140:, :3, :3] @ np.diag([-1.0, -1.0, 1.0])      # discontinuity -> latch
    long[2, 129, :3, :3] = np.diag([-1.0, 1.0, 1.0])                                # invalid rotation right after a block edge
    long[3, 127, :3, :3] = np.diag([-1.0, 1.0, 1.0])                                # ... and right before one
    hit_clamp = wound = False

    same = assert_phased_equals_serial

    for name, M in (("golden", g["M"]), ("multi-turn", go["mt_M"]), ("unfreeze", go["unf_M"][None]), ("long", long)):
        M = np.ascontiguousarray(M)
        want = hs_continuous(hs, oracle, cfg, par, arm, M)
        for force in (0, 1, 7, 97):
            same(hs_continuous(hs, oracle, cfg, par, arm, M, phased=True, force_serial=force), want, f"{name} force={force}")
        hit_clamp = hit_clamp or bool((want[3]["emergency_bits"] & 7).any())
        wound = wound or bool((np.abs(np.nan_to_num(want[0])) > np.pi + 1e-6).any())
        Mr = np.ascontiguousarray(M[:, ::-1])       # resume the reversed trajectories from the returned states
        same(hs_continuous(hs, oracle, cfg, par, arm, Mr, states=want[3], phased=True),
             hs_continuous(hs, oracle, cfg, par, arm, Mr, states=want[3]), f"{name} resumed")
    assert hit_clamp and wound, "no trajectory wound past pi / reached the +-6 pi clamp"


@pytest.mark.parametrize("arm", ARMS)
@pytest.mark.parametrize("phased", [False, True])
def test_ctl_unfreeze(hs, oracle, arm, phased):
    """Emergency latch, frozen returns, then control_type="unfreeze" (control_ik.py:198-212) on the kernel source."""
    g = load(f"ctl_overrides_{arm}.npz")
    cfg = cfg_for(arm, urdf_params(), -1.01)
    par = ctl_params(oracle, arm)
    M = g["unf_M"]
    st0 = np.zeros(1, dtype=_abi.TRAJ_STATE_DTYPE)
    st0["init"] = 1
    seg = lambda m, st: hs_continuous(hs, oracle, cfg, par, arm, m, states=st, phased=phased)  # noqa: E731
    joints, reach, state, st = run_with_unfreeze(seg, M, g["unf_at"], st0)
    rep = Report(f"hostsim ctl unfreeze {arm} phased={phased}", len(M))
    rep.exact("reachable", reach, g["unf_reachable"])
    rep.exact("state", state, g["unf_state"])
    rep.close("joints", joints, g["unf_joints"])
    rep.check()
    assert bool(st["emergency_stop"][0]) == bool(g["unf_emergency_after"][-1])
    np.testing.assert_allclose(st["previous_theta"][0], g["unf_final_theta"], atol=1e-9)


def test_limit_orbita3d_wrist_fast_route(hs):
    """utl:508-532: the algebraic clamp of the kernels against (i) the reference outputs in the helper
    fixtures and (ii) scipy's own conversions on random wrists, incl. near the cone boundary."""
    from scipy.spatial.transform import Rotation as R

    def run(w, max_angle):
        w = np.ascontiguousarray(w, dtype=np.float64)
        out = np.empty_like(w)
        hs.hs_limit_orbita3d(dp(w), C.c_int64(len(w)), C.c_double(max_angle), dp(out))
        return out

    h = load("helpers.npz")
    mx = np.deg2rad(42.5)
    assert np.abs(run(h["wrist_in"], mx) - h["wrist_out"]).max() < 1e-12

    def ref(w, max_angle):   # the reference function, restated with scipy
        zyz = R.from_euler("XYZ", w).as_euler("ZYZ")
        zyz[:, 1] = np.clip(zyz[:, 1], -max_angle, max_angle)
        return R.from_euler("ZYZ", zyz).as_euler("XYZ")

    rng = np.random.default_rng(0)
    w = np.concatenate([rng.uniform(-1.2, 1.2, (20000, 3)), rng.uniform(-np.pi, np.pi, (20000, 3))])
    # wrists right at the cone boundary: beta = max +- 1e-9 .. 1e-3
    al, ga = rng.uniform(-np.pi, np.pi, (2, 2000))
    be = mx + rng.choice([-1, 1], 2000) * 10.0 ** rng.uniform(-9, -3, 2000)
    w = np.concatenate([w, R.from_euler("ZYZ", np.stack([al, be, ga], 1)).as_euler("XYZ")])
    import warnings
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        want = ref(w, mx)
    got = run(w, mx)
    # compare as rotations (angle triples near +-pi wrap) and as angles away from the wrap
    err_rot = (R.from_euler("XYZ", got).inv() * R.from_euler("XYZ", want)).magnitude()
    assert err_rot.max() < 1e-12, err_rot.max()
    d = np.abs(np.angle(np.exp(1j * (got - want))))
    assert d.max() < 1e-11, d.max()
    exact = np.abs(got - want) < 1e-11
    assert exact.mean() > 0.999      # the rest sit at the +-pi wrap of an output angle


# ---------------------------------------------------------------------------------------------------
# FP32 fast path (csrc/r2ik_device_f32.cuh) on the host: states identical to the FP64 oracle on the widened
# inputs, joints / intervals within 1e-4 rad on poses that are well-conditioned at FP32 resolution.
# ---------------------------------------------------------------------------------------------------
def fp(a):
    return a.ctypes.data_as(C.POINTER(C.c_float))


def hs_symik_f32(hs, cfg, P32, theta=None, mode=0):
    P32 = np.ascontiguousarray(P32, dtype=np.float32)
    n = len(P32)
    kind = _abi.POSE_MAT4 if P32.shape[1:] == (4, 4) else _abi.POSE_EULER6
    reach = np.zeros(n, np.uint8); state = np.zeros(n, np.uint8); esc = np.zeros(n, np.uint8)
    itv = np.empty((n, 2), np.float32); j = np.empty((n, 7), np.float32); e = np.empty((n, 3), np.float32)
    th = None if theta is None else np.ascontiguousarray(theta, dtype=np.float32)
    hs.hs_symik_batch_f32(C.byref(cfg), kind, fp(P32), fp(th) if th is not None else None, C.c_int64(n), C.c_int(mode), u8(reach),
                          u8(state), fp(itv), fp(j), fp(e), u8(esc))
    return reach.astype(bool), itv, state, j, e, esc.astype(bool)


@pytest.mark.parametrize("arm", ARMS)
@pytest.mark.parametrize("layout", ["euler", "mat4"])
def test_symik_f32_random(hs, oracle, arm, layout):
    g = load(f"symik_random_{arm}.npz")
    P32 = (g["goal_pose"] if layout == "euler" else g["M"]).astype(np.float32)
    check_f32(f"hostsim f32 random {arm} {layout}", oracle, arm, P32, hs_symik_f32(hs, cfg_for(arm), P32))
    th = g["theta2"].astype(np.float32)
    check_f32(f"hostsim f32 random {arm} {layout} @theta2", oracle, arm, P32, hs_symik_f32(hs, cfg_for(arm), P32, th), theta=th)


@pytest.mark.parametrize("arm", ARMS)
@pytest.mark.parametrize("variant", sorted(CTOR_VARIANTS))
def test_symik_f32_constructor_variants(hs, oracle, arm, variant):
    """The FP32 fast path under non-default limits / margins / singularity plane: its error bands and escalation
    tests are written against the constants of the handle, not the default ones."""
    g = load("symik_ctor.npz")
    kw = dict(elbow_limit=127, wrist_limit=42.5, projection_margin=1e-8, backward_limit=0.02, normal_vector_margin=1e-7,
              singularity_offset=0.03, singularity_limit_coeff=1.0)
    kw.update(CTOR_VARIANTS[variant])
    cfg = _abi.make_arm_config(arm, kw.get("ik_parameters", _abi.DEFAULT_IK_PARAMETERS), kw["elbow_limit"], kw["wrist_limit"], kw["projection_margin"],
                               kw["backward_limit"], kw["normal_vector_margin"], kw["singularity_offset"],
                               kw["singularity_limit_coeff"])
    ocfg = oracle.arm_config(arm, **CTOR_VARIANTS[variant])
    P32 = g[f"{arm}_M"].astype(np.float32)
    check_f32(f"hostsim f32 ctor {variant} {arm}", oracle, arm, P32, hs_symik_f32(hs, cfg, P32), ocfg=ocfg, max_ill=0.04)


@pytest.mark.parametrize("arm", ARMS)
def test_symik_f32_stretched_arm_boundary(hs, oracle, arm):
    """FK samples with an elbow pitch of 1e-6 .. 2e-3 rad put the wrist within ~1e-7 m of the range sphere d = L1 + L2.
    The FP32 path's wrist centre carries the ~1e-8 m error of its FP32 rotation, so "wrist out of range" against "reachable"
    must be settled by the FP64 solver there (2 of 1 000 000 plain FK samples differed before the band on d^2 existed:
    profiles/r1_experiments.md).  States identical to the FP64 oracle; the raw FP32 decision alone is not."""
    from reachy2_symbolic_ik_b200 import fk

    rng = np.random.default_rng(5)
    q = fk.sample_fk_joints(150_000, rng)
    q[:, 3] = -10.0 ** rng.uniform(-6, -2.7, len(q))
    M = fk.forward_kinematics(q, arm)
    M = M[M[:, 0, 3] > 0.1]
    P32 = M.astype(np.float32)
    want = oracle.symik_batch(oracle.arm_config(arm), P32.astype(np.float64))
    assert 0.05 < (want[2] == 3).mean() < 0.95            # the sample straddles the sphere
    got = hs_symik_f32(hs, cfg_for(arm), P32)
    assert np.array_equal(got[2], want[2]) and np.array_equal(got[0], want[0])
    raw = hs_symik_f32(hs, cfg_for(arm), P32, mode=1)
    assert (raw[2] != want[2]).sum() > 0


@pytest.mark.parametrize("arm", ARMS)
def test_symik_f32_fk_20k(hs, oracle, arm):
    from reachy2_symbolic_ik_b200 import fk

    P32 = np.concatenate([fk.sample_fk_poses(15000, arm, seed=21), fk.sample_task_space_poses(5000, arm, seed=22)]).astype(np.float32)
    check_f32(f"hostsim f32 fk+task {arm}", oracle, arm, P32, hs_symik_f32(hs, cfg_for(arm), P32))


def test_symik_f32_named_and_degenerate(hs, oracle):
    g = load("symik_named.npz")
    for arm in ARMS:
        P32 = g[f"{arm}_poses"].astype(np.float32)
        got = hs_symik_f32(hs, cfg_for(arm), P32)
        # every named pose keeps the reference's state (float32 inputs widened), however close to a boundary
        want = oracle.symik_batch(oracle.arm_config(arm), P32.astype(np.float64))
        assert np.array_equal(got[2], want[2])
        assert np.array_equal(got[0], want[0])
    # exact-zero / scaled / left-handed rotations are handed to the FP64 solver
    M = np.tile(np.eye(4, dtype=np.float32), (4, 1, 1))
    M[:, :3, 3] = [0.3, -0.2, -0.3]
    M[1, :3, :3] *= 1.5
    M[2, 0, 0] = -1.0
    M[3, :3, :3] = 0.0
    r, itv, st, j, e, esc = hs_symik_f32(hs, cfg_for("r_arm"), M)
    want = oracle.symik_batch(oracle.arm_config("r_arm"), M.astype(np.float64))
    assert np.array_equal(st, want[2]) and esc[1:].all()
    assert np.nanmax(np.abs(j - want[3])) < 1e-5


# ---------------------------------------------------------------------------------------------------
# K2's analytic elbow search (search_analytic) against the exhaustive scan of the K samples
# ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("nb", [8, 10, 20, 360, 3600])
@pytest.mark.parametrize("mode", ["full", "interval"])
def test_search_analytic_equals_scan(hs, nb, mode):
    rng = np.random.default_rng(nb + (0 if mode == "full" else 1))
    n = 50000
    plans = np.empty((n, 9))
    if mode == "full":                                   # utl:366-369 full circle: [pi/2, 5pi/2]
        plans[:, 0] = np.pi / 2; plans[:, 1] = np.pi / 2 + 2 * np.pi
    else:                                                # utl:370-375 interval, unrolled past pi when wrapped
        i0 = rng.uniform(-np.pi, np.pi, n); i1 = rng.uniform(-np.pi, np.pi, n)
        plans[:, 0] = i0; plans[:, 1] = np.where(i0 < i1, i1, i1 + 2 * np.pi)
    for c in (2, 3, 5, 6):                               # half-plane tests with the magnitudes of the arm (r <= 0.28 m)
        plans[:, c] = rng.uniform(-0.28, 0.28, n)
    for c in (4, 7):
        plans[:, c] = rng.uniform(-0.35, 0.2, n)
    plans[:, 8] = rng.choice([-2 * np.pi / 3, -np.pi / 3, 0.3, 2.5], n)
    # samples exactly on a crossing / on the preferred angle
    plans[:100, 8] = plans[:100, 0] + (plans[:100, 1] - plans[:100, 0]) * rng.integers(0, nb, 100) / (nb - 1)
    bs = np.empty(n); ba = np.empty(n); ks = np.empty(n, np.int32); ka = np.empty(n, np.int32); ok = np.empty(n, np.uint8)
    vp = lambda a: a.ctypes.data_as(C.c_void_p)  # noqa: E731
    hs.hs_search_compare(vp(plans), C.c_int64(n), C.c_int(nb), vp(bs), vp(ks), vp(ba), vp(ka), vp(ok))
    assert ok.all()
    found = np.isfinite(bs)
    assert 0.3 < found.mean() < 0.99
    assert np.array_equal(found, np.isfinite(ba))
    assert np.array_equal(ks, ka), f"{int((ks != ka).sum())} arg-min differ"
    assert np.array_equal(bs[found], ba[found])


# ---------------------------------------------------------------------------------------------------
# K4's mixed-precision flag (reach_flag_mixed + FP64 escalation) against the oracle's reach map: identical counts
# ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("arm", ARMS)
def test_reach_map_mixed_flag_counts(hs, oracle, arm):
    from reachy2_symbolic_ik_b200 import fk, workspace

    n, no = 36, 40
    shoulder = np.array([0.0, -0.2 if arm == "r_arm" else 0.2, 0.0])
    origin, step, dims = workspace.reach_grid(shoulder, 0.66, n)
    origin = origin + 3e-4                      # off the symmetric grid
    ori = fk.fibonacci_orientations(no)
    vp = lambda a: a.ctypes.data_as(C.c_void_p)  # noqa: E731
    want = oracle.reach_map(oracle.arm_config(arm), origin, step, dims, ori).reshape(-1)
    cfg = cfg_for(arm)
    res = {}
    for mode in (0, 1):
        counts = np.zeros(n ** 3, np.uint32)
        n_esc, n_live = C.c_uint64(), C.c_uint64()
        hs.hs_reach_map_mixed(C.byref(cfg), vp(origin), vp(step), vp(dims), vp(ori), C.c_int32(0), C.c_int32(no), C.c_int(mode),
                              vp(counts), C.byref(n_esc), C.byref(n_live))
        res[mode] = (counts, n_esc.value / max(n_live.value, 1))
    assert np.array_equal(res[0][0], want), "mixed-precision reach map differs from the oracle"
    assert res[0][1] < 2e-3, f"too many pairs escalated to FP64: {res[0][1]:.2e}"
    # without the escalation only a handful of pairs differ: the bands are what makes the counts exact
    assert np.abs(res[1][0].astype(np.int64) - want.astype(np.int64)).sum() < 1e-4 * want.sum()


@pytest.mark.parametrize("variant", sorted(CTOR_VARIANTS))
def test_reach_map_mixed_flag_constructor_variants(hs, oracle, variant):
    """K4's mixed-precision flag under non-default limits / margins / geometry: its FP32 error bands are written against
    the constants of the handle; the counts must still be the oracle's."""
    from reachy2_symbolic_ik_b200 import fk, workspace

    arm = "l_arm"
    kw = dict(elbow_limit=127, wrist_limit=42.5, projection_margin=1e-8, backward_limit=0.02, normal_vector_margin=1e-7,
              singularity_offset=0.03, singularity_limit_coeff=1.0)
    kw.update(CTOR_VARIANTS[variant])
    params = kw.get("ik_parameters", _abi.DEFAULT_IK_PARAMETERS)
    cfg = _abi.make_arm_config(arm, params, kw["elbow_limit"], kw["wrist_limit"], kw["projection_margin"],
                               kw["backward_limit"], kw["normal_vector_margin"], kw["singularity_offset"],
                               kw["singularity_limit_coeff"])
    n, no = 30, 32
    origin, step, dims = workspace.reach_grid(np.asarray(params["l_shoulder_position"], dtype=np.float64), 0.66, n)
    origin = origin + 3e-4
    ori = fk.fibonacci_orientations(no)
    vp = lambda a: a.ctypes.data_as(C.c_void_p)  # noqa: E731
    want = oracle.reach_map(oracle.arm_config(arm, **CTOR_VARIANTS[variant]), origin, step, dims, ori).reshape(-1)
    counts = np.zeros(n ** 3, np.uint32)
    n_esc, n_live = C.c_uint64(), C.c_uint64()
    hs.hs_reach_map_mixed(C.byref(cfg), vp(origin), vp(step), vp(dims), vp(ori), C.c_int32(0), C.c_int32(no), C.c_int(0),
                          vp(counts), C.byref(n_esc), C.byref(n_live))
    assert want.sum() > 10_000
    assert np.array_equal(counts, want), f"{int((counts != want).sum())} voxels differ from the oracle"
    assert n_esc.value < 2e-3 * n_live.value


def test_reach_map_mixed_flag_regression_pairs(hs, oracle):
    """Two (voxel, orientation) pairs of the full 256^3 x 512 map whose discriminant is 3e-9 from zero while the planes
    are 3 degrees from parallel (the cancellation in 1 - Ca^2 is then the largest FP32 error): they must be escalated."""
    from reachy2_symbolic_ik_b200 import fk, workspace

    origin, step, dims = workspace.reach_grid(np.array([0.0, -0.2, 0.0]), 0.66, 256)
    ori = fk.fibonacci_orientations(512)
    one = np.array([1, 1, 1], np.int32)
    vp = lambda a: a.ctypes.data_as(C.c_void_p)  # noqa: E731
    cfg = cfg_for("r_arm")
    for vox, o in (([196, 191, 113], 17), ([223, 115, 124], 118)):
        p = origin + np.array(vox) * step
        oo = np.ascontiguousarray(ori[o:o + 1])
        want = oracle.reach_map(oracle.arm_config("r_arm"), p, step, one, oo).reshape(-1)[0]
        counts = np.zeros(1, np.uint32)
        n_esc, n_live = C.c_uint64(), C.c_uint64()
        hs.hs_reach_map_mixed(C.byref(cfg), vp(p), vp(step), vp(one), vp(oo), C.c_int32(0), C.c_int32(1), C.c_int(0), vp(counts),
                              C.byref(n_esc), C.byref(n_live))
        assert counts[0] == want == 0 and n_esc.value == 1


@pytest.mark.parametrize("arm", ARMS)
def test_reference_example_matrices(hs, oracle, arm):
    """The goal matrices printed in the reference's examples (tests/golden/ctl_examples.npz) through the kernel source:
    SymbolicIK (4x4 input), ControlIK discrete, ControlIK continuous (serial and phased forms)."""
    g = load("ctl_examples.npz")
    params = urdf_params()
    M = np.ascontiguousarray(g[f"{arm}_M"])
    n = len(M)
    reach, itv, state, joints, elbow = hs_symik(hs, cfg_for(arm), M)
    assert np.array_equal(state, g[f"{arm}_sym_state"]) and np.array_equal(reach, g[f"{arm}_sym_reachable"])
    np.testing.assert_allclose(itv, g[f"{arm}_sym_interval"], atol=1e-9, equal_nan=True)
    np.testing.assert_allclose(joints, g[f"{arm}_sym_joints"], atol=1e-9, equal_nan=True)
    cfg = cfg_for(arm, params, -1.01)
    par = ctl_params(oracle, arm)
    prev = np.array(oracle.DEFAULT_PREV_JOINTS[arm])
    dj = np.empty((n, 7)); dr = np.zeros(n, np.uint8); ds = np.zeros(n, np.uint8); de = np.zeros(n, np.uint8)
    hs.hs_ctl_discrete_batch(C.byref(cfg), C.byref(par), dp(M), C.c_int64(n), dp(prev), dp(prev), dp(dj), u8(dr), u8(ds), u8(de))
    assert np.array_equal(ds, g[f"{arm}_dis_state"]) and np.array_equal(dr.astype(bool), g[f"{arm}_dis_reachable"])
    np.testing.assert_allclose(dj, g[f"{arm}_dis_joints"], atol=1e-9)
    W = g[f"{arm}_con_joints"].shape[1]
    MT = np.ascontiguousarray(np.repeat(M[:, None], W, axis=1))
    cj = np.empty((n, 7)); cp = np.empty((n, 4, 4))
    cj[:] = oracle.DEFAULT_PREV_JOINTS[arm]; cp[:] = oracle.DEFAULT_CURRENT_POSE[arm]
    for entry in ("hs_ctl_continuous_batch", "hs_ctl_continuous_phased_batch"):
        st = np.zeros(n, dtype=_abi.TRAJ_STATE_DTYPE); st["init"] = 1
        j = np.empty((n, W, 7)); r = np.zeros((n, W), np.uint8); s_ = np.zeros((n, W), np.uint8)
        args = [C.byref(cfg), C.byref(par), dp(MT), C.c_int64(n), C.c_int32(W), dp(cj), dp(cp), st.ctypes.data_as(C.c_void_p),
                dp(j), u8(r), u8(s_)]
        if entry.endswith("phased_batch"):
            ws = np.empty((n, W)); cd = np.zeros((n, W), np.uint16)
            args += [dp(ws), cd.ctypes.data_as(C.c_void_p), C.c_int(0)]
        getattr(hs, entry)(*args)
        assert np.array_equal(s_, g[f"{arm}_con_state"]) and np.array_equal(r.astype(bool), g[f"{arm}_con_reachable"]), entry
        np.testing.assert_allclose(j, g[f"{arm}_con_joints"], atol=1e-9)
        assert np.array_equal(st["emergency_stop"].astype(bool), g[f"{arm}_con_emergency"])


def test_task_space_sweep(hs):
    """Kernel source on the reference's task_space_test grid (37 376 poses, Euler angles in steps of 45 degrees: a dense
    sample of the solver's special cases): states equal the reference's, FP64 and FP32 paths."""
    from reachy2_symbolic_ik_b200 import workspace

    g = load("task_space.npz")
    poses = workspace.task_space_grid([0.0, -0.2, 0.0])
    want = np.unpackbits(g["reachable_packed"])[: len(poses)].astype(bool)
    reach, itv, state, joints, elbow = hs_symik(hs, cfg_for("r_arm"), poses)
    assert np.array_equal(state, g["state"]) and np.array_equal(reach, want)
    r32, i32, s32, j32, e32, esc = hs_symik_f32(hs, cfg_for("r_arm"), poses.astype(np.float32))
    assert int((s32 != g["state"]).sum()) <= 40       # the FP32 path sees the float32-rounded grid
    assert 0.02 < esc.mean() < 0.3                    # axis-aligned orientations sit on the special cases: many re-solves


@pytest.mark.parametrize("kind", ["float32_rounded", "five_digits"])
def test_non_orthonormal_rotation_blocks(hs, oracle, kind):
    """4x4 goals whose rotation block is not orthonormal (float32-rounded, or printed with 5 digits like the matrices in
    the reference's examples): scipy replaces the block by its polar factor; the kernel source uses that factor directly
    outside the gimbal band (no quaternion / as_euler / from_euler detour).  FP64 path against the oracle, 1e-9 rad."""
    from reachy2_symbolic_ik_b200 import fk

    M = fk.sample_fk_poses(20000, "r_arm", seed=5)
    X = M.astype(np.float32).astype(np.float64) if kind == "float32_rounded" else np.round(M, 5)
    ocfg = oracle.arm_config("r_arm")
    ill = ill_conditioned_mask(lambda p: oracle.symik_batch(ocfg, p.reshape(X.shape))[:4], X.reshape(len(X), -1), n_trials=2)
    want = oracle.symik_batch(ocfg, X)
    reach, itv, state, joints, elbow = hs_symik(hs, cfg_for("r_arm"), X)
    rep = Report(f"hostsim non-orthonormal {kind}", len(X), ill)
    rep.exact("state", state, want[2])
    rep.close("interval", itv, want[1])
    rep.close("joints", joints, want[3])
    rep.check(max_ill_fraction=0.03)   # FK-sampled poses reach down to a straight arm: ~1.7 % move by > 1e-10 under 3e-13


@pytest.mark.parametrize("is_dvt", [False, True])
def test_constructor_previous_theta(hs, is_dvt):
    """ControlIK.previous_theta as the reference's constructor seeds it (control_ik.py:142-159; ternary search over the
    two-arm joint list) on the kernel source: default and custom current_joints / current_pose (tests/golden/ctl_ctor.npz)."""
    g = load("ctl_ctor.npz")
    tag = "dvt" if is_dvt else "std"
    params = urdf_params()
    hs.hs_ctl_ctor_theta.restype = C.c_double
    hs.hs_ctl_ctor_theta.argtypes = [C.c_void_p, C.c_double, C.POINTER(C.c_double), C.c_int, C.POINTER(C.c_double)]
    default_cj = np.array([[0.0, 0.2617993877991494, -0.17453292519943295, 0.0, 0.0, 0.0, 0.0],
                           [0.0, -0.2617993877991494, 0.17453292519943295, 0.0, 0.0, 0.0, 0.0]])
    default_cp = np.array([[[1, 0, 0, 0], [0, 1, 0, -0.2], [0, 0, 1, -0.66], [0, 0, 0, 1]],
                           [[1, 0, 0, 0], [0, 1, 0, 0.2], [0, 0, 1, -0.66], [0, 0, 0, 1]]], dtype=np.float64)
    cases = [("default", default_cj, default_cp)] + [(f"v{v}", g[f"v{v}_current_joints"], g[f"v{v}_current_pose"])
                                                     for v in range(int(g["n_variants"]))]
    for name, cj, cp in cases:
        for k, arm in enumerate(ARMS):
            cfg = cfg_for(arm, params, 0.03 if is_dvt else -1.01)
            pref = -4 * np.pi / 6 if arm == "r_arm" else -np.pi + 4 * np.pi / 6
            rows = np.ascontiguousarray(cj, dtype=np.float64)
            pose = np.ascontiguousarray(cp[k], dtype=np.float64)
            got = hs.hs_ctl_ctor_theta(C.byref(cfg), pref, dp(rows), len(rows), dp(pose))
            assert abs(got - float(g[f"{tag}_{name}_{arm}"])) < 1e-9, (name, arm, got, float(g[f"{tag}_{name}_{arm}"]))


@pytest.mark.parametrize("arm", ARMS)
def test_elbow_positions(hs, oracle, arm):
    """get_elbow_position after is_reachable / is_reachable_no_limits and the projection predicate on the kernel source
    (tests/golden/symik_elbow.npz; the GPU twin is tests/test_gpu_api_r2.py::test_elbow_positions_entry)."""
    g = load("symik_elbow.npz")
    cfg = cfg_for(arm)
    ocfg = oracle.arm_config(arm)
    P = np.ascontiguousarray(g[f"{arm}_goal_pose"].reshape(-1, 6))
    n, K = g[f"{arm}_thetas"].shape
    th, nth = np.ascontiguousarray(g[f"{arm}_thetas"]), np.ascontiguousarray(g[f"{arm}_nl_thetas"])
    run = lambda p: (oracle.elbow_positions_batch(ocfg, p.reshape(n, 2, 3), th),  # noqa: E731
                     oracle.elbow_positions_batch(ocfg, p.reshape(n, 2, 3), nth, no_limits=True))
    ill = ill_conditioned_mask(run, P)
    rep = Report(f"hostsim elbow {arm}", n, ill)
    for no_limits, thetas, want, want_len in ((0, th, g[f"{arm}_elbow_position"], g[f"{arm}_gj_elbow_len"]),
                                              (1, nth, g[f"{arm}_nl_elbow_position"], g[f"{arm}_nl_elbow_len"])):
        E = np.empty((n, K, 3)); proj = np.zeros((n, K), np.uint8)
        hs.hs_elbow_positions(C.byref(cfg), _abi.POSE_EULER6, dp(P), dp(thetas), K, C.c_int64(n), no_limits, dp(E), u8(proj))
        rep.close(f"get_elbow_position (no_limits={no_limits})", E, want[:, :, :3])
        valid = want_len > 0
        rep.exact(f"elbow shape of get_joints (no_limits={no_limits})", np.where(valid, np.where(proj.astype(bool), 3, 4), 0), want_len)
    rep.check(max_ill_fraction=0.03)


@pytest.mark.parametrize("arm", ARMS)
@pytest.mark.parametrize("variant", ["k20", "k360", "low", "dvt"])
def test_ctl_discrete_three_passes_equal_one_pass(hs, oracle, arm, variant):
    """The three passes of r2ik_ctl_discrete_compact_f64 (classify -> search list -> finish list, the finish pass redoing
    only the elbow circle unless the solve was the literal one) on the host, against the one-pass form: the same bytes,
    whatever order the list entries arrive in; invalid rotation blocks and a wound previous solution included."""
    from reachy2_symbolic_ik_b200 import fk

    params = urdf_params()
    off = 0.03 if variant == "dvt" else -1.01
    kw = dict(nb_search_points=360 if variant == "k360" else 20,
              constrained_mode="low_elbow" if variant == "low" else "unconstrained")
    cfg = cfg_for(arm, params, off)
    par = ctl_params(oracle, arm, **kw)
    g = load(f"ctl_discrete_{arm}.npz")
    M = np.ascontiguousarray(np.concatenate([g["M"], fk.sample_fk_poses(6000, arm, seed=123), fk.sample_task_space_poses(3000, arm, seed=124),
                                             np.eye(4)[None]]))
    # tool axis along +-e_x: the wrist-limit plane normal hits rotation_matrix_from_vector's special cases (utils.py:66-70),
    # which the solver hands to its literal instantiation -- the list entries that carry the flag
    from scipy.spatial.transform import Rotation
    s_pos = np.array(oracle.arm_config(arm, ik_parameters=params, singularity_offset=off).shoulder_position)
    rng = np.random.default_rng(5)
    ahead = np.tile(np.eye(4), (400, 1, 1))
    for q in range(400):
        ahead[q, :3, :3] = (Rotation.from_euler("y", (np.pi / 2) * (1 if q % 2 else -1)) * Rotation.from_euler("z", rng.uniform(-np.pi, np.pi))).as_matrix()
    ahead[:, :3, 3] = s_pos + np.array([0.38, 0.0, -0.12]) + rng.uniform(-0.12, 0.12, (400, 3))
    M = np.ascontiguousarray(np.concatenate([M, ahead]))
    M[::97, :3, :3] = np.diag([1.0, 1.0, -1.0])        # det < 0
    n = len(M)
    n_literal = 0
    for prev, cur in ((np.array(oracle.DEFAULT_PREV_JOINTS[arm]),) * 2,
                      (np.array([0.3, -0.2, 7.0, -1.0, 0.1, 0.2, -6.5]), np.array([0.1, 0.2, 0.3, -0.4, 0.5, 0.6, 19.5]))):
        one = [np.full((n, 7), 5.0), np.full(n, 9, np.uint8), np.full(n, 99, np.uint8), np.full(n, 99, np.uint8)]
        hs.hs_ctl_discrete_batch(C.byref(cfg), C.byref(par), dp(M), C.c_int64(n), dp(prev), dp(cur), dp(one[0]), u8(one[1]), u8(one[2]), u8(one[3]))
        for order in (0, 1):
            three = [np.full((n, 7), 5.0), np.full(n, 9, np.uint8), np.full(n, 99, np.uint8), np.full(n, 99, np.uint8)]
            lists = np.zeros(3, np.int64)
            hs.hs_ctl_discrete_compact_batch(C.byref(cfg), C.byref(par), dp(M), C.c_int64(n), dp(prev), dp(cur), C.c_int(order), dp(three[0]),
                                             u8(three[1]), u8(three[2]), u8(three[3]), lists.ctypes.data_as(C.POINTER(C.c_int64)))
            for a, b in zip(one, three):
                assert np.array_equal(a, b, equal_nan=True)
            assert 0 < lists[0] < n and lists[0] * 0.2 < lists[1] < n
            assert int(three[1].sum()) == lists[1] and int((three[2] == 9).sum()) == len(M[::97])
            n_literal += int(lists[2])
    assert n_literal > 0, "no pose of the sample took the literal solve: the flag path of the finish pass was not exercised"
