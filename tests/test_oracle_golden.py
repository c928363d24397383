"""Pins the CPU oracle (oracle/r2ik_oracle.c) to the reference's own outputs.

The fixtures under tests/golden/ were produced by the unmodified reference
(tests/golden/gen_golden.py; numpy / scipy versions stored inside each file).  The
reference's own CI test (tests/test_ik.py:12-79) only pins flags and shapes on 6 poses; those
6 poses are the first rows of symik_named.npz and are re-asserted literally below.
"""
import numpy as np
import pytest

from parity import CTOR_VARIANTS, OVERRIDE_DISCRETE, OVERRIDE_VARIANTS, Report, ill_conditioned_mask, load, run_with_unfreeze

ARMS = ("r_arm", "l_arm")


def test_reference_ci_assertions(oracle):
    """tests/test_ik.py:12-79 restated against the oracle (default right arm)."""
    g = load("symik_named.npz")
    cfg = oracle.arm_config("r_arm")
    P = g["r_arm_poses"][:6]
    reach, itv, state, joints, _ = oracle.symik_batch(cfg, P)
    assert not reach[0] and np.isnan(itv[0]).all()
    assert reach[1] and itv[1][0] >= -np.pi and itv[1][1] <= np.pi and np.isfinite(joints[1]).all()
    assert reach[2] and np.all(itv[2] == [-np.pi, np.pi])
    assert not reach[3]
    assert not reach[4]
    assert reach[5]
    # README.md:73-79 example
    reach, itv, state, joints, _ = oracle.symik_batch(cfg, g["r_arm_poses"][6:7])
    assert reach[0] and oracle.STATE_STRINGS[int(state[0])] == "reachable"
    np.testing.assert_allclose(itv[0], [2.18952378, -0.22393633], atol=1e-8)


@pytest.mark.parametrize("arm", ARMS)
def test_named_poses(oracle, arm):
    g = load("symik_named.npz")
    cfg = oracle.arm_config(arm)
    P = g[f"{arm}_poses"]
    run = lambda p: oracle.symik_batch(cfg, p.reshape(-1, 2, 3))[:4]  # noqa: E731
    ill = ill_conditioned_mask(run, P.reshape(len(P), 6))
    reach, itv, state, joints, elbow = oracle.symik_batch(cfg, P)
    rep = Report(f"oracle named {arm}", len(P), ill)
    rep.exact("reachable", reach, g[f"{arm}_reachable"])
    rep.exact("state", state, g[f"{arm}_state"])
    rep.close("interval", itv, g[f"{arm}_interval"])
    rep.close("joints", joints, g[f"{arm}_joints"])
    rep.close("elbow", elbow, g[f"{arm}_elbow"])
    _, _, _, j0, e0 = oracle.symik_batch(cfg, P, np.zeros(len(P)))
    rep.close("joints(theta=0)", j0, g[f"{arm}_joints_theta0"])
    rep.close("elbow(theta=0)", e0, g[f"{arm}_elbow_theta0"])
    rep.check(max_ill_fraction=0.1)  # the fully stretched arm (#10) is a true kinematic singularity


@pytest.mark.parametrize("arm", ARMS)
@pytest.mark.parametrize("layout", ["euler", "mat4"])
def test_random_poses(oracle, arm, layout):
    g = load(f"symik_random_{arm}.npz")
    cfg = oracle.arm_config(arm)
    P = g["goal_pose"] if layout == "euler" else g["M"]
    flat = P.reshape(len(P), -1)
    run = lambda p: oracle.symik_batch(cfg, p.reshape(P.shape))[:4]  # noqa: E731
    ill = ill_conditioned_mask(run, flat)
    reach, itv, state, joints, elbow = oracle.symik_batch(cfg, P)
    rep = Report(f"oracle random {arm} {layout}", len(P), ill)
    rep.exact("reachable", reach, g["reachable"])
    rep.exact("state", state, g["state"])
    rep.close("interval", itv, g["interval"])
    rep.close("joints@interval[0]", joints, g["joints"])
    rep.close("elbow", elbow, g["elbow"])
    _, _, _, j2, e2 = oracle.symik_batch(cfg, P, g["theta2"])
    rep.close("joints@theta2", j2, g["joints_theta2"])
    rep.close("elbow@theta2", e2, g["elbow_theta2"])
    rep.check()


@pytest.mark.parametrize("arm", ARMS)
@pytest.mark.parametrize("variant", sorted(CTOR_VARIANTS))
def test_constructor_variants(oracle, arm, variant):
    """Non-default elbow / wrist limits, margins and singularity plane (symbolic_ik.py:26-37)."""
    g = load("symik_ctor.npz")
    cfg = oracle.arm_config(arm, **CTOR_VARIANTS[variant])
    pre = f"{arm}_{variant}_"
    for layout in ("euler", "mat4"):
        P = g[f"{arm}_goal_pose"] if layout == "euler" else g[f"{arm}_M"]
        run = lambda p: oracle.symik_batch(cfg, p.reshape(P.shape))[:4]  # noqa: E731
        ill = ill_conditioned_mask(run, P.reshape(len(P), -1))
        reach, itv, state, joints, elbow = oracle.symik_batch(cfg, P)
        rep = Report(f"oracle ctor {variant} {arm} {layout}", len(P), ill)
        rep.exact("reachable", reach, g[pre + "reachable"])
        rep.exact("state", state, g[pre + "state"])
        rep.close("interval", itv, g[pre + "interval"])
        rep.close("joints@interval[0]", joints, g[pre + "joints"])
        rep.close("elbow", elbow, g[pre + "elbow"])
        _, _, _, j2, e2 = oracle.symik_batch(cfg, P, g[pre + "theta2"])
        rep.close("joints@theta2", j2, g[pre + "joints_theta2"])
        rep.close("elbow@theta2", e2, g[pre + "elbow_theta2"])
        rep.check(max_ill_fraction=0.03)
        # is_reachable_no_limits (symbolic_ik.py:85-119) on the first / last h poses (FK-sampled / task space)
        h = len(g[pre + "nl_theta"]) // 2
        sel = np.r_[0:h, len(P) - h:len(P)]
        nj, ne = oracle.symik_no_limits_batch(cfg, P[sel], g[pre + "nl_theta"])
        ill_nl = ill_conditioned_mask(lambda p: oracle.symik_no_limits_batch(cfg, p.reshape(P[sel].shape), g[pre + "nl_theta"]),
                                      P[sel].reshape(len(sel), -1))
        rep = Report(f"oracle ctor {variant} {arm} {layout} no_limits", len(sel), ill_nl)
        rep.close("no_limits joints", nj, g[pre + "nl_joints"])
        rep.close("no_limits elbow", ne, g[pre + "nl_elbow"])
        rep.check(max_ill_fraction=0.03)


@pytest.mark.parametrize("arm", ARMS)
def test_elbow_positions_and_return_shape(oracle, arm):
    """get_elbow_position(theta) after is_reachable and after is_reachable_no_limits (symbolic_ik.py:684-695, circle
    stored at :197 / :114-116), get_joints(theta, previous_joints) after is_reachable_no_limits, and the branch that
    decides the SHAPE of the elbow get_joints returns ((4,) [x, y, z, 1]; (3,) once make_elbow_projection fired, :714)."""
    g = load("symik_elbow.npz")
    cfg = oracle.arm_config(arm)
    P = g[f"{arm}_goal_pose"]
    n, K = g[f"{arm}_thetas"].shape
    flat = P.reshape(n, 6)
    th, nth = g[f"{arm}_thetas"], g[f"{arm}_nl_thetas"]
    run = lambda p: (oracle.symik_batch(cfg, p.reshape(P.shape))[0], oracle.elbow_positions_batch(cfg, p.reshape(P.shape), th),  # noqa: E731
                     oracle.elbow_positions_batch(cfg, p.reshape(P.shape), nth, no_limits=True))
    ill = ill_conditioned_mask(run, flat)
    rep = Report(f"oracle elbow {arm}", n, ill)
    reach = g[f"{arm}_reachable"]
    E, proj = oracle.elbow_positions_batch(cfg, P, th, with_projected=True)
    has_circle = reach | (g[f"{arm}_state"] == 4)          # stored at sik:197, also for "limited by wrist"
    rep.exact("circle stored (NaN rows otherwise)", np.isfinite(E).all(axis=(1, 2)), has_circle)
    rep.close("get_elbow_position after is_reachable", E, g[f"{arm}_elbow_position"][:, :, :3])
    assert np.all(g[f"{arm}_elbow_position"][has_circle][:, :, 3] == 1.0)
    rep.exact("elbow shape of get_joints (3 <=> projection fired)", np.where(reach[:, None], np.where(proj, 3, 4), 0),
              g[f"{arm}_gj_elbow_len"])
    Enl, proj_nl = oracle.elbow_positions_batch(cfg, P, nth, no_limits=True, with_projected=True)
    rep.close("get_elbow_position after is_reachable_no_limits", Enl, g[f"{arm}_nl_elbow_position"][:, :, :3])
    rep.exact("elbow shape of get_joints after no_limits", np.where(proj_nl, 3, 4), g[f"{arm}_nl_elbow_len"])
    for k in range(K):
        _, _, _, j, e = oracle.symik_batch(cfg, P, th[:, k])
        rep.close(f"get_joints(theta[{k}])", j, g[f"{arm}_gj_joints"][:, k])
        rep.close(f"elbow of get_joints(theta[{k}])", e, g[f"{arm}_gj_elbow"][:, k])
        j, e, pr = oracle.symik_no_limits_batch(cfg, P, nth[:, k], g[f"{arm}_nl_prev"], with_projected=True)
        rep.close(f"no_limits get_joints(theta[{k}], previous_joints)", j, g[f"{arm}_nl_joints"][:, k])
        rep.close(f"no_limits elbow of get_joints(theta[{k}])", e, g[f"{arm}_nl_elbow"][:, k])
        assert np.array_equal(pr, proj_nl[:, k])
    rep.check(max_ill_fraction=0.03)


@pytest.mark.parametrize("arm", ARMS)
def test_scalar_call_sequence_record(oracle, arm):
    """orc_symik_scalar (the checker of r2ik_symik_scalar_f64) against what the reference's scalar calls return and leave
    on the solver: goal_pose / wrist_position after is_reachable (sik:143-171) and after get_joints (sik:711-716)."""
    g = load("symik_elbow.npz")
    cfg = oracle.arm_config(arm)
    P = g[f"{arm}_goal_pose"]
    nf = int(g["n_fk"])
    idx = np.r_[0:120, nf:nf + 120, len(P) - 24:len(P)]  # FK-sampled, task-space and the named poses
    singular = len(P) - 24 + 10                           # the fully stretched arm: a true singularity (see test_named_poses)
    worst = 0.0
    for i in idx[idx != singular]:
        for k in (0, 3):
            th = g[f"{arm}_thetas"][i, k]
            r = oracle.symik_scalar(cfg, P[i], theta=th)
            assert r["state"] == g[f"{arm}_state"][i] and bool(r["reachable"]) == bool(g[f"{arm}_reachable"][i])
            for got, want in ((r["goal_position_solved"], g[f"{arm}_ir_goal"][i]), (r["wrist_position_solved"], g[f"{arm}_ir_wrist"][i]),
                              (r["elbow_on_circle"], g[f"{arm}_elbow_position"][i, k, :3]), (r["joints"], g[f"{arm}_gj_joints"][i, k]),
                              (r["elbow"], g[f"{arm}_gj_elbow"][i, k]), (r["goal_position"], g[f"{arm}_gj_goal"][i, k]),
                              (r["wrist_position"], g[f"{arm}_gj_wrist"][i, k])):
                assert np.array_equal(np.isnan(got), np.isnan(want)), (i, k)
                worst = max(worst, float(np.nanmax(np.abs(got - want), initial=0.0)))
            if r["reachable"]:
                assert (3 if r["projected"] else 4) == g[f"{arm}_gj_elbow_len"][i, k]
            th = g[f"{arm}_nl_thetas"][i, k]
            r = oracle.symik_scalar(cfg, P[i], no_limits=True, theta=th, previous_joints=g[f"{arm}_nl_prev"][i])
            assert r["reachable"] and (3 if r["projected"] else 4) == g[f"{arm}_nl_elbow_len"][i, k]
            for got, want in ((r["elbow_on_circle"], g[f"{arm}_nl_elbow_position"][i, k, :3]), (r["joints"], g[f"{arm}_nl_joints"][i, k]),
                              (r["elbow"], g[f"{arm}_nl_elbow"][i, k])):
                worst = max(worst, float(np.nanmax(np.abs(got - want), initial=0.0)))
    assert worst < 1e-9, worst


@pytest.mark.parametrize("arm", ARMS)
def test_big_euler_angles(oracle, arm):
    """Goal orientations as euler angles far outside [-pi, pi] (tests/golden/symik_big_euler.npz)."""
    g = load("symik_big_euler.npz")
    cfg = oracle.arm_config(arm)
    P = g[f"{arm}_goal_pose"]
    ill = ill_conditioned_mask(lambda p: oracle.symik_batch(cfg, p.reshape(P.shape))[:4], P.reshape(len(P), -1))
    reach, itv, state, joints, elbow = oracle.symik_batch(cfg, P)
    rep = Report(f"oracle big euler {arm}", len(P), ill)
    rep.exact("reachable", reach, g[f"{arm}_reachable"])
    rep.exact("state", state, g[f"{arm}_state"])
    rep.close("interval", itv, g[f"{arm}_interval"])
    rep.close("joints@interval[0]", joints, g[f"{arm}_joints"])
    rep.close("elbow", elbow, g[f"{arm}_elbow"])
    rep.check(max_ill_fraction=0.03)


def _urdf_cfg(oracle, g, arm, singularity_offset=-1.01):
    params = {k[len("param_"):]: g[k] for k in g.files if k.startswith("param_")}
    return oracle.arm_config(arm, ik_parameters=params, singularity_offset=singularity_offset)


@pytest.mark.parametrize("arm", ARMS)
def test_urdf_params_and_no_limits(oracle, arm):
    g = load("symik_urdf.npz")
    cfg = _urdf_cfg(oracle, g, arm)
    M = g[f"{arm}_M"]
    run = lambda p: oracle.symik_batch(cfg, p.reshape(M.shape))[:4] + oracle.symik_no_limits_batch(  # noqa: E731
        cfg, p.reshape(M.shape), g[f"{arm}_nl_theta"])
    ill = ill_conditioned_mask(run, M.reshape(len(M), -1))
    reach, itv, state, joints, elbow = oracle.symik_batch(cfg, M)
    rep = Report(f"oracle urdf {arm}", len(M), ill)
    rep.exact("reachable", reach, g[f"{arm}_reachable"])
    rep.exact("state", state, g[f"{arm}_state"])
    rep.close("interval", itv, g[f"{arm}_interval"])
    rep.close("joints", joints, g[f"{arm}_joints"])
    rep.close("elbow", elbow, g[f"{arm}_elbow"])
    nj, ne = oracle.symik_no_limits_batch(cfg, M, g[f"{arm}_nl_theta"])
    rep.close("no_limits joints", nj, g[f"{arm}_nl_joints"])
    rep.close("no_limits elbow", ne, g[f"{arm}_nl_elbow"])
    rep.check()


@pytest.mark.parametrize("arm", ARMS)
@pytest.mark.parametrize("variant", ["k20", "k360", "low", "dvt"])
def test_ctl_discrete(oracle, arm, variant):
    g = load(f"ctl_discrete_{arm}.npz")
    u = load("symik_urdf.npz")
    cfg = _urdf_cfg(oracle, u, arm, singularity_offset=0.03 if variant == "dvt" else -1.01)
    want_j, want_f, want_s = g[f"joints_{variant}"], g[f"reachable_{variant}"], g[f"state_{variant}"]
    M = g["M"][: len(want_j)]
    par = oracle.ControlParams(arm=arm, nb_search_points=360 if variant == "k360" else 20,
                               constrained_mode="low_elbow" if variant == "low" else "unconstrained")
    run = lambda p: oracle.ctl_discrete_batch(cfg, par, p.reshape(M.shape))[:3]  # noqa: E731
    ill = ill_conditioned_mask(run, M.reshape(len(M), -1))
    joints, reach, state, emg = oracle.ctl_discrete_batch(cfg, par, M)
    rep = Report(f"oracle ctl discrete {arm} {variant}", len(M), ill)
    rep.exact("reachable", reach, want_f)
    rep.exact("state", state, want_s)
    rep.close("joints", joints, want_j)
    assert not emg.any()
    rep.check(max_ill_fraction=0.02)


@pytest.mark.parametrize("arm", ARMS)
@pytest.mark.parametrize("variant", ["default", "cj", "dvt"])
def test_ctl_continuous(oracle, arm, variant):
    g = load(f"ctl_continuous_{arm}.npz")
    u = load("symik_urdf.npz")
    cfg = _urdf_cfg(oracle, u, arm, singularity_offset=0.03 if variant == "dvt" else -1.01)
    par = oracle.ControlParams(arm=arm)
    pre = {"default": "", "cj": "cj_", "dvt": "dvt_"}[variant]
    want_j, want_f, want_s = g[pre + "joints"], g[pre + "reachable"], g[pre + "state"]
    T, W = want_j.shape[:2]
    M = g["M"][:T]
    kw = {}
    if variant == "cj":
        kw = dict(current_joints=g["cj_current_joints"], current_pose=g["cj_current_pose"])
    joints, reach, state, st = oracle.ctl_continuous_batch(cfg, par, M, **kw)
    # a trajectory is a sequential recursion: compare every waypoint, report per trajectory
    for t in range(T):
        rep = Report(f"oracle ctl continuous {arm} {variant} traj {t}", W)
        rep.exact("reachable", reach[t], want_f[t])
        rep.exact("state", state[t], want_s[t])
        rep.close("joints", joints[t], want_j[t])
        rep.check()
    np.testing.assert_array_equal(st["emergency_stop"].astype(bool), g[pre + "emergency"])
    np.testing.assert_allclose(st["previous_theta"], g[pre + "final_theta"], atol=1e-9)


@pytest.mark.parametrize("arm", ARMS)
@pytest.mark.parametrize("variant", sorted(OVERRIDE_VARIANTS))
def test_ctl_continuous_overrides(oracle, arm, variant):
    """Per-call d_theta_max / preferred_theta / constrained_mode (control_ik.py:162-172) in continuous mode."""
    g = load(f"ctl_overrides_{arm}.npz")
    cfg = _urdf_cfg(oracle, load("symik_urdf.npz"), arm, singularity_offset=-1.01)
    par = oracle.ControlParams(arm=arm, **OVERRIDE_VARIANTS[variant])
    pre = f"con_{variant}_"
    M = g["M"]
    T, W = M.shape[:2]
    joints, reach, state, st = oracle.ctl_continuous_batch(cfg, par, M)
    for t in range(T):
        rep = Report(f"oracle ctl continuous override {variant} {arm} traj {t}", W)
        rep.exact("reachable", reach[t], g[pre + "reachable"][t])
        rep.exact("state", state[t], g[pre + "state"][t])
        rep.close("joints", joints[t], g[pre + "joints"][t])
        rep.check()
    np.testing.assert_array_equal(st["emergency_stop"].astype(bool), g[pre + "emergency"])
    np.testing.assert_allclose(st["previous_theta"], g[pre + "final_theta"], atol=1e-9)


@pytest.mark.parametrize("arm", ARMS)
@pytest.mark.parametrize("variant", sorted(OVERRIDE_DISCRETE))
def test_ctl_discrete_overrides(oracle, arm, variant):
    g = load(f"ctl_overrides_{arm}.npz")
    cfg = _urdf_cfg(oracle, load("symik_urdf.npz"), arm, singularity_offset=-1.01)
    par = oracle.ControlParams(arm=arm, **OVERRIDE_DISCRETE[variant])
    M = g["dis_M"]
    run = lambda p: oracle.ctl_discrete_batch(cfg, par, p.reshape(M.shape))[:3]  # noqa: E731
    ill = ill_conditioned_mask(run, M.reshape(len(M), -1))
    joints, reach, state, emg = oracle.ctl_discrete_batch(cfg, par, M)
    rep = Report(f"oracle ctl discrete override {variant} {arm}", len(M), ill)
    rep.exact("reachable", reach, g[f"dis_{variant}_reachable"])
    rep.exact("state", state, g[f"dis_{variant}_state"])
    rep.close("joints", joints, g[f"dis_{variant}_joints"])
    assert not emg.any()
    rep.check(max_ill_fraction=0.02)


@pytest.mark.parametrize("arm", ARMS)
def test_ctl_discrete_multiturn_previous_solution(oracle, arm):
    """Discrete mode from a multi-turn previous solution: allow_multiturn, the +-6 pi clamp and the emergency bits of
    multiturn_safety_check (utils.py:493-568); explicit current_joints come back for unreachable poses."""
    g = load(f"ctl_overrides_{arm}.npz")
    cfg = _urdf_cfg(oracle, load("symik_urdf.npz"), arm, singularity_offset=-1.01)
    par = oracle.ControlParams(arm=arm)
    n = g["dis_mt_joints"].shape[1]
    M = g["dis_M"][:n]
    assert (g["dis_mt_bits"] != 0).mean() > 0.3
    for k in range(len(g["dis_mt_prev"])):
        kw = dict(prev_joints=g["dis_mt_prev"][k], current_joints=g["dis_mt_current"])
        run = lambda p: oracle.ctl_discrete_batch(cfg, par, p.reshape(M.shape), **kw)[:3]  # noqa: E731
        ill = ill_conditioned_mask(run, M.reshape(len(M), -1))
        joints, reach, state, emg = oracle.ctl_discrete_batch(cfg, par, M, **kw)
        rep = Report(f"oracle ctl discrete multiturn {arm} prev {k}", n, ill)
        rep.exact("reachable", reach, g["dis_mt_reachable"][k])
        rep.exact("state", state, g["dis_mt_state"][k])
        rep.exact("emergency bits", emg, g["dis_mt_bits"][k])
        rep.close("joints", joints, g["dis_mt_joints"][k])
        rep.check(max_ill_fraction=0.03)


@pytest.mark.parametrize("arm", ARMS)
def test_ctl_continuous_multiturn(oracle, arm):
    """Joint-space ramps through several turns: allow_multiturn unwraps wrist yaw up to the +-6 pi clamp of
    multiturn_safety_check, which latches the emergency (utils.py:493-568)."""
    g = load(f"ctl_overrides_{arm}.npz")
    cfg = _urdf_cfg(oracle, load("symik_urdf.npz"), arm, singularity_offset=-1.01)
    par = oracle.ControlParams(arm=arm)
    M = g["mt_M"]
    T, W = M.shape[:2]
    assert np.abs(g["mt_joints"][..., 6]).max() > 5.9 * np.pi and g["mt_emergency"].any()
    joints, reach, state, st = oracle.ctl_continuous_batch(cfg, par, M)
    for t in range(T):
        rep = Report(f"oracle ctl continuous multi-turn {arm} traj {t}", W)
        rep.exact("reachable", reach[t], g["mt_reachable"][t])
        rep.exact("state", state[t], g["mt_state"][t])
        rep.close("joints", joints[t], g["mt_joints"][t])
        rep.check()
    np.testing.assert_array_equal(st["emergency_stop"].astype(bool), g["mt_emergency"])
    np.testing.assert_allclose(st["previous_theta"], g["mt_final_theta"], atol=1e-9)


@pytest.mark.parametrize("arm", ARMS)
def test_ctl_unfreeze(oracle, arm):
    """Emergency latch (continuity violation), the frozen returns, then control_type="unfreeze" (control_ik.py:198-212)."""
    g = load(f"ctl_overrides_{arm}.npz")
    cfg = _urdf_cfg(oracle, load("symik_urdf.npz"), arm, singularity_offset=-1.01)
    par = oracle.ControlParams(arm=arm)
    M = g["unf_M"]
    seg = lambda m, st: oracle.ctl_continuous_batch(cfg, par, m, states=st)  # noqa: E731
    joints, reach, state, st = run_with_unfreeze(seg, M, g["unf_at"], oracle.new_ctl_states(1))
    assert g["unf_emergency_after"].sum() > 10 and (g["unf_state"] == 8).sum() > 10
    rep = Report(f"oracle ctl unfreeze {arm}", len(M))
    rep.exact("reachable", reach, g["unf_reachable"])
    rep.exact("state", state, g["unf_state"])
    rep.close("joints", joints, g["unf_joints"])
    rep.check()
    assert bool(st["emergency_stop"][0]) == bool(g["unf_emergency_after"][-1])
    np.testing.assert_allclose(st["previous_theta"][0], g["unf_final_theta"], atol=1e-9)


def test_helpers(oracle):
    h = load("helpers.npz")
    eul = np.array([oracle.euler_xyz_from_matrix(m) for m in h["mat"]])
    # orthonormal inputs: 1e-14; truncated (5-digit) matrices go through the polar-factor
    # projection (scipy: SVD), where the agreement is limited by conditioning to ~1e-12
    assert np.abs(eul - h["mat_euler"])[:150].max() < 1e-14
    assert np.abs(eul - h["mat_euler"])[500:].max() < 1e-14
    assert np.abs(eul - h["mat_euler"]).max() < 1e-11
    orb = np.array([oracle.limit_orbita3d_joints(w, np.deg2rad(42.5)) for w in h["wrist_in"]])
    assert np.abs(orb - h["wrist_out"]).max() < 1e-13
    ad = np.array([oracle.angle_diff(a, b) for a, b in zip(h["ad_a"], h["ad_b"])])
    assert np.array_equal(ad, h["ad"])
    lt = np.array([oracle.limit_theta_to_interval(t, 0.0, i) for t, i in zip(h["lt_theta"], h["lt_interval"])])
    assert np.array_equal(lt, h["lt_out"])
    rm = np.array([oracle.rotation_matrix_from_vector(v) for v in h["rmfv_v"]])
    assert np.abs(rm - h["rmfv"]).max() < 1e-14


def test_invalid_rotation_is_flagged(oracle):
    cfg = oracle.arm_config("r_arm")
    M = np.eye(4)[None].copy()
    M[0, 0, 0] = -1.0  # det < 0: scipy's from_matrix raises ValueError
    M[0, :3, 3] = [0.3, -0.2, -0.3]
    reach, itv, state, joints, _ = oracle.symik_batch(cfg, M)
    assert not reach[0] and state[0] == 9 and np.isnan(joints).all()
    with pytest.raises(ValueError):
        oracle.euler_xyz_from_matrix(M[0, :3, :3])


@pytest.mark.parametrize("arm", ARMS)
def test_reference_example_matrices(oracle, arm):
    """The goal matrices printed in the reference's examples (src/example/test_continuous_ik.py:345-370,
    test_go_to.py:250-257; truncated decimals, so scipy projects them) through SymbolicIK, ControlIK discrete and
    ControlIK continuous: tests/golden/ctl_examples.npz."""
    g = load("ctl_examples.npz")
    u = load("symik_urdf.npz")
    M = g[f"{arm}_M"]
    reach, itv, state, joints, elbow = oracle.symik_batch(oracle.arm_config(arm), g[f"{arm}_goal_pose"])
    assert np.array_equal(state, g[f"{arm}_sym_state"]) and np.array_equal(reach, g[f"{arm}_sym_reachable"])
    np.testing.assert_allclose(itv, g[f"{arm}_sym_interval"], atol=1e-9, equal_nan=True)
    np.testing.assert_allclose(joints, g[f"{arm}_sym_joints"], atol=1e-9, equal_nan=True)
    cfg = _urdf_cfg(oracle, u, arm)
    par = oracle.ControlParams(arm=arm)
    j, r, s, e = oracle.ctl_discrete_batch(cfg, par, M)
    assert np.array_equal(s, g[f"{arm}_dis_state"]) and np.array_equal(r, g[f"{arm}_dis_reachable"])
    np.testing.assert_allclose(j, g[f"{arm}_dis_joints"], atol=1e-9)
    W = g[f"{arm}_con_joints"].shape[1]
    cj, cr, cs, st = oracle.ctl_continuous_batch(cfg, par, np.repeat(M[:, None], W, axis=1))
    assert np.array_equal(cs, g[f"{arm}_con_state"]) and np.array_equal(cr, g[f"{arm}_con_reachable"])
    np.testing.assert_allclose(cj, g[f"{arm}_con_joints"], atol=1e-9)
    assert np.array_equal(st["emergency_stop"].astype(bool), g[f"{arm}_con_emergency"])


def test_task_space_sweep(oracle, tmp_path):
    """The reference's task_space_test sweep (src/benchmark/ik_comparison.py:137-181): the grid builder reproduces its
    37 376 goal poses, and the oracle reproduces the reference's flags / states on them (tests/golden/task_space.npz)."""
    from reachy2_symbolic_ik_b200 import workspace

    g = load("task_space.npz")
    poses = workspace.task_space_grid([0.0, -0.2, 0.0])
    assert len(poses) == int(g["n_poses"]) == 37376
    # spot-check the loop order of the reference: position-major, then roll, pitch, yaw
    np.testing.assert_allclose(poses[0, 1], [0, 0, 0]); np.testing.assert_allclose(poses[1, 1], [0, 0, np.radians(45)])
    np.testing.assert_allclose(poses[8, 1], [0, np.radians(45), 0]); assert np.array_equal(poses[0, 0], poses[511, 0])
    want = np.unpackbits(g["reachable_packed"])[: len(poses)].astype(bool)
    reach, itv, state, joints, elbow = oracle.symik_batch(oracle.arm_config("r_arm"), poses)
    assert np.array_equal(state, g["state"]) and np.array_equal(reach, want)
    assert int(reach.sum()) == int(g["reachable_count"]) == 13492
    # export / import of a count volume
    counts = np.arange(24, dtype=np.uint32).reshape(2, 3, 4)
    f = str(tmp_path / "map.npz")
    workspace.save_reach_map(f, counts, [0.1, 0.2, 0.3], [0.01] * 3, np.zeros((8, 3)), arm="r_arm")
    d = workspace.load_reach_map(f)
    assert np.array_equal(d["counts"], counts) and d["arm"] == "r_arm" and d["fraction"].max() == 23 / 8


@pytest.mark.parametrize("arm", ["r_arm", "l_arm"])
def test_legacy_continuous_theta_policy(oracle, arm):
    """reachy2_symbolic_ik_b200.legacy.get_best_continuous_theta / tend_to_preferred_theta (the reference's first
    continuous policy, utils.py:130-217 / :115-127, still imported by its example scripts) against the reference's own
    flag, theta and debug text; the elbow callback here is the oracle's get_elbow_position (on the GPU box it is
    SymbolicIK.get_elbow_position, tests/test_gpu_api_r2.py)."""
    from reachy2_symbolic_ik_b200 import legacy

    g = load("legacy_theta.npz")
    rows, texts = g[f"{arm}_rows"], g[f"{arm}_text"]
    cfg = oracle.arm_config(arm)
    n_text = 0
    for row, want_text in zip(rows, texts):
        pose, interval, prev, d, pref = row[:6], row[6:8], row[8], row[9], row[10]
        elbow = lambda th: np.append(oracle.elbow_positions_batch(cfg, pose[None, :], np.array([[th]]))[0, 0], 1.0)  # noqa: E731
        flag, theta, text = legacy.get_best_continuous_theta(prev, interval, elbow, d, pref, arm, *g[f"{arm}_singularity"],
                                                             g[f"{arm}_elbow_singularity_position"])
        assert bool(flag) == bool(row[11]) and theta == row[12], (row, flag, theta)
        n_text += text == str(want_text)
        t_flag, t_theta = legacy.tend_to_preferred_theta(prev, interval, None, d, pref)
        assert bool(t_flag) == bool(row[13]) and t_theta == row[14]
    assert n_text == len(rows), f"{len(rows) - n_text} debug texts differ from the reference's"
    # every branch of the policy is in the fixture
    last = {str(t).split("\n")[-1].rstrip("TrueFalse") for t in texts}
    assert len(last) >= 5, last
