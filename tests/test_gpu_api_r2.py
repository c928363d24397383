"""GPU tests of the scalar call sequence (get_elbow_position / get_joints return shapes, is_reachable_no_limits),
the lean host record, the one-process multi-GPU entry and the host-pipeline input handling, through the facade ->
ctypes -> C ABI, against the reference-generated fixtures (tests/golden/symik_elbow.npz, ctl_ctor.npz) and the oracle."""
import ctypes as C

import numpy as np
import pytest

from parity import Report, ill_conditioned_mask, load

pytestmark = pytest.mark.gpu
ARMS = ("r_arm", "l_arm")


@pytest.fixture(scope="module")
def solvers():
    from reachy2_symbolic_ik_b200 import SymbolicIK

    return {arm: SymbolicIK(arm=arm) for arm in ARMS}


@pytest.mark.parametrize("arm", ARMS)
def test_elbow_positions_entry(solvers, oracle, arm):
    """r2ik_elbow_positions_f64 (both modes) and r2ik_symik_no_limits_f64 with previous_joints against the reference's
    get_elbow_position / get_joints values (symbolic_ik.py:684-695, :85-119, :697-863) and the oracle's projection flag."""
    g = load("symik_elbow.npz")
    ik = solvers[arm]
    cfg = oracle.arm_config(arm)
    P = g[f"{arm}_goal_pose"]
    n, K = g[f"{arm}_thetas"].shape
    th, nth = g[f"{arm}_thetas"], g[f"{arm}_nl_thetas"]
    run = lambda p: (oracle.symik_batch(cfg, p.reshape(P.shape))[0], oracle.elbow_positions_batch(cfg, p.reshape(P.shape), th),  # noqa: E731
                     oracle.elbow_positions_batch(cfg, p.reshape(P.shape), nth, no_limits=True))
    ill = ill_conditioned_mask(run, P.reshape(n, 6))
    rep = Report(f"gpu elbow {arm}", n, ill)
    reach = g[f"{arm}_reachable"]
    has_circle = reach | (g[f"{arm}_state"] == 4)
    E, proj = ik.get_elbow_position_batch(P, th, with_projected=True)
    rep.exact("circle stored (NaN rows otherwise)", np.isfinite(E).all(axis=(1, 2)), has_circle)
    rep.close("get_elbow_position after is_reachable", E, g[f"{arm}_elbow_position"][:, :, :3])
    rep.exact("elbow shape of get_joints (3 <=> projection fired)", np.where(reach[:, None], np.where(proj, 3, 4), 0),
              g[f"{arm}_gj_elbow_len"])
    Enl, proj_nl = ik.get_elbow_position_batch(P, nth, no_limits=True, with_projected=True)
    rep.close("get_elbow_position after is_reachable_no_limits", Enl, g[f"{arm}_nl_elbow_position"][:, :, :3])
    rep.exact("elbow shape of get_joints after no_limits", np.where(proj_nl, 3, 4), g[f"{arm}_nl_elbow_len"])
    _, oproj = oracle.elbow_positions_batch(cfg, P, th, with_projected=True)
    rep.exact("projection flag vs oracle", proj & reach[:, None], oproj & reach[:, None])
    for k in range(K):
        j, e, pr = ik.is_reachable_no_limits_batch(P, nth[:, k], g[f"{arm}_nl_prev"], with_projected=True)
        rep.close(f"no_limits get_joints(theta[{k}], previous_joints)", j, g[f"{arm}_nl_joints"][:, k])
        rep.close(f"no_limits elbow of get_joints(theta[{k}])", e, g[f"{arm}_nl_elbow"][:, k])
        rep.exact(f"no_limits projected[{k}]", pr, proj_nl[:, k])
    j7, e7 = ik.is_reachable_no_limits_batch(P, nth[:, 0], g[f"{arm}_nl_prev"][0])      # one vector, broadcast
    jn, en = ik.is_reachable_no_limits_batch(P, nth[:, 0])
    assert np.array_equal(j7, jn, equal_nan=True)       # previous_joints only matter at exact singularities
    rep.check(max_ill_fraction=0.03)


@pytest.mark.parametrize("arm", ARMS)
def test_scalar_call_sequence(oracle, arm):
    """The reference's scalar API on the facade: values, the (4,) / (3,) elbow of get_joints (symbolic_ik.py:694-695,
    :714, :863), get_elbow_position after is_reachable AND after is_reachable_no_limits, the goal_pose / wrist_position
    attributes the calls leave behind."""
    from reachy2_symbolic_ik_b200 import SymbolicIK

    g = load("symik_elbow.npz")
    ik = SymbolicIK(arm=arm)
    cfg = oracle.arm_config(arm)
    P = g[f"{arm}_goal_pose"]
    nf = int(g["n_fk"])                                   # FK-sampled poses first, then task space, then the 24 named poses
    idx = np.r_[0:60, nf:nf + 60, len(P) - 24:len(P)]
    singular = len(P) - 24 + 10                           # the fully stretched arm (see test_named_poses)
    tol = 1e-9
    n_proj = n_plain = 0
    for i in idx[idx != singular]:
        ok, itv, fn, state = ik.is_reachable(P[i])
        assert ok == bool(g[f"{arm}_reachable"][i])
        o = oracle.symik_scalar(cfg, P[i])
        assert state == oracle.STATE_STRINGS[o["state"]]
        if not np.isnan(g[f"{arm}_ir_goal"][i, 0]):
            np.testing.assert_allclose(ik.goal_pose[0], g[f"{arm}_ir_goal"][i], atol=tol)
            np.testing.assert_allclose(ik.wrist_position, g[f"{arm}_ir_wrist"][i], atol=tol)
        if g[f"{arm}_state"][i] in (0, 4):
            for k in (0, 3):
                e = ik.get_elbow_position(g[f"{arm}_thetas"][i, k])
                assert e.shape == (4,) and e[3] == 1.0
                np.testing.assert_allclose(e, g[f"{arm}_elbow_position"][i, k], atol=tol)
        if ok:
            assert fn is not None and len(itv) == 2
            for k in (0, 1, 3):
                ik.is_reachable(P[i])
                j, e = fn(g[f"{arm}_thetas"][i, k])
                np.testing.assert_allclose(j, g[f"{arm}_gj_joints"][i, k], atol=tol)
                assert len(e) == g[f"{arm}_gj_elbow_len"][i, k]
                np.testing.assert_allclose(e[:3], g[f"{arm}_gj_elbow"][i, k], atol=tol)
                np.testing.assert_allclose(ik.goal_pose[0], g[f"{arm}_gj_goal"][i, k], atol=tol)
                np.testing.assert_allclose(ik.wrist_position, g[f"{arm}_gj_wrist"][i, k], atol=tol)
                np.testing.assert_array_equal(ik.elbow_position, e)
                n_proj += len(e) == 3
                n_plain += len(e) == 4
        else:
            assert fn is None and len(itv) == 0
        ok, itv, fn = ik.is_reachable_no_limits(P[i])
        assert ok and np.all(itv == [-np.pi, np.pi])
        for k in (0, 3):
            e = ik.get_elbow_position(g[f"{arm}_nl_thetas"][i, k])
            np.testing.assert_allclose(e, g[f"{arm}_nl_elbow_position"][i, k], atol=tol)
            j, e = fn(g[f"{arm}_nl_thetas"][i, k], list(g[f"{arm}_nl_prev"][i]))
            np.testing.assert_allclose(j, g[f"{arm}_nl_joints"][i, k], atol=tol)
            assert len(e) == g[f"{arm}_nl_elbow_len"][i, k]
            np.testing.assert_allclose(e[:3], g[f"{arm}_nl_elbow"][i, k], atol=tol)
    assert n_proj > 20 and n_plain > 20


def test_scalar_entry_device_memory(solvers, oracle):
    """r2ik_symik_scalar_f64 writing a record in DEVICE memory (the facade uses mapped pinned memory)."""
    import torch

    from reachy2_symbolic_ik_b200 import _abi, _native

    ik = solvers["r_arm"]
    q = _abi.ScalarQuery()
    pose = [0.55, -0.3, -0.15, 0.0, -np.pi / 2, 0.0]
    q.goal_pose[:] = pose
    q.has_theta, q.theta = 1, 0.3
    rec = torch.zeros(_abi.SCALAR_RESULT_DTYPE.itemsize, dtype=torch.uint8, device="cuda")
    _native.check(ik._handle.lib.r2ik_symik_scalar_f64(ik._handle.h, C.byref(q), C.c_void_p(rec.data_ptr()), None), "scalar")
    r = rec.cpu().numpy().view(_abi.SCALAR_RESULT_DTYPE)[0]
    o = oracle.symik_scalar(oracle.arm_config("r_arm"), pose, theta=0.3)
    for f in ("interval", "joints", "elbow", "elbow_on_circle", "goal_position", "wrist_position"):
        np.testing.assert_allclose(r[f], o[f], atol=1e-9)
    assert (r["reachable"], r["state"], r["projected"]) == (o["reachable"], o["state"], o["projected"])


@pytest.mark.parametrize("arm", ARMS)
def test_lean_host_record(solvers, arm):
    """is_reachable_batch_host with the reference's own input format (N,6) and want=LEAN (state + joints, 57 B / pose):
    the same bytes the full record carries, nothing else touched."""
    import torch

    g = load(f"symik_random_{arm}.npz")
    ik = solvers[arm]
    gp = torch.from_numpy(np.ascontiguousarray(g["goal_pose"].reshape(-1, 6))).pin_memory()
    full = ik.is_reachable_batch_host(gp, chunk=1000)
    lean = ik.is_reachable_batch_host(gp, chunk=700, want=ik.LEAN)
    assert lean.reachable is None and lean.theta_interval is None and lean.elbow is None
    assert torch.equal(lean.state, full.state)
    assert torch.equal(lean.joints.nan_to_num(), full.joints.nan_to_num())
    assert np.array_equal(lean.state.numpy() == 0, g["reachable"])
    np.testing.assert_allclose(lean.joints.numpy(), g["joints"], atol=1e-9, equal_nan=True)
    with pytest.raises(ValueError, match="unknown output fields"):
        ik.is_reachable_batch_host(gp, want=("joints", "velocity"))


@pytest.mark.parametrize("n_dev", [1, 2])
def test_one_process_multi_gpu_symik(solvers, n_dev):
    """SymbolicIK.is_reachable_batch(..., devices=[...]): one host batch, contiguous slices over the node's GPUs."""
    import torch

    if torch.cuda.device_count() < n_dev:
        pytest.skip(f"needs {n_dev} GPUs")
    from reachy2_symbolic_ik_b200 import fk

    ik = solvers["r_arm"]
    M = fk.sample_fk_poses(30_011, "r_arm", seed=77)
    one = ik.is_reachable_batch(M)
    many = ik.is_reachable_batch(M, devices=list(range(n_dev)))
    for f in ("reachable", "state", "theta_interval", "joints", "elbow"):
        assert np.array_equal(getattr(one, f), getattr(many, f), equal_nan=True), f
    lean = ik.is_reachable_batch_host(torch.from_numpy(M), want=ik.LEAN, devices=list(range(n_dev)), chunk=4096)
    assert np.array_equal(lean.joints.numpy(), one.joints, equal_nan=True)


@pytest.mark.parametrize("n_dev", [1, 2])
def test_one_process_multi_gpu_control(n_dev):
    import torch

    if torch.cuda.device_count() < n_dev:
        pytest.skip(f"needs {n_dev} GPUs")
    from reachy2_symbolic_ik_b200 import ControlIK, fk

    ctl = ControlIK(urdf_path="../config_files/reachy2.urdf")
    M = fk.sample_fk_poses(20_003, "l_arm", seed=78)
    one = ctl.symbolic_inverse_kinematics_batch("l_arm", M, "discrete")
    many = ctl.symbolic_inverse_kinematics_batch("l_arm", M, "discrete", devices=list(range(n_dev)))
    for a, b in zip(one, many):
        assert np.array_equal(a, b, equal_nan=True)
    MT = fk.sinusoidal_trajectories(301, 64, "l_arm", seed=79)[0]
    one = ctl.symbolic_inverse_kinematics_batch("l_arm", MT, "continuous")
    many = ctl.symbolic_inverse_kinematics_batch("l_arm", MT, "continuous", devices=list(range(n_dev)))
    for a, b in zip(one[:3], many[:3]):
        assert np.array_equal(a, b, equal_nan=True)
    for f in one[3].dtype.names:
        assert np.array_equal(one[3][f], many[3][f]), f


def test_continuous_host_pipeline_input_forms():
    """symbolic_inverse_kinematics_batch_host addresses raw rows of its host buffers: float32 input and strided views are
    normalised first, malformed output buffers are rejected (they used to be read / written with the wrong pitch)."""
    import torch

    from reachy2_symbolic_ik_b200 import ControlIK, fk

    ctl = ControlIK(urdf_path="../config_files/reachy2.urdf")
    T, W = 96, 40
    big = torch.from_numpy(fk.sinusoidal_trajectories(T, 2 * W, "r_arm", seed=80)[0])
    dense = big[:, :W].contiguous()
    want = ctl.symbolic_inverse_kinematics_batch_host("r_arm", dense, "continuous", chunk=16)
    view = ctl.symbolic_inverse_kinematics_batch_host("r_arm", big[:, :W], "continuous", chunk=16)       # strided view
    for a, b in zip(want, view):
        assert torch.equal(a.nan_to_num() if a.dtype.is_floating_point else a, b.nan_to_num() if b.dtype.is_floating_point else b)
    f32 = ctl.symbolic_inverse_kinematics_batch_host("r_arm", dense.float(), "continuous", chunk=16)
    ref32 = ctl.symbolic_inverse_kinematics_batch_host("r_arm", dense.float().double(), "continuous", chunk=16)
    assert torch.equal(f32[0].nan_to_num(), ref32[0].nan_to_num())
    out = list(ctl.alloc_host_outputs("continuous", (T, W)))
    out[0] = torch.empty((T, 2 * W, 7), dtype=torch.float64)[:, :W]
    with pytest.raises(ValueError, match="contiguous CPU tensor"):
        ctl.symbolic_inverse_kinematics_batch_host("r_arm", dense, "continuous", out=tuple(out))
    with pytest.raises(ValueError, match="takes host matrices"):
        ctl.symbolic_inverse_kinematics_batch_host("r_arm", dense.cuda(), "continuous")


def test_invalid_rotation_keeps_controller_state():
    """scipy raises on a left-handed matrix before the reference touches any controller state (control_ik.py:216): after the
    ValueError the next call works and sees the state of before."""
    from reachy2_symbolic_ik_b200 import ControlIK, fk

    ctl = ControlIK(urdf_path="../config_files/reachy2.urdf")
    M = fk.sample_fk_poses(4, "r_arm", seed=81)
    j0, ok0, _ = ctl.symbolic_inverse_kinematics("r_arm", M[0], "continuous")
    before = (ctl.previous_sol["r_arm"].copy(), ctl.previous_theta["r_arm"], ctl.init, ctl.last_call_t["r_arm"])
    bad = M[1].copy()
    bad[:3, :3] = np.diag([-1.0, 1.0, 1.0])
    for mode in ("continuous", "discrete"):
        with pytest.raises(ValueError, match="Non-positive determinant"):
            ctl.symbolic_inverse_kinematics("r_arm", bad, mode)
    assert np.array_equal(ctl.previous_sol["r_arm"], before[0]) and ctl.previous_theta["r_arm"] == before[1]
    assert ctl.init == before[2] and ctl.last_call_t["r_arm"] == before[3]
    twin = ControlIK(urdf_path="../config_files/reachy2.urdf")       # the same calls without the two that raised
    twin.symbolic_inverse_kinematics("r_arm", M[0], "continuous")
    for mode in ("discrete", "continuous", "continuous"):
        j, ok, state = ctl.symbolic_inverse_kinematics("r_arm", M[2], mode)
        jt, okt, statet = twin.symbolic_inverse_kinematics("r_arm", M[2], mode)
        np.testing.assert_allclose(j, jt, atol=1e-12)
        assert (ok, state) == (okt, statet)


def test_f32_empty_batch_sets_the_escalation_count(solvers):
    res = solvers["r_arm"].is_reachable_batch(np.zeros((0, 4, 4), np.float32), precision="fp32")
    assert res.n_escalated == 0 and len(res.state) == 0


@pytest.mark.parametrize("is_dvt", [False, True])
def test_constructor_previous_theta(is_dvt):
    """ControlIK.previous_theta as the reference's constructor seeds it (control_ik.py:142-159; the ternary search over the
    two-arm joint list, SURVEY.md A.6.11) -- default and custom current_joints / current_pose (tests/golden/ctl_ctor.npz)."""
    from reachy2_symbolic_ik_b200 import ControlIK

    g = load("ctl_ctor.npz")
    tag = "dvt" if is_dvt else "std"
    ctl = ControlIK(urdf_path="../config_files/reachy2.urdf", is_dvt=is_dvt)
    for arm in ARMS:
        assert abs(ctl.previous_theta[arm] - float(g[f"{tag}_default_{arm}"])) < 1e-9
    for v in range(int(g["n_variants"])):
        ctl = ControlIK(current_joints=[list(r) for r in g[f"v{v}_current_joints"]], current_pose=list(g[f"v{v}_current_pose"]),
                        urdf_path="../config_files/reachy2.urdf", is_dvt=is_dvt)
        for arm in ARMS:
            assert abs(ctl.previous_theta[arm] - float(g[f"{tag}_v{v}_{arm}"])) < 1e-9, (v, arm)


@pytest.mark.parametrize("arm", ARMS)
@pytest.mark.parametrize("n", [1, 33, 5_000, 300_001])
def test_discrete_compacted_passes_equal_single_kernel(arm, n):
    """r2ik_ctl_discrete_compact_f64 (classify / search / finish over compacted index lists) against the one-kernel
    r2ik_ctl_discrete_f64: the same per-pose device functions on the same inputs -> identical bytes, every pose written
    exactly once (poisoned outputs), invalid rotation blocks and a wound previous solution included."""
    import torch

    from reachy2_symbolic_ik_b200 import ControlIK, fk

    ctl = ControlIK(urdf_path="../config_files/reachy2.urdf")
    M = np.concatenate([fk.sample_fk_poses(n - n // 4, arm, seed=77 + n), fk.sample_task_space_poses(n // 4, arm, seed=78 + n)]) if n > 3 \
        else fk.sample_fk_poses(n, arm, seed=77)
    rng = np.random.default_rng(n)
    if n > 1000:
        # tool axis along +-e_x: the solver's literal instantiation (flagged list entries, full re-solve in the finish pass)
        from scipy.spatial.transform import Rotation

        m = 400
        for q in range(m):
            M[q, :3, :3] = (Rotation.from_euler("y", (np.pi / 2) * (1 if q % 2 else -1)) * Rotation.from_euler("z", rng.uniform(-np.pi, np.pi))).as_matrix()
        M[:m, :3, 3] = np.array([0.38, -0.2 if arm == "r_arm" else 0.2, -0.12]) + rng.uniform(-0.12, 0.12, (m, 3))
    bad = rng.integers(0, n, size=max(1, n // 50)) if n > 1 else []
    for b in bad:
        M[b, :3, :3] = np.diag([1.0, 1.0, -1.0])           # det < 0: no rotation
    Md = torch.from_numpy(M).cuda()
    for prev in (None, np.array([0.3, -0.2, 7.0, -1.0, 0.1, 0.2, -6.5])):
        for K, mode in ((20, "unconstrained"), (360, "unconstrained"), (20, "low_elbow")):
            ctl.nb_search_points = K
            outs = {}
            for compact in (False, True):
                out = (torch.full((n, 7), 123.0, dtype=torch.float64, device="cuda"), torch.full((n,), 7, dtype=torch.uint8, device="cuda").view(torch.bool),
                       torch.full((n,), 77, dtype=torch.uint8, device="cuda"), torch.full((n,), 99, dtype=torch.uint8, device="cuda"))
                res = ctl.symbolic_inverse_kinematics_batch(arm, Md, "discrete", constrained_mode=mode, previous_joints=prev,
                                                            out=out, compact=compact)
                outs[compact] = [x.view(torch.uint8).cpu().numpy() if x.dtype == torch.bool else x.cpu().numpy() for x in res]
            for a, b in zip(outs[False], outs[True]):
                np.testing.assert_array_equal(a, b)
            assert not (outs[True][2] == 77).any() and not (outs[True][3] == 99).any()
            if n > 1000:
                assert (outs[True][2] == 9).sum() == len(set(bad)) and 0.2 < outs[True][1].mean() < 0.9


def test_discrete_compact_entry_argument_checks():
    import torch

    from reachy2_symbolic_ik_b200 import ControlIK

    ctl = ControlIK(urdf_path="../config_files/reachy2.urdf")
    solver = ctl.symbolic_ik_solver["r_arm"]
    lib = solver._handle.lib
    assert lib.r2ik_ctl_discrete_workspace_bytes(C.c_int64(1000)) == 256 + 80 * 1000
    assert lib.r2ik_ctl_discrete_workspace_bytes(C.c_int64(-1)) == -1
    par = ctl._ctl_params("r_arm", "unconstrained", -4 * np.pi / 6, 0.01)
    n = 64
    M = torch.eye(4, dtype=torch.float64, device="cuda").repeat(n, 1, 1).reshape(n, 16)
    j = torch.empty((n, 7), dtype=torch.float64, device="cuda")
    b = [torch.empty(n, dtype=torch.uint8, device="cuda") for _ in range(3)]
    prev = torch.zeros(7, dtype=torch.float64, device="cuda")
    ws = torch.empty(256 + 80 * n, dtype=torch.uint8, device="cuda")
    p = lambda t: C.c_void_p(t.data_ptr())  # noqa: E731
    call = lambda wsp, nbytes: lib.r2ik_ctl_discrete_compact_f64(solver._handle.h, C.byref(par), p(M), C.c_int64(n), p(prev), p(prev), p(j),  # noqa: E731
                                                                 p(b[0]), p(b[1]), p(b[2]), wsp, C.c_int64(nbytes), None)
    assert call(p(ws), ws.numel() - 1) != 0 and "workspace smaller" in lib.r2ik_last_error().decode()
    assert call(None, ws.numel()) != 0
    assert call(C.c_void_p(ws.data_ptr() + 8), ws.numel()) != 0 and "aligned" in lib.r2ik_last_error().decode()
    assert call(p(ws), ws.numel()) == 0
    torch.cuda.synchronize()


@pytest.mark.parametrize("arm", ARMS)
def test_legacy_continuous_theta_policy_on_the_scalar_api(arm):
    """The reference's example scripts drive get_best_continuous_theta (utils.py:130-217) with the solver's own
    get_elbow_position; here the callback is the scalar kernel.  Flag and theta as in the reference's fixture."""
    from reachy2_symbolic_ik_b200 import SymbolicIK, legacy

    g = load("legacy_theta.npz")
    rows, texts = g[f"{arm}_rows"], g[f"{arm}_text"]
    ik = SymbolicIK(arm=arm)
    np.testing.assert_allclose(ik.elbow_singularity_position, g[f"{arm}_elbow_singularity_position"], atol=1e-15)
    checked = 0
    for row, want_text in list(zip(rows, texts))[::5]:
        ok, interval, _, _ = ik.is_reachable([row[:3], row[3:6]])
        assert ok
        np.testing.assert_allclose(interval, row[6:8], atol=1e-9)
        flag, theta, text = legacy.get_best_continuous_theta(row[8], interval, ik.get_elbow_position, row[9], row[10], arm,
                                                             ik.singularity_offset, ik.singularity_limit_coeff,
                                                             ik.elbow_singularity_position)
        assert bool(flag) == bool(row[11]) and abs(theta - row[12]) < 1e-9
        assert text.split("\n")[-1] == str(want_text).split("\n")[-1]
        checked += 1
    assert checked > 80
