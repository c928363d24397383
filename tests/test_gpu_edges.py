"""Extreme inputs (tests/edge_inputs.py) through the C ABI on the GPU, against the CPU oracle, and the FP32 families that
the host harness used to be the only one to run.

FP64 entries: states, flags and NaN pattern identical to the oracle's, values within 1e-9 rad.  No pose is excused by a
conditioning test except in the `near_shoulder` family, whose wrist direction (w - s) / |w - s| below |w - s| = 1e-7 m
is not determined to 1e-9 by the rounding of w itself: those poses are reported, and their states still compared.

Where the oracle's arithmetic could part from the reference's numpy on these inputs:
  * a goal beyond ~1.3e154 m (sik:284-307): np.linalg.norm of a 3-vector is sqrt(dot(v, v)), which overflows to inf
    exactly as the oracle's norm3 does; the goal then becomes shoulder + v / inf * L = the shoulder, in both.
  * scaled rotation blocks (rxp:78-95): scipy replaces a non-orthonormal block by U @ Vt of its SVD, which does not
    depend on the block's scale.  The oracle's Newton iteration for that factor scales the block to unit size first
    (exact powers of two), so it reaches the same factor for a block scaled by 10^-100 as for one scaled by 10^100.
    Scales beyond 10^+-100 are left out: there the determinant whose sign decides validity (scipy raises for
    det <= 0) under- or overflows, and whether it does depends on how it is evaluated (numpy's LU against the closed
    form of the oracle and the kernels), not on the rotation.
"""
import ctypes as C

import numpy as np
import pytest

import edge_inputs as E
from parity import CTOR_VARIANTS, TOL_F32, Report, check_f32, load

pytestmark = pytest.mark.gpu
ARMS = ("r_arm", "l_arm")


@pytest.fixture(scope="module")
def solvers():
    from reachy2_symbolic_ik_b200 import SymbolicIK

    return {arm: SymbolicIK(arm=arm) for arm in ARMS}


def _ill(name, arm, P):
    return E.undetermined_wrist_direction(arm, P) if name == "near_shoulder" else None


def _families(arm):
    return {**E.mat4_families(arm), **E.euler_families(arm)}


@pytest.mark.parametrize("arm", ARMS)
def test_symik_solve_edges(solvers, oracle, arm):
    """r2ik_symik_solve_f64 on MAT4, MAT34 (the 3x4 top of the same matrices) and EULER6 inputs, with theta = the
    interval start and with theta = 1e3 .. 1e15 rad."""
    ik, ocfg = solvers[arm], oracle.arm_config(arm)
    for name, P in _families(arm).items():
        ill = _ill(name, arm, P)
        layouts = [("", P)] + ([("mat34", np.ascontiguousarray(P[:, :3, :]))] if P.shape[1:] == (4, 4) else [])
        want = oracle.symik_batch(ocfg, P)
        th = E.big_thetas(len(P))
        want_th = oracle.symik_batch(ocfg, P, th)
        for lay, X in layouts:
            res = ik.is_reachable_batch(X)
            rep = Report(f"gpu edges {name} {lay or P.shape[1:]} {arm}", len(P), ill)
            rep.exact("reachable", res.reachable, want[0])
            rep.exact("state", res.state, want[2])
            rep.close("interval", res.theta_interval, want[1])
            rep.close("joints", res.joints, want[3])
            rep.close("elbow", res.elbow, want[4])
            res = ik.is_reachable_batch(X, theta=th)
            rep.close("joints@big theta", res.joints, want_th[3])
            rep.close("elbow@big theta", res.elbow, want_th[4])
            rep.check(max_ill_fraction=1.0 if ill is not None else 0.0)
            assert np.array_equal(res.state, want_th[2]) and np.array_equal(ik.is_reachable_batch(X).state, want[2])


@pytest.mark.parametrize("arm", ARMS)
def test_no_limits_and_elbow_positions_edges(solvers, oracle, arm):
    """r2ik_symik_no_limits_f64 (ordinary and 1e3 .. 1e15 rad thetas) and r2ik_elbow_positions_f64 on the same
    families.  The no-limits solve does not stop at the reach pre-check, so a goal past the dg2 overflow reaches the
    solver as the projected position."""
    ik, ocfg = solvers[arm], oracle.arm_config(arm)
    rng = np.random.default_rng(3)
    for name, P in _families(arm).items():
        ill = _ill(name, arm, P)
        th = np.where(rng.random(len(P)) < 0.5, rng.uniform(-np.pi, np.pi, len(P)), E.big_thetas(len(P)))
        nj, ne = ik.is_reachable_no_limits_batch(P, th)
        wj, we = oracle.symik_no_limits_batch(ocfg, P, th)[:2]
        thk = np.stack([th, rng.uniform(-np.pi, np.pi, len(P))], axis=1)
        rep = Report(f"gpu edges no-limits / elbow {name} {arm}", len(P), ill)
        rep.close("no_limits joints", nj, wj)
        rep.close("no_limits elbow", ne, we)
        for nl in (False, True):
            got = ik.get_elbow_position_batch(P, thk, no_limits=nl)
            want = oracle.elbow_positions_batch(ocfg, P, thk, no_limits=nl)
            rep.close(f"elbow positions no_limits={nl}", got, want)
        rep.check(max_ill_fraction=1.0 if ill is not None else 0.0)


def urdf_params():
    u = load("symik_urdf.npz")
    return {k[len("param_"):]: u[k] for k in u.files if k.startswith("param_")}


@pytest.mark.parametrize("arm", ARMS)
def test_ctl_discrete_edges(oracle, arm):
    """r2ik_ctl_discrete_f64 and r2ik_ctl_discrete_compact_f64 on the matrix families (goal rotation through
    rotation_from_mat4 with the identity snap and the literal route, then the interval plan and the discrete search):
    joints, flags, states and emergency codes against the oracle's ControlIK.symbolic_inverse_kinematics."""
    from reachy2_symbolic_ik_b200 import ControlIK

    ctl = ControlIK(urdf_path="../config_files/reachy2.urdf")
    ocfg = oracle.arm_config(arm, ik_parameters=urdf_params(), singularity_offset=-1.01)
    opar = oracle.ControlParams(arm=arm)
    for name, P in E.mat4_families(arm).items():
        ill = _ill(name, arm, P)
        wj, wr, ws, we = oracle.ctl_discrete_batch(ocfg, opar, P)
        rep = Report(f"gpu edges ctl discrete {name} {arm}", len(P), ill)
        for compact in (False, True):
            joints, reach, state, emg = ctl.symbolic_inverse_kinematics_batch(arm, P, "discrete", compact=compact)
            tag = " compact" if compact else ""
            rep.exact(f"reachable{tag}", reach, wr)
            rep.exact(f"state{tag}", state, ws)
            rep.exact(f"emergency{tag}", emg, we)
            rep.close(f"joints{tag}", joints, wj)
            assert np.array_equal(np.asarray(state), ws)
        rep.check(max_ill_fraction=1.0 if ill is not None else 0.0)


@pytest.mark.parametrize("arm", ARMS)
def test_scalar_entry_edges(solvers, oracle, arm):
    """r2ik_symik_scalar_f64 (one launch per call, EULER6 goal) on a seeded subsample of the euler families -- goals at
    10^-300 .. 10^200 m, angles of 1e3 .. 1e15 rad -- with and without limits, theta = the interval start or 1e3 ..
    1e15 rad: every field of the record against the oracle's scalar call sequence (positions relative to their size)."""
    import torch

    from reachy2_symbolic_ik_b200 import _abi, _native

    ik, ocfg = solvers[arm], oracle.arm_config(arm)
    rng = np.random.default_rng(11)
    fams = E.euler_families(arm)
    P = np.concatenate([fams["far_euler"][rng.choice(600, 60, replace=False)], fams["big_euler"][rng.choice(3000, 60, replace=False)]])
    thetas = E.big_thetas(len(P))
    rec = torch.zeros(_abi.SCALAR_RESULT_DTYPE.itemsize, dtype=torch.uint8, device="cuda")
    worst, n = 0.0, 0
    for i, pose in enumerate(P.reshape(-1, 6)):
        for no_limits in (0, 1):
            for theta in (None, float(thetas[i])):
                q = _abi.ScalarQuery()
                q.goal_pose[:] = pose.tolist()
                q.no_limits = no_limits
                q.has_theta, q.theta = (0, 0.0) if theta is None else (1, theta)
                _native.check(ik._handle.lib.r2ik_symik_scalar_f64(ik._handle.h, C.byref(q), C.c_void_p(rec.data_ptr()), None), "scalar")
                r = rec.cpu().numpy().view(_abi.SCALAR_RESULT_DTYPE)[0]
                o = oracle.symik_scalar(ocfg, pose, no_limits=bool(no_limits), theta=theta)
                what = f"pose {i} no_limits={no_limits} theta={theta}"
                assert (r["reachable"], r["state"], r["projected"]) == (o["reachable"], o["state"], o["projected"]), what
                for f in ("interval", "joints", "elbow", "elbow_on_circle", "goal_position_solved", "wrist_position_solved",
                          "goal_position", "wrist_position"):
                    a, b = np.asarray(r[f], np.float64), np.asarray(o[f], np.float64)
                    assert np.array_equal(np.isnan(a), np.isnan(b)), f"{what}: {f} NaN pattern"
                    ok = ~np.isnan(b)
                    e = float(np.max(np.abs(a[ok] - b[ok]) / np.maximum(1.0, np.abs(b[ok])), initial=0.0))
                    worst = max(worst, e)
                    assert e <= 1e-9, f"{what}: {f} {a} vs {b}"
                n += 1
    print(f"[gpu edges scalar entry {arm}] {n} calls, worst |err| / max(1, |value|) {worst:.3e}")


@pytest.mark.parametrize("arm", ARMS)
def test_edges_mixed_with_ordinary_poses(solvers, arm):
    """Extreme poses interleaved with ordinary ones leave the ordinary poses' results bit-identical to a batch of the
    ordinary poses alone (no state leaks between threads, warps or the literal re-solve of a neighbour)."""
    from reachy2_symbolic_ik_b200 import fk

    ik = solvers[arm]
    plain = np.concatenate([fk.sample_fk_poses(3000, arm, seed=41), fk.sample_task_space_poses(1000, arm, seed=42)])
    edge = np.concatenate([P for P in E.mat4_families(arm).values()])
    rng = np.random.default_rng(43)
    mixed = np.concatenate([plain, edge])
    order = rng.permutation(len(mixed))
    where = np.argsort(order)[: len(plain)]           # positions of the ordinary poses in the mixed batch
    alone = ik.is_reachable_batch(plain)
    both = ik.is_reachable_batch(mixed[order])
    for f in ("reachable", "state", "theta_interval", "joints", "elbow"):
        np.testing.assert_array_equal(getattr(both, f)[where], getattr(alone, f), err_msg=f)


# ------------------------------------------------------------------------------------------------------ FP32 families
@pytest.mark.parametrize("arm", ARMS)
def test_fp32_stretched_arm_boundary(solvers, oracle, arm):
    """Elbow pitch 1e-6 .. 2e-3 rad: the wrist within ~1e-7 m of the range sphere, where the FP32 wrist centre cannot
    decide "wrist out of range" and the FP64 re-solve must: states identical to the oracle's."""
    from reachy2_symbolic_ik_b200 import fk

    rng = np.random.default_rng(5)
    q = fk.sample_fk_joints(150_000, rng)
    q[:, 3] = -10.0 ** rng.uniform(-6, -2.7, len(q))
    M = fk.forward_kinematics(q, arm)
    P32 = M[M[:, 0, 3] > 0.1].astype(np.float32)
    want = oracle.symik_batch(oracle.arm_config(arm), P32.astype(np.float64))
    assert 0.05 < (want[2] == 3).mean() < 0.95
    res = solvers[arm].is_reachable_batch(P32, precision="fp32")
    print(f"[gpu f32 stretched arm {arm}] n={len(P32)}, out of range {int((want[2] == 3).sum())}, "
          f"escalated to FP64 {res.n_escalated}")
    assert np.array_equal(res.state, want[2]) and np.array_equal(res.reachable, want[0])


@pytest.mark.parametrize("arm", ARMS)
@pytest.mark.parametrize("variant", sorted(CTOR_VARIANTS))
def test_fp32_constructor_variants(oracle, arm, variant):
    from reachy2_symbolic_ik_b200 import SymbolicIK

    P32 = load("symik_ctor.npz")[f"{arm}_M"].astype(np.float32)
    res = SymbolicIK(arm=arm, **CTOR_VARIANTS[variant]).is_reachable_batch(P32, precision="fp32")
    esc = np.zeros(len(P32), bool); esc[:res.n_escalated] = True
    check_f32(f"gpu f32 ctor {variant} {arm}", oracle, arm, P32, (res.reachable, res.theta_interval, res.state, res.joints,
                                                                  res.elbow, esc), ocfg=oracle.arm_config(arm, **CTOR_VARIANTS[variant]))


def _check_f32_all_escalated(name, oracle, arm, P32, res, must_escalate):
    """A family the FP32 kernel hands to the FP64 solver by design: states identical and every pose within TOL_F32
    (instead of check_f32's cap on the re-solved share), and at least the poses of `must_escalate` re-solved."""
    want = oracle.symik_batch(oracle.arm_config(arm), P32.astype(np.float64))
    rep = Report(name, len(P32))
    rep.exact("state", res.state, want[2])
    rep.exact("reachable", res.reachable, want[0])
    rep.close("interval", res.theta_interval, want[1], tol=TOL_F32)
    rep.close("joints", res.joints, want[3], tol=TOL_F32)
    rep.close("elbow", res.elbow, want[4], tol=TOL_F32)
    rep.lines.append(f"escalated to FP64: {res.n_escalated}, of which required {int(must_escalate.sum())}")
    rep.check()
    assert res.n_escalated >= int(must_escalate.sum()), rep.summary()


@pytest.mark.parametrize("arm", ARMS)
def test_fp32_big_euler_and_non_orthonormal(solvers, oracle, arm):
    """Euler angles far outside [-pi, pi] and non-orthonormal blocks.  The golden big-euler poses and the
    float32-rounded blocks are held to check_f32.  Two families lie outside what the FP32 kernel solves itself and must
    be re-solved in FP64: euler angles of 1e3 .. 1e15 rad (|angle| > 64, R2IK_ESC 3) and blocks printed with 5 digits
    (Gram matrix off the identity by more than 2e-6, R2IK_ESC 2)."""
    fams = E.mat4_families(arm)
    for name, P in {"big euler golden": load("symik_big_euler.npz")[f"{arm}_goal_pose"], "float32": fams["float32"]}.items():
        P32 = P.astype(np.float32)
        res = solvers[arm].is_reachable_batch(P32, precision="fp32")
        esc = np.zeros(len(P32), bool); esc[:res.n_escalated] = True
        check_f32(f"gpu f32 {name} {arm}", oracle, arm, P32, (res.reachable, res.theta_interval, res.state, res.joints,
                                                              res.elbow, esc))
    P32 = E.euler_families(arm)["big_euler"].astype(np.float32)
    _check_f32_all_escalated(f"gpu f32 big euler 1e3..1e15 {arm}", oracle, arm, P32,
                             solvers[arm].is_reachable_batch(P32, precision="fp32"), (np.abs(P32[:, 1]) > 64).any(axis=1))
    P32 = fams["five_digits"].astype(np.float32)
    R = P32[:, :3, :3].astype(np.float64)
    gram_off = np.abs(R @ R.transpose(0, 2, 1) - np.eye(3)).max(axis=(1, 2)) > 1e-5
    _check_f32_all_escalated(f"gpu f32 five digits {arm}", oracle, arm, P32,
                             solvers[arm].is_reachable_batch(P32, precision="fp32"), gram_off)


@pytest.mark.parametrize("arm", ARMS)
def test_fp32_vs_oracle_3m(solvers, oracle, arm):
    """2 M FK samples and 1 M task-space poses per arm, seeded."""
    from reachy2_symbolic_ik_b200 import fk

    seed = 51 if arm == "r_arm" else 52
    P32 = np.concatenate([fk.sample_fk_poses(2_000_000, arm, seed=seed),
                          fk.sample_task_space_poses(1_000_000, arm, seed=seed + 100)]).astype(np.float32)
    res = solvers[arm].is_reachable_batch(P32, precision="fp32")
    esc = np.zeros(len(P32), bool); esc[:res.n_escalated] = True
    check_f32(f"gpu f32 vs oracle 3M {arm}", oracle, arm, P32, (res.reachable, res.theta_interval, res.state, res.joints,
                                                                res.elbow, esc))
