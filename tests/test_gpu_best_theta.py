"""GPU tier of the batched get_best_theta_to_current_joints (r2ik_symik_best_theta_f64,
SymbolicIK.get_best_theta_to_current_joints_batch): held to the host build of its item function and to the CPU oracle's
search by the rule of tests/best_theta_util.py, its joints bit-identical to the one-angle solve at the returned angle,
a broadcast row identical to the row repeated, MAT34 identical to MAT4, across block boundaries and through the
facade."""
import ctypes as C

import numpy as np
import pytest

import best_theta_util as B
from parity import MAX_ILL_FRACTION, TOL

pytestmark = pytest.mark.gpu
ARMS = B.ARMS


@pytest.fixture(scope="module")
def solvers():
    from reachy2_symbolic_ik_b200 import SymbolicIK

    return {arm: SymbolicIK(arm=arm) for arm in ARMS}


@pytest.fixture(scope="module")
def libs(tmp_path_factory):
    return B.build_libs(str(tmp_path_factory.mktemp("best_theta_gpu")))


def _p(t):
    return C.c_void_p(None if t is None else t.data_ptr())


def entry(sv, P, cj, no_limits=False, kind=None, pref=None):
    """The C entry on device tensors: state, theta, joints (NumPy)."""
    import torch

    from reachy2_symbolic_ik_b200 import _native
    from reachy2_symbolic_ik_b200.symbolic_ik import normalise_poses

    dev = sv._device
    if kind is None:
        P, kind, _ = normalise_poses(torch, P, dev)
    n = P.shape[0]
    cj = torch.as_tensor(np.ascontiguousarray(cj, dtype=np.float64), device=dev)
    stride = 0 if cj.dim() == 1 else 7
    state = torch.empty(n, dtype=torch.uint8, device=dev)
    theta = torch.empty(n, dtype=torch.float64, device=dev)
    joints = torch.empty((n, 7), dtype=torch.float64, device=dev)
    s = torch.cuda.current_stream(dev).cuda_stream
    rc = sv._handle.lib.r2ik_symik_best_theta_f64(sv._handle.h, kind, _p(P), C.c_int64(n), _p(cj), C.c_int32(stride),
                                                  C.c_double(B.preferred_theta(sv.arm) if pref is None else pref),
                                                  C.c_int32(int(no_limits)), _p(state), _p(theta), _p(joints), C.c_void_p(s))
    _native.check(rc, "r2ik_symik_best_theta_f64")
    return state.cpu().numpy(), theta.cpu().numpy(), joints.cpu().numpy()


def one_angle(sv, P, theta, no_limits):
    """joints of r2ik_symik_solve_f64 / r2ik_symik_no_limits_f64 at theta (NaN theta -> 0), NaN rows where theta is."""
    nan = np.isnan(theta)
    th = np.where(nan, 0.0, theta)
    if no_limits:
        j, _ = sv.is_reachable_no_limits_batch(P, th)
    else:
        j = sv.is_reachable_batch(P, theta=th).joints
    return np.where(nan[:, None], np.nan, j)


def check_all(sv, hs, orc, oracle, P, cj, no_limits, mm, name, joints_tol=True):
    got = entry(sv, P, cj, no_limits)
    want = B.oracle_best_theta(orc, oracle, sv.arm, P, cj, no_limits=no_limits)
    mm.check(f"{name} vs oracle", got, want)
    host = B.hs_best_theta(hs, sv.arm, P, cj, no_limits=no_limits)
    np.testing.assert_array_equal(got[0], host[0], err_msg=name)
    mm.check(f"{name} vs host", got, want[:1] + (host[1], host[2]) + want[3:])
    np.testing.assert_array_equal(got[2], one_angle(sv, P, got[1], no_limits), err_msg=name)
    # joints within the parity tolerance of the oracle's where the angles agree
    same = got[1] == want[1]
    if joints_tol and same.any():
        err = np.abs(got[2][same] - want[2][same]).max(axis=1)
        assert (err <= TOL).mean() >= 1 - MAX_ILL_FRACTION, f"{name}: joints off the oracle by up to {err.max():.2e}"
    return got


@pytest.mark.parametrize("arm", ARMS)
@pytest.mark.parametrize("no_limits", [False, True])
def test_100k_poses_against_host_and_oracle(solvers, libs, oracle, arm, no_limits):
    from reachy2_symbolic_ik_b200 import fk

    sv = solvers[arm]
    hs, orc = libs
    rng = np.random.default_rng(21 + no_limits)
    q = fk.sample_fk_joints(100_000, rng)
    M = fk.forward_kinematics(q, arm)
    cj = np.where(rng.random((len(q), 1)) < 0.5, q, q + rng.normal(scale=0.3, size=q.shape))
    mm = B.Mismatches(f"gpu {arm} no_limits={no_limits}")
    st, th, j = check_all(sv, hs, orc, oracle, M, cj, no_limits, mm, "fk 100k")
    # the shortcut: current joints at the preferred angle's joints, and 1e-4 of 0.01 either side
    j_pref = one_angle(sv, M, np.where(st == 0, B.preferred_theta(arm), np.nan), no_limits)
    ok = st == 0
    exact, below, above = B.near_shortcut(j_pref[ok], rng)
    for cjs, hit in ((exact, True), (below, True), (above, False)):
        g = check_all(sv, hs, orc, oracle, M[ok], cjs, no_limits, mm, f"shortcut hit={hit}")
        assert ((g[1] == B.preferred_theta(arm)) == hit).all()
    print(mm.report())


@pytest.mark.parametrize("arm", ARMS)
def test_edge_families(solvers, libs, oracle, arm):
    sv = solvers[arm]
    hs, orc = libs
    mm = B.Mismatches(f"gpu {arm} families")
    for layout in ("mat4", "euler"):
        for name, (P, cj) in B.families(arm, layout, n_fk=2000, seed=31).items():
            for nl in (False, True):
                # the extreme-input families are ill-conditioned by construction (tests/edge_inputs.py): states and
                # angles only
                check_all(sv, hs, orc, oracle, P, cj, nl, mm, f"{layout} {name} nl={nl}",
                          joints_tol=name in ("fk", "golden", "named"))
    print(mm.report())


@pytest.mark.parametrize("arm", ARMS)
def test_broadcast_row_and_mat34(solvers, arm):
    import torch

    from reachy2_symbolic_ik_b200 import _abi, fk

    sv = solvers[arm]
    M = fk.sample_fk_poses(20_000, arm, seed=41)
    row = fk.sample_fk_joints(1, np.random.default_rng(42))[0]
    for nl in (False, True):
        a = entry(sv, M, row, nl)
        b = entry(sv, M, np.repeat(row[None], len(M), axis=0), nl)
        for x, y in zip(a, b):
            np.testing.assert_array_equal(x, y)
        P34 = torch.as_tensor(np.ascontiguousarray(M[:, :3, :]).reshape(-1, 12), device=sv._device)
        c = entry(sv, P34, row, nl, kind=_abi.POSE_MAT34)
        for x, y in zip(a, c):
            np.testing.assert_array_equal(x, y)


@pytest.mark.parametrize("n", [0, 1, 2, 127, 128, 129, 255, 257, 1000])
def test_block_boundaries(solvers, n):
    from reachy2_symbolic_ik_b200 import fk

    sv = solvers["r_arm"]
    M = fk.sample_fk_poses(1000, "r_arm", seed=43)
    cj = fk.sample_fk_joints(1000, np.random.default_rng(44))
    full = entry(sv, M, cj)
    part = entry(sv, M[:n], cj[:n])
    for x, y in zip(part, full):
        np.testing.assert_array_equal(x, y[:n])


def test_facade(solvers):
    import torch

    from reachy2_symbolic_ik_b200 import fk

    sv = solvers["l_arm"]
    M = fk.sample_fk_poses(3000, "l_arm", seed=45)
    cj = fk.sample_fk_joints(3000, np.random.default_rng(46))
    a = sv.get_best_theta_to_current_joints_batch(M, cj)
    b = sv.get_best_theta_to_current_joints_batch(torch.as_tensor(M, device=sv._device),
                                                  torch.as_tensor(cj, device=sv._device))
    assert isinstance(a.theta, np.ndarray) and b.theta.is_cuda
    assert a.joints.shape == (3000, 7) and a.reachable.dtype == bool
    for f in a._fields:
        np.testing.assert_array_equal(getattr(a, f), getattr(b, f).cpu().numpy(), err_msg=f)
    want = entry(sv, M, cj)
    np.testing.assert_array_equal(a.state, want[0])
    np.testing.assert_array_equal(a.theta, want[1])
    np.testing.assert_array_equal(a.joints, want[2])
    np.testing.assert_array_equal(a.reachable, sv.is_reachable_batch(M).reachable)
    # the default preferred angle is ControlIK's; a (7,) row broadcasts; no joints on request
    c = sv.get_best_theta_to_current_joints_batch(M, cj[0], preferred_theta=B.preferred_theta("l_arm"), want_joints=False,
                                                  no_limits=True)
    assert c.joints is None
    np.testing.assert_array_equal(c.theta, entry(sv, M, cj[0], no_limits=True)[1])
    empty = sv.get_best_theta_to_current_joints_batch(torch.empty((0, 4, 4), dtype=torch.float64, device=sv._device), cj[0])
    assert empty.theta.shape == (0,) and empty.joints.shape == (0, 7)
    with pytest.raises(ValueError):
        sv.get_best_theta_to_current_joints_batch(M, cj[:10])
