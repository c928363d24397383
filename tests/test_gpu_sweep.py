"""GPU tier of the elbow-angle sweep (r2ik_symik_sweep_f64, SymbolicIK.get_joints_sweep_batch): bit-identical to the
one-angle batched solve (r2ik_symik_solve_f64 / r2ik_symik_no_limits_f64) on the pose repeated K times, across tile
boundaries, through the facade, and within the parity tolerances of the CPU oracle."""
import ctypes as C

import numpy as np
import pytest

import edge_inputs as E
from parity import Report, ill_conditioned_mask, load

pytestmark = pytest.mark.gpu
ARMS = ("r_arm", "l_arm")


@pytest.fixture(scope="module")
def solvers():
    from reachy2_symbolic_ik_b200 import SymbolicIK

    return {arm: SymbolicIK(arm=arm) for arm in ARMS}


def _p(t):
    return C.c_void_p(None if t is None else t.data_ptr())


def sweep(sv, P, K, thetas=None, no_limits=False, kind=None):
    """The C entry on device tensors: state, interval, thetas_used, joints, elbow, projected."""
    import torch

    from reachy2_symbolic_ik_b200.symbolic_ik import normalise_poses

    dev = sv._device
    if kind is None:
        P, kind, _ = normalise_poses(torch, P, dev)
    n = P.shape[0]
    stride = 0 if thetas is None or thetas.shape[0] == 1 else K
    state = torch.empty(n, dtype=torch.uint8, device=dev)
    itv = torch.empty((n, 2), dtype=torch.float64, device=dev)
    used = torch.empty((n, K), dtype=torch.float64, device=dev)
    j = torch.empty((n, K, 7), dtype=torch.float64, device=dev)
    e = torch.empty((n, K, 3), dtype=torch.float64, device=dev)
    proj = torch.empty((n, K), dtype=torch.uint8, device=dev)
    s = torch.cuda.current_stream(dev).cuda_stream
    rc = sv._handle.lib.r2ik_symik_sweep_f64(sv._handle.h, kind, _p(P), C.c_int64(n), _p(thetas), C.c_int32(stride),
                                             C.c_int32(K), C.c_int32(int(no_limits)), None, _p(state), _p(itv), _p(used),
                                             _p(j), _p(e), _p(proj), C.c_void_p(s))
    from reachy2_symbolic_ik_b200 import _native

    _native.check(rc, "r2ik_symik_sweep_f64")
    return tuple(x.cpu().numpy() for x in (state, itv, used, j, e, proj))


def expanded(sv, P, K, th, no_limits=False, kind=None):
    """The one-angle solve on the pose repeated K times with the flattened (N,K) angles."""
    import torch

    from reachy2_symbolic_ik_b200.symbolic_ik import normalise_poses

    dev = sv._device
    if kind is None:
        P, kind, _ = normalise_poses(torch, P, dev)
    Pe = P.repeat_interleave(K, dim=0).contiguous()
    n = Pe.shape[0]
    tf = torch.as_tensor(th, dtype=torch.float64, device=dev).reshape(-1).contiguous()
    j = torch.empty((n, 7), dtype=torch.float64, device=dev)
    e = torch.empty((n, 3), dtype=torch.float64, device=dev)
    s = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
    from reachy2_symbolic_ik_b200 import _native

    lib, h = sv._handle.lib, sv._handle.h
    if no_limits:
        _native.check(lib.r2ik_symik_no_limits_f64(h, kind, _p(Pe), _p(tf), None, C.c_int32(0), C.c_int64(n), _p(j), _p(e), None, s),
                      "r2ik_symik_no_limits_f64")
        st = itv = None
    else:
        st = torch.empty(n, dtype=torch.uint8, device=dev)
        itv = torch.empty((n, 2), dtype=torch.float64, device=dev)
        _native.check(lib.r2ik_symik_solve_f64(h, kind, _p(Pe), _p(tf), None, C.c_int64(n), None, _p(st), _p(itv), _p(j), _p(e), s),
                      "r2ik_symik_solve_f64")
        st, itv = st.cpu().numpy(), itv.cpu().numpy()
    return st, itv, j.cpu().numpy(), e.cpu().numpy()


def check_identical(sv, P, K, th_given=None, no_limits=False, name="", kind=None):
    import torch

    th = None if th_given is None else torch.as_tensor(th_given, dtype=torch.float64, device=sv._device).contiguous()
    state, itv, used, j, e, proj = sweep(sv, P, K, th, no_limits, kind)
    n = len(state)
    ok = state == 0
    angles = np.where(ok[:, None], used, 0.0)
    if th_given is not None:
        full = np.broadcast_to(np.asarray(th_given), (n, K))
        np.testing.assert_array_equal(used, np.where(ok[:, None], full, np.nan), err_msg=name)
        angles = np.array(full)
    st1, itv1, j1, e1 = expanded(sv, P, K, angles, no_limits, kind)
    if st1 is not None:
        np.testing.assert_array_equal(np.repeat(state, K), st1, err_msg=name)
        np.testing.assert_array_equal(np.repeat(itv, K, axis=0), itv1, err_msg=name)
    np.testing.assert_array_equal(j.reshape(-1, 7), j1, err_msg=name)
    np.testing.assert_array_equal(e.reshape(-1, 3), e1, err_msg=name)
    assert not proj[~ok].any(), name
    return state, itv, used, j, e, proj


@pytest.mark.parametrize("arm", ARMS)
@pytest.mark.parametrize("no_limits", [False, True])
def test_100k_poses_k16_bit_identical(solvers, arm, no_limits):
    from reachy2_symbolic_ik_b200 import fk

    sv = solvers[arm]
    M = fk.sample_fk_poses(100_000, arm, seed=5)
    rng = np.random.default_rng(6)
    for layout in ("mat4", "euler"):
        if layout == "euler":
            from scipy.spatial.transform import Rotation

            P = np.concatenate([M[:, :3, 3], Rotation.from_matrix(M[:, :3, :3]).as_euler("xyz")], axis=1)
        else:
            P = M
        check_identical(sv, P, 16, rng.uniform(-4, 4, (len(P), 16)), no_limits, f"{arm} {layout} given")
        check_identical(sv, P, 16, rng.uniform(-4, 4, (1, 16)), no_limits, f"{arm} {layout} shared row")
        check_identical(sv, P, 16, None, no_limits, f"{arm} {layout} sampled")
    # MAT34, the 3x4 top of the same matrices: the sweep of the MAT4 rows, and K1 on the expanded batch
    import torch

    from reachy2_symbolic_ik_b200 import _abi

    P34 = torch.as_tensor(np.ascontiguousarray(M[:, :3, :]).reshape(-1, 12), device=sv._device)
    got, want = sweep(sv, P34, 16, None, no_limits, _abi.POSE_MAT34), sweep(sv, M, 16, None, no_limits)
    for x, y in zip(got, want):
        np.testing.assert_array_equal(x, y, err_msg=f"{arm} mat34")
    if not no_limits:   # r2ik_symik_no_limits_f64 takes MAT4 / EULER6 rows only
        check_identical(sv, P34, 16, None, False, f"{arm} mat34 sampled", kind=_abi.POSE_MAT34)


@pytest.mark.parametrize("arm", ARMS)
def test_edge_families(solvers, arm):
    sv = solvers[arm]
    rng = np.random.default_rng(8)
    fams = dict(E.mat4_families(arm))
    fams.update(E.euler_families(arm))
    for name, P in fams.items():
        P = np.ascontiguousarray(P, dtype=np.float64)
        th = rng.uniform(-4, 4, (len(P), 5))
        th[:, -1] = E.big_thetas(len(P))
        for nl in (False, True):
            check_identical(sv, P, 5, th, nl, f"{arm} {name} nl={nl}")
        check_identical(sv, P, 9, None, False, f"{arm} {name} sampled")


@pytest.mark.parametrize("n,K", [(1, 1), (1000, 1), (129, 7), (300, 130), (3, 4096), (2, 1500), (1, 5000), (37, 1025)])
def test_tile_boundaries(solvers, n, K):
    """n and K off the tile sizes, K = 1, many angles on few poses (each pose split over several tiles)."""
    from reachy2_symbolic_ik_b200 import fk

    sv = solvers["r_arm"]
    M = fk.sample_fk_poses(n, "r_arm", seed=n + K)
    state, itv, used, j, e, proj = check_identical(sv, M, K, None, False, f"n={n} K={K}")
    rng = np.random.default_rng(K)
    check_identical(sv, M, K, rng.uniform(-4, 4, (n, K)), False, f"n={n} K={K} given")
    ok = state == 0
    assert np.isfinite(j[ok]).all()


def test_empty_batch(solvers):
    import torch

    sv = solvers["r_arm"]
    out = sv.get_joints_sweep_batch(torch.empty((0, 4, 4), dtype=torch.float64, device=sv._device), n_samples=8)
    assert out.joints.shape == (0, 8, 7) and out.thetas.shape == (0, 8)


def test_facade_round_trip(solvers):
    import torch

    from reachy2_symbolic_ik_b200 import fk

    sv = solvers["l_arm"]
    M = fk.sample_fk_poses(2000, "l_arm", seed=9)
    a = sv.get_joints_sweep_batch(M, n_samples=12)
    b = sv.get_joints_sweep_batch(torch.as_tensor(M, device=sv._device), n_samples=12)
    assert isinstance(a.joints, np.ndarray) and b.joints.is_cuda
    assert a.joints.shape == (2000, 12, 7) and a.elbow.shape == (2000, 12, 3) and a.projected.dtype == bool
    for f in ("reachable", "state", "theta_interval", "thetas", "joints", "elbow", "projected"):
        np.testing.assert_array_equal(getattr(a, f), getattr(b, f).cpu().numpy(), err_msg=f)
    ref = sv.is_reachable_batch(M)
    np.testing.assert_array_equal(a.reachable, ref.reachable)
    np.testing.assert_array_equal(a.theta_interval, ref.theta_interval)
    # a shared row and given angles; previous_joints only matters at the exact singularities
    row = np.linspace(-3, 3, 5)[None]
    c = sv.get_joints_sweep_batch(M, thetas=row, previous_joints=np.zeros(7))
    d = sv.get_joints_sweep_batch(M, thetas=np.repeat(row, 2000, axis=0))
    np.testing.assert_array_equal(c.joints, d.joints)
    one = sv.is_reachable_batch(M, theta=np.full(2000, row[0, 2]))
    np.testing.assert_array_equal(c.joints[:, 2], one.joints)
    nl = sv.get_joints_sweep_batch(M, thetas=row, no_limits=True)
    jn, en = sv.is_reachable_no_limits_batch(M, np.full(2000, row[0, 3]))
    np.testing.assert_array_equal(nl.joints[:, 3], jn)
    with pytest.raises(ValueError):
        sv.get_joints_sweep_batch(M, thetas=row, n_samples=5)
    with pytest.raises(ValueError):
        sv.get_joints_sweep_batch(M)
    with pytest.raises(ValueError):
        sv.get_joints_sweep_batch(M, thetas=np.zeros((3, 5)))


@pytest.mark.parametrize("arm", ARMS)
def test_oracle_agreement(solvers, oracle, arm):
    """The sweep against the CPU oracle's symik_batch on the expanded batch, parity tolerances, with the
    ill-conditioned classification of the other parity tests."""
    g = load(f"symik_random_{arm}.npz")
    P = g["M"][:1500]
    K = 6
    sv = solvers[arm]
    out = sv.get_joints_sweep_batch(P, n_samples=K)
    ok = out.reachable
    th = np.where(ok[:, None], out.thetas, 0.0).reshape(-1)
    Pe = np.repeat(P, K, axis=0)
    ocfg = oracle.arm_config(arm)
    want = oracle.symik_batch(ocfg, Pe, th)
    ill = ill_conditioned_mask(lambda p: oracle.symik_batch(ocfg, p.reshape(Pe.shape), th)[:4], Pe.reshape(len(Pe), -1))
    rep = Report(f"sweep vs oracle {arm}", len(Pe), ill)
    rep.exact("reachable", np.repeat(ok, K), want[0])
    rep.exact("state", np.repeat(out.state, K), want[2])
    rep.close("interval", np.repeat(out.theta_interval, K, axis=0), want[1])
    rep.close("joints", out.joints.reshape(-1, 7), want[3])
    rep.close("elbow", out.elbow.reshape(-1, 3), want[4])
    rep.check()
