"""The elbow-angle sweep (r2ik_symik_sweep_f64) on the host: tests/hostsim/sweep.cpp runs the sweep with the item
functions of k_symik_sweep (one solve per pose, then K samples) and this file holds it bit for bit to the one-angle
batched solve of the host harness (tests/hostsim/hostsim.cpp) on the pose repeated K times, to numpy's linspace for
the sampled angles, and to forward kinematics.  The argument checks of the C entry are exercised on libr2ik.so without
a device."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import edge_inputs as E
from parity import REPO, load
from reachy2_symbolic_ik_b200 import _abi

HS_DIR = os.path.join(REPO, "tests", "hostsim")
ARMS = ("r_arm", "l_arm")


@pytest.fixture(scope="module")
def hs():
    subprocess.run(["make", "-C", HS_DIR], check=True, capture_output=True)
    return C.CDLL(os.path.join(HS_DIR, "_build", "libr2ik_hostsim.so"))


@pytest.fixture(scope="module")
def sw(tmp_path_factory):
    """tests/hostsim/sweep.cpp built with the harness's flags (tests/hostsim/Makefile) into a temporary directory."""
    out = str(tmp_path_factory.mktemp("hostsim_sweep") / "libr2ik_hostsim_sweep.so")
    subprocess.run(["g++", "-O2", "-fPIC", "-std=c++17", "-ffp-contract=off", "-Wall", "-Wno-unknown-pragmas", "-shared",
                    "-o", out, os.path.join(HS_DIR, "sweep.cpp"), "-lm"], check=True, capture_output=True)
    return C.CDLL(out)


def dp(a):
    return None if a is None else a.ctypes.data_as(C.POINTER(C.c_double))


def u8(a):
    return a.ctypes.data_as(C.POINTER(C.c_uint8))


def cfg_for(arm, singularity_offset=0.03):
    return _abi.make_arm_config(arm, _abi.DEFAULT_IK_PARAMETERS, 127, 42.5, 1e-8, 0.02, 1e-7, singularity_offset, 1.0)


def kind_of(P):
    return _abi.POSE_MAT4 if P.shape[1:] == (4, 4) else _abi.POSE_EULER6


def hs_sweep(sw, cfg, P, K, thetas=None, no_limits=False):
    """hs_symik_sweep; thetas (N,K) or (1,K) or None (sampled).  Returns state, interval, thetas_used, joints, elbow,
    projected."""
    P = np.ascontiguousarray(P, dtype=np.float64)
    n = len(P)
    th, stride = None, 0
    if thetas is not None:
        th = np.ascontiguousarray(thetas, dtype=np.float64)
        stride = K if th.shape[0] == n and n != 1 else 0
    state = np.zeros(n, np.uint8); itv = np.empty((n, 2)); used = np.empty((n, K))
    j = np.empty((n, K, 7)); e = np.empty((n, K, 3)); proj = np.zeros((n, K), np.uint8)
    sw.hs_symik_sweep(C.byref(cfg), kind_of(P), dp(P), C.c_int64(n), dp(th), C.c_int(stride), C.c_int(K), C.c_int(int(no_limits)),
                      None, u8(state), dp(itv), dp(used), dp(j), dp(e), u8(proj))
    return state, itv, used, j, e, proj.astype(bool)


def hs_symik(hs, cfg, P, theta):
    P = np.ascontiguousarray(P, dtype=np.float64)
    n = len(P)
    reach = np.zeros(n, np.uint8); state = np.zeros(n, np.uint8)
    itv = np.empty((n, 2)); j = np.empty((n, 7)); e = np.empty((n, 3))
    th = np.ascontiguousarray(theta, dtype=np.float64)
    hs.hs_symik_batch(C.byref(cfg), kind_of(P), dp(P), dp(th), C.c_int64(n), u8(reach), u8(state), dp(itv), dp(j), dp(e))
    return state, itv, j, e


def hs_no_limits(hs, cfg, P, theta):
    P = np.ascontiguousarray(P, dtype=np.float64)
    n = len(P)
    j = np.empty((n, 7)); e = np.empty((n, 3))
    hs.hs_no_limits_batch(C.byref(cfg), kind_of(P), dp(P), dp(np.ascontiguousarray(theta, dtype=np.float64)), C.c_int64(n), dp(j), dp(e))
    return j, e


def hs_projected(hs, cfg, P, thetas, no_limits):
    """hs_elbow_positions' projection flags at (N,K) angles."""
    P = np.ascontiguousarray(P, dtype=np.float64)
    n, K = thetas.shape
    e = np.empty((n, K, 3)); proj = np.zeros((n, K), np.uint8)
    hs.hs_elbow_positions(C.byref(cfg), kind_of(P), dp(P), dp(np.ascontiguousarray(thetas)), C.c_int(K), C.c_int64(n),
                          C.c_int(int(no_limits)), dp(e), u8(proj))
    return proj.astype(bool)


def reference_samples(itv, K):
    """get_best_discrete_theta's sample angles (utils.py:366-375) for each interval, NaN rows where the interval is."""
    out = np.full((len(itv), K), np.nan)
    for r, (i0, i1) in enumerate(itv):
        if np.isnan(i0):
            continue
        if abs(abs(i0) + abs(i1) - 2 * np.pi) < 0.00001:
            out[r] = np.linspace(np.pi / 2, 5 * np.pi / 2, K)
        elif i0 < i1:
            out[r] = np.linspace(i0, i1, K)
        else:
            out[r] = np.linspace(i0, i1 + 2 * np.pi, K)
    return out


def families(arm, layout):
    from scipy.spatial.transform import Rotation

    g = load(f"symik_random_{arm}.npz")
    named = load("symik_named.npz")[f"{arm}_poses"]
    if layout == "mat4":
        M = np.tile(np.eye(4), (len(named), 1, 1))
        M[:, :3, :3] = Rotation.from_euler("xyz", named[:, 1]).as_matrix()
        M[:, :3, 3] = named[:, 0]
        fam = {"random": g["M"], "named": M}
        fam.update(E.mat4_families(arm))
    else:
        fam = {"random": g["goal_pose"], "named": named}
        fam.update(E.euler_families(arm))
    return {k: np.ascontiguousarray(v, dtype=np.float64) for k, v in fam.items()}


def expand(P, K):
    return np.repeat(P, K, axis=0)


@pytest.mark.parametrize("arm", ARMS)
@pytest.mark.parametrize("layout", ["mat4", "euler"])
@pytest.mark.parametrize("shared_row", [False, True])
def test_given_angles_match_the_one_angle_solve(hs, sw, arm, layout, shared_row):
    """Given angles, per pose or one shared row: every (pose, angle) is bit-identical to the one-angle batched solve of
    the pose repeated K times with the flattened angles."""
    cfg = cfg_for(arm)
    rng = np.random.default_rng(7 + shared_row)
    K = 5
    for name, P in families(arm, layout).items():
        n = len(P)
        th = rng.uniform(-4.0, 4.0, (1 if shared_row else n, K))
        if name in ("big_euler", "far"):
            th[:, -1] = E.big_thetas(th.shape[0])
        full = np.broadcast_to(th, (n, K))
        state, itv, used, j, e, proj = hs_sweep(sw, cfg, P, K, th)
        st1, itv1, j1, e1 = hs_symik(hs, cfg, expand(P, K), full.reshape(-1))
        np.testing.assert_array_equal(np.repeat(state, K), st1, err_msg=name)
        np.testing.assert_array_equal(np.repeat(itv, K, axis=0), itv1, err_msg=name)
        np.testing.assert_array_equal(j.reshape(-1, 7), j1, err_msg=name)
        np.testing.assert_array_equal(e.reshape(-1, 3), e1, err_msg=name)
        ok = state == 0
        np.testing.assert_array_equal(used, np.where(ok[:, None], full, np.nan), err_msg=name)
        assert not proj[~ok].any(), name
        np.testing.assert_array_equal(proj[ok], hs_projected(hs, cfg, P, np.ascontiguousarray(full), False)[ok], err_msg=name)


@pytest.mark.parametrize("arm", ARMS)
@pytest.mark.parametrize("layout", ["mat4", "euler"])
def test_no_limits_matches_the_no_limits_solve(hs, sw, arm, layout):
    cfg = cfg_for(arm)
    rng = np.random.default_rng(11)
    K = 4
    for name, P in families(arm, layout).items():
        n = len(P)
        th = rng.uniform(-4.0, 4.0, (n, K))
        state, itv, used, j, e, proj = hs_sweep(sw, cfg, P, K, th, no_limits=True)
        j1, e1 = hs_no_limits(hs, cfg, expand(P, K), th.reshape(-1))
        np.testing.assert_array_equal(j.reshape(-1, 7), j1, err_msg=name)
        np.testing.assert_array_equal(e.reshape(-1, 3), e1, err_msg=name)
        ok = state == 0
        np.testing.assert_array_equal(proj, hs_projected(hs, cfg, P, th, True) & ok[:, None], err_msg=name)
        # is_reachable_no_limits always answers [-pi, pi] (symbolic_ik.py:117)
        assert np.all(itv[ok] == [-np.pi, np.pi]), name
    # sampled: the full circle of get_best_discrete_theta
    P = families(arm, layout)["random"]
    state, itv, used, j, e, proj = hs_sweep(sw, cfg, P, 6, None, no_limits=True)
    ok = state == 0
    np.testing.assert_array_equal(used[ok], np.broadcast_to(np.linspace(np.pi / 2, 5 * np.pi / 2, 6), (ok.sum(), 6)))


@pytest.mark.parametrize("arm", ARMS)
@pytest.mark.parametrize("layout", ["mat4", "euler"])
@pytest.mark.parametrize("K", [1, 2, 7, 20])
def test_sampled_angles(hs, sw, arm, layout, K):
    """Sampled angles are numpy's linspace over the reference's range rule on the returned interval, and the joints at
    them are the one-angle solve's at the same angles."""
    cfg = cfg_for(arm)
    for name, P in families(arm, layout).items():
        state, itv, used, j, e, proj = hs_sweep(sw, cfg, P, K)
        np.testing.assert_array_equal(used, reference_samples(itv, K), err_msg=name)
        ok = state == 0
        th = np.where(ok[:, None], used, 0.0)
        st1, itv1, j1, e1 = hs_symik(hs, cfg, expand(P, K), th.reshape(-1))
        np.testing.assert_array_equal(j.reshape(-1, 7), j1, err_msg=name)
        np.testing.assert_array_equal(e.reshape(-1, 3), e1, err_msg=name)
        np.testing.assert_array_equal(proj[ok], hs_projected(hs, cfg, P, th, False)[ok], err_msg=name)
        assert not proj[~ok].any()


def test_sample_placement_on_special_intervals(sw):
    """sweep_theta on intervals chosen to hit each branch of the range rule: full circle (either sign, within the 1e-5
    band and just outside it), wrapped, single point [a, a], and K = 1."""
    d = 2 * np.pi
    itv = np.array([[-np.pi, np.pi], [np.pi, -np.pi], [-np.pi + 4e-6, np.pi], [-np.pi + 2e-5, np.pi], [2.5, -2.0],
                    [3.0, -3.1], [0.7, 0.7], [-1.2, -1.2], [-3.0, 1.0], [0.0, 1e-12], [1.0, -d + 1.0 + 1e-9]])
    for K in (1, 2, 3, 20, 4096):
        out = np.empty((len(itv), K))
        sw.hs_sweep_theta(dp(np.ascontiguousarray(itv)), C.c_int64(len(itv)), C.c_int(K), dp(out))
        np.testing.assert_array_equal(out, reference_samples(itv, K), err_msg=f"K={K}")


@pytest.mark.parametrize("arm", ARMS)
def test_fk_round_trip(sw, arm):
    """With the elbow projection disabled (singularity_offset = -1.01), forward kinematics of the joints at every
    sampled angle reproduces the goal (tolerances of test_hostsim_parity.py::test_fk_round_trip), so all K solutions
    of a pose reach the same tip pose."""
    from reachy2_symbolic_ik_b200 import fk

    K = 6
    q = fk.sample_fk_joints(10_000, np.random.default_rng(23))
    M = fk.forward_kinematics(q, arm)
    state, itv, used, j, e, proj = hs_sweep(sw, cfg_for(arm, -1.01), M, K)
    ok = state == 0
    assert 0.3 < ok.mean() < 0.7
    assert not proj.any()
    M2 = fk.forward_kinematics(j[ok].reshape(-1, 7), arm).reshape(-1, K, 4, 4)
    goal = M[ok][:, None]
    rot_err = np.abs(M2[..., :3, :3] - goal[..., :3, :3]).max(axis=(2, 3))
    pos_err = np.linalg.norm(M2[..., :3, 3] - goal[..., :3, 3], axis=2)
    assert np.quantile(rot_err, 0.999) < 1e-5
    assert np.median(pos_err) < 1e-6 and (pos_err < 1e-5).mean() > 0.9
    # the K tips of one pose agree with each other as well as each agrees with the goal
    spread = np.linalg.norm(M2[..., :3, 3] - M2[:, :1, :3, 3], axis=2)
    assert np.median(spread) < 2e-6 and (spread < 2e-5).mean() > 0.9


# --------------------------------------------------------------------------- argument checks of the C entry
@pytest.fixture(scope="module")
def lib():
    from reachy2_symbolic_ik_b200 import _native, build

    build.build()
    return _native.load()


def test_argument_errors_do_not_need_a_device(lib):
    """Each invalid argument is refused before any CUDA call (the handle is never dereferenced on these paths)."""
    buf = (C.c_double * 64)()
    base = C.addressof(buf)
    aligned = base + (-base) % 16
    fake_handle = C.c_void_p(aligned)
    poses, out = C.c_void_p(aligned), C.c_void_p(aligned + 16)
    i64, i32 = C.c_int64, C.c_int32

    def call(h=fake_handle, kind=_abi.POSE_MAT4, P=poses, n=4, th=None, stride=0, K=3, nl=0, state=out, joints=out):
        return lib.r2ik_symik_sweep_f64(h, kind, P, i64(n), th, i32(stride), i32(K), i32(nl), None, state, None, None,
                                        joints, None, None, None)

    ERR_NULL, ERR_ARG = 1, 2
    assert call(K=0) == ERR_ARG
    assert call(K=-1) == ERR_ARG
    assert call(stride=2, th=poses) == ERR_ARG
    assert call(stride=-3, th=poses) == ERR_ARG
    assert call(n=-1) == ERR_ARG
    assert call(kind=7) == ERR_ARG
    assert call(n=(1 << 62), K=1 << 20) == ERR_ARG          # n * K * 7 overflows int64
    assert call(P=C.c_void_p(aligned + 8)) == ERR_ARG       # misaligned poses
    assert b"r2ik_symik_sweep_f64" in lib.r2ik_last_error()
    assert call(h=None) == ERR_NULL
    assert call(P=None) == ERR_NULL
    assert call(state=None) == ERR_NULL
    assert call(joints=None) == ERR_NULL
    assert b"r2ik_symik_sweep_f64" in lib.r2ik_last_error()
    assert call(h=None, n=0) == ERR_NULL                     # a null handle is refused even for an empty batch
