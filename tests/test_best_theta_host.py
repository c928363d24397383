"""The batched get_best_theta_to_current_joints (r2ik_symik_best_theta_f64) on the host: tests/hostsim/best_theta.cpp runs
symik_best_theta, the per-pose body of k_symik_best_theta, and this file holds it to the CPU oracle's search by the rule
of tests/best_theta_util.py (states identical; angles identical wherever no decision of the search is within rounding
of a tie; joints within the parity tolerance), checks that the reference's state leak between the search's evaluations
is reproduced, pins the shortcut at the preferred angle, and exercises the argument checks of the C entry on
libr2ik.so without a device."""
import ctypes as C

import numpy as np
import pytest

import best_theta_util as B
from parity import MAX_ILL_FRACTION, Report, ill_conditioned_mask
from reachy2_symbolic_ik_b200 import _abi

ARMS = B.ARMS
ORDINARY = ("fk", "golden", "named", "shortcut_exact", "shortcut_below", "shortcut_above")


@pytest.fixture(scope="module")
def libs(tmp_path_factory):
    return B.build_libs(str(tmp_path_factory.mktemp("best_theta")))


@pytest.fixture(scope="module")
def hs_one(tmp_path_factory):
    """The one-angle host solve of tests/hostsim/hostsim.cpp (K1 / K1b on the host)."""
    import os
    import subprocess

    subprocess.run(["make", "-C", B.HS_DIR], check=True, capture_output=True)
    return C.CDLL(os.path.join(B.HS_DIR, "_build", "libr2ik_hostsim.so"))


def one_angle(hs, arm, P, theta, no_limits=False, singularity_offset=0.03):
    """joints of the one-angle host solve (hs_symik_batch / hs_no_limits_batch) at theta (n,)."""
    P, kind = B._rows(P)
    n = len(P)
    cfg = _abi.make_arm_config(arm, _abi.DEFAULT_IK_PARAMETERS, 127, 42.5, 1e-8, 0.02, 1e-7, singularity_offset, 1.0)
    th = np.ascontiguousarray(theta, dtype=np.float64)
    j = np.empty((n, 7)); e = np.empty((n, 3))
    if no_limits:
        hs.hs_no_limits_batch(C.byref(cfg), kind, B._dp(P), B._dp(th), C.c_int64(n), B._dp(j), B._dp(e))
    else:
        reach = np.zeros(n, np.uint8); state = np.zeros(n, np.uint8); itv = np.empty((n, 2))
        hs.hs_symik_batch(C.byref(cfg), kind, B._dp(P), B._dp(th), C.c_int64(n), B._u8(reach), B._u8(state), B._dp(itv),
                          B._dp(j), B._dp(e))
    return j


def check_joints(name, oracle, arm, P, theta, joints, no_limits):
    """joints against the oracle's one-angle solve at the same angles, parity tolerances, ill-conditioned poses excused
    as in the other parity tests."""
    ocfg = oracle.arm_config(arm)
    th = np.where(np.isnan(theta), 0.0, theta)
    rows, _ = B._rows(P)
    if no_limits:
        run = lambda p: oracle.symik_no_limits_batch(ocfg, p.reshape(rows.shape), th)[:1]   # noqa: E731
    else:
        run = lambda p: (oracle.symik_batch(ocfg, p.reshape(rows.shape), th)[3],)          # noqa: E731
    want = run(rows)[0]
    want = np.where(np.isnan(theta)[:, None], np.nan, want)
    ill = ill_conditioned_mask(run, rows)
    rep = Report(name, len(P), ill)
    rep.close("joints", joints, want)
    rep.check(max_ill_fraction=1.0)    # small families: the share of ill-conditioned poses is bounded over the whole test
    return int(ill.sum()), len(P)


@pytest.mark.parametrize("arm", ARMS)
@pytest.mark.parametrize("layout", ["mat4", "euler"])
@pytest.mark.parametrize("no_limits", [False, True])
def test_host_build_matches_the_oracle(libs, oracle, hs_one, arm, layout, no_limits):
    """Every family with its current joints (the generating joints for FK poses, random joints otherwise), and the
    FK poses with current joints at distance 0, just below and just above 0.01 of the preferred angle's joints."""
    hs, orc = libs
    mm = B.Mismatches(f"host {arm} {layout} no_limits={no_limits}")
    fams = B.families(arm, layout, n_fk=1500, seed=3)
    P_fk = fams["fk"][0]
    j_pref = one_angle(hs_one, arm, P_fk, np.full(len(P_fk), B.preferred_theta(arm)), no_limits)
    ok = ~np.isnan(j_pref).any(axis=1)
    exact, below, above = B.near_shortcut(np.where(ok[:, None], j_pref, 0.0), np.random.default_rng(4))
    fams.update({"shortcut_exact": (P_fk, exact), "shortcut_below": (P_fk, below), "shortcut_above": (P_fk, above)})
    n_ill = n_all = 0
    for name, (P, cj) in fams.items():
        got = B.hs_best_theta(hs, arm, P, cj, no_limits=no_limits)
        want = B.oracle_best_theta(orc, oracle, arm, P, cj, no_limits=no_limits, check=(name == "fk"))
        if want[5] is not None:   # the margin-recording search is the oracle's own function's search
            np.testing.assert_array_equal(want[1], want[5])
        same = mm.check(name, got, want)
        # joints are the one-angle solve's at the returned angle, bit for bit, and the oracle's within tolerance
        nan = np.isnan(got[1])
        one = one_angle(hs_one, arm, P, np.where(nan, 0.0, got[1]), no_limits)
        np.testing.assert_array_equal(got[2], np.where(nan[:, None], np.nan, one), err_msg=name)
        i, m = check_joints(f"{arm} {layout} {name} nl={no_limits}", oracle, arm, P, got[1], got[2], no_limits)
        if name in ORDINARY:   # the extreme-input families are ill-conditioned by construction (tests/edge_inputs.py)
            n_ill += i; n_all += m
        assert same.any() or not (got[0] == 0).any()
    print(mm.report())
    assert n_ill <= MAX_ILL_FRACTION * n_all, f"{n_ill} of {n_all} poses ill-conditioned"


@pytest.mark.parametrize("arm", ARMS)
def test_shortcut_edge(libs, hs_one, arm):
    """Current joints at distance < 0.01 from the preferred angle's joints give exactly preferred_theta; at > 0.01 the
    search runs and returns another angle.  Also for a preferred angle that is not ControlIK's."""
    hs, _ = libs
    P = B.families(arm, "mat4", n_fk=800, seed=5)["fk"][0]
    for pref in (B.preferred_theta(arm), 0.3):
        j_pref = one_angle(hs_one, arm, P, np.full(len(P), pref))
        ok = ~np.isnan(j_pref).any(axis=1)
        exact, below, above = B.near_shortcut(j_pref[ok], np.random.default_rng(6))
        for cj, hit in ((exact, True), (below, True), (above, False)):
            st, th, j = B.hs_best_theta(hs, arm, P[ok], cj, pref=pref)
            assert (st == 0).all()
            if hit:
                assert (th == pref).all()
                np.testing.assert_array_equal(j, j_pref[ok])
            else:
                assert not (th == pref).any()


@pytest.mark.parametrize("arm", ARMS)
def test_the_state_leak_is_reproduced(libs, oracle, hs_one, arm):
    """Searches in which make_elbow_projection fires: the entry follows the reference's closure, whose evaluations see
    the goal / wrist the previous ones moved, and a control search that runs every evaluation on a fresh solve gives a
    different angle on some of them.  Where the projection never fires (singularity_offset = -1.01 puts its plane out
    of reach) the two searches agree."""
    hs, orc = libs
    P, cj = B.families(arm, "mat4", n_fk=3000, seed=8)["fk"]
    st, th, j = B.hs_best_theta(hs, arm, P, cj)
    ok = st == 0
    fresh = B.fresh_search(lambda t: one_angle(hs_one, arm, P[ok], t), int(ok.sum()), arm, cj[ok])
    differ = fresh != th[ok]
    want = B.oracle_best_theta(orc, oracle, arm, P[ok], cj[ok])
    margin = np.minimum(want[3], want[4])
    print(f"[{arm}] {int(ok.sum())} reachable poses; the fresh-solve search differs on {int(differ.sum())}, "
          f"{int((differ & (margin > B.THETA_MARGIN)).sum())} of them clear of a tie")
    assert (differ & (margin > B.THETA_MARGIN)).sum() >= 10
    # without the projection there is nothing to leak
    st2, th2, _ = B.hs_best_theta(hs, arm, P, cj, singularity_offset=-1.01)
    ok2 = st2 == 0
    fresh2 = B.fresh_search(lambda t: one_angle(hs_one, arm, P[ok2], t, singularity_offset=-1.01), int(ok2.sum()), arm,
                            cj[ok2])
    assert (fresh2 == th2[ok2]).mean() > 0.99


def test_iterations_do_not_depend_on_the_pose():
    """2 pi (2/3)^16 < 0.01 < 2 pi (2/3)^15: every search runs 16 iterations, whichever side each comparison takes."""
    for lo, hi in ((-np.pi, np.pi), (0.0, 2 * np.pi)):
        for bits in range(0, 1 << 16, 257):
            a, b, k = lo, hi, 0
            while b - a > B.SHORTCUT:
                m1, m2 = a + (b - a) / 3, b - (b - a) / 3
                if (bits >> k) & 1:
                    b = m2
                else:
                    a = m1
                k += 1
            assert k == 16


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

    def call(h=fake_handle, kind=_abi.POSE_MAT4, P=poses, n=4, cj=out, stride=7, nl=0, state=out, theta=out, joints=None):
        return lib.r2ik_symik_best_theta_f64(h, kind, P, i64(n), cj, i32(stride), C.c_double(-2.0), i32(nl), state, theta,
                                             joints, None)

    ERR_NULL, ERR_ARG = 1, 2
    assert call(stride=1) == ERR_ARG
    assert call(stride=-7) == ERR_ARG
    assert call(n=-1) == ERR_ARG
    assert call(kind=7) == ERR_ARG
    assert call(P=C.c_void_p(aligned + 8)) == ERR_ARG       # misaligned poses
    assert b"r2ik_symik_best_theta_f64" in lib.r2ik_last_error()
    assert call(h=None) == ERR_NULL
    assert call(P=None) == ERR_NULL
    assert call(cj=None) == ERR_NULL
    assert call(state=None) == ERR_NULL
    assert call(theta=None) == ERR_NULL
    assert b"r2ik_symik_best_theta_f64" in lib.r2ik_last_error()
    assert call(h=None, n=0) == ERR_NULL                     # a null handle is refused even for an empty batch
