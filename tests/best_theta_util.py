"""Shared by tests/test_best_theta_host.py and tests/test_gpu_best_theta.py: the host builds that the batched
get_best_theta_to_current_joints (r2ik_symik_best_theta_f64) is held to, the input families, and the comparison rule.

  hostsim  tests/hostsim/best_theta.cpp: symik_best_theta, the per-pose body of k_symik_best_theta, on the CPU
  oracle   tests/hostsim/best_theta_oracle.c: the CPU oracle's search (oracle/r2ik_oracle.c) batched, with the margins of
           each search's decisions

The search compares two joint distances per iteration and the shortcut compares one with 0.01.  Joints that agree within
the parity tolerance TOL per joint give distances that agree within sqrt(7) TOL each, so a decision whose two sides
differ by more than THETA_MARGIN = 2 sqrt(7) TOL cannot be flipped by rounding within tolerance: there the angle must be
identical, and elsewhere a different angle is a tie decided by rounding, counted and reported.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

from parity import REPO, TOL
from reachy2_symbolic_ik_b200 import _abi, fk

HS_DIR = os.path.join(REPO, "tests", "hostsim")
THETA_MARGIN = 2 * np.sqrt(7) * TOL
ARMS = ("r_arm", "l_arm")
SHORTCUT = 0.01     # utils.py:283


def preferred_theta(arm: str) -> float:
    """ControlIK's preferred elbow angle for the arm (control_ik.py: -4 pi / 6, mirrored for l_arm)."""
    return -4 * np.pi / 6 if arm == "r_arm" else -np.pi - (-4 * np.pi / 6)


def build_libs(out_dir: str):
    """(hostsim, oracle) built into out_dir with the flags of tests/hostsim/Makefile and oracle/Makefile."""
    hs = os.path.join(out_dir, "libr2ik_hostsim_best_theta.so")
    orc = os.path.join(out_dir, "libr2ik_oracle_best_theta.so")
    subprocess.run(["g++", "-O2", "-fPIC", "-std=c++17", "-ffp-contract=off", "-Wall", "-Wno-unknown-pragmas", "-shared",
                    "-o", hs, os.path.join(HS_DIR, "best_theta.cpp"), "-lm"], check=True, capture_output=True)
    subprocess.run(["gcc", "-O2", "-fPIC", "-fopenmp", "-ffp-contract=off", "-fno-fast-math", "-std=c11", "-shared",
                    "-o", orc, os.path.join(HS_DIR, "best_theta_oracle.c"), "-lm"], check=True, capture_output=True)
    return C.CDLL(hs), C.CDLL(orc)


def _dp(a):
    return None if a is None else a.ctypes.data_as(C.POINTER(C.c_double))


def _u8(a):
    return a.ctypes.data_as(C.POINTER(C.c_uint8))


def _rows(P):
    P = np.ascontiguousarray(P, dtype=np.float64)
    if P.shape[1:] in ((4, 4), (16,)):
        return P.reshape(len(P), 16), _abi.POSE_MAT4
    return P.reshape(len(P), 6), _abi.POSE_EULER6


def _cj(cj, n):
    cj = np.ascontiguousarray(cj, dtype=np.float64)
    return cj, (0 if cj.shape in ((7,), (1, 7)) else 7)


def hs_best_theta(hs, arm, P, cj, pref=None, no_limits=False, singularity_offset=0.03):
    """hostsim: state, theta, joints."""
    P, kind = _rows(P)
    n = len(P)
    cj, stride = _cj(cj, n)
    cfg = _abi.make_arm_config(arm, _abi.DEFAULT_IK_PARAMETERS, 127, 42.5, 1e-8, 0.02, 1e-7, singularity_offset, 1.0)
    state = np.zeros(n, np.uint8); theta = np.empty(n); joints = np.empty((n, 7))
    hs.hs_symik_best_theta(C.byref(cfg), kind, _dp(P), C.c_int64(n), _dp(cj), C.c_int(stride),
                           C.c_double(preferred_theta(arm) if pref is None else pref), C.c_int(int(no_limits)),
                           _u8(state), _dp(theta), _dp(joints))
    return state, theta, joints


def oracle_best_theta(orc, oracle, arm, P, cj, pref=None, no_limits=False, check=False):
    """oracle: state, theta, joints, cmp_margin, shortcut_margin, theta of the oracle's own function (check) or None."""
    P, kind = _rows(P)
    n = len(P)
    cj, stride = _cj(cj, n)
    ocfg = oracle.arm_config(arm)
    state = np.zeros(n, np.uint8); theta = np.empty(n); joints = np.empty((n, 7))
    cmp_m = np.empty(n); short_m = np.empty(n); chk = np.empty(n) if check else None
    orc.orc_best_theta_batch(C.byref(ocfg), kind, _dp(P), C.c_int64(n), _dp(cj), C.c_int(stride),
                             C.c_double(preferred_theta(arm) if pref is None else pref), C.c_int(int(no_limits)),
                             _u8(state), _dp(theta), _dp(joints), _dp(cmp_m), _dp(short_m), _dp(chk))
    return state, theta, joints, cmp_m, short_m, chk


def fresh_search(solve, n, arm, cj, pref=None):
    """Control for the state leak: the reference's search with every get_joints on a FRESH solve of the pose.
    solve(theta (n,)) -> joints (n,7) of the one-angle solve.  Vectorised over the poses: 33 calls of solve."""
    pref = preferred_theta(arm) if pref is None else pref
    cj = np.broadcast_to(np.asarray(cj, dtype=np.float64), (n, 7))

    def dist(j):
        d = np.remainder(j - cj + np.pi, 2 * np.pi) - np.pi     # angle_diff (utils.py:468-490)
        return np.sqrt((d * d).sum(axis=1))

    lo = np.full(n, 0.0 if arm == "l_arm" else -np.pi)
    hi = np.full(n, 2 * np.pi if arm == "l_arm" else np.pi)
    short = dist(solve(np.full(n, pref))) < SHORTCUT
    while (hi - lo > SHORTCUT).any():
        m1 = lo + (hi - lo) / 3
        m2 = hi - (hi - lo) / 3
        f1, f2 = dist(solve(m1)), dist(solve(m2))
        better1 = f1 < f2
        hi = np.where(better1, m2, hi)
        lo = np.where(better1, lo, m1)
    return np.where(short, pref, (lo + hi) / 2)


def families(arm, layout, n_fk=2000, seed=0):
    """Poses with current joints of four kinds.  Returns {name: (poses, current_joints (N,7))}; the FK family's
    current joints are the joints that generated each pose.  The shortcut kinds are built by the caller (they need a
    solve at the preferred angle)."""
    import edge_inputs as E
    from parity import load
    from scipy.spatial.transform import Rotation

    rng = np.random.default_rng(seed + (arm == "l_arm"))
    q = fk.sample_fk_joints(n_fk, rng)
    M = fk.forward_kinematics(q, arm)
    g = load(f"symik_random_{arm}.npz")
    named = load("symik_named.npz")[f"{arm}_poses"]
    if layout == "mat4":
        Mn = np.tile(np.eye(4), (len(named), 1, 1))
        Mn[:, :3, :3] = Rotation.from_euler("xyz", named[:, 1]).as_matrix()
        Mn[:, :3, 3] = named[:, 0]
        fam = {"fk": M, "golden": g["M"], "named": Mn}
        fam.update(E.mat4_families(arm))
    else:
        def to6(X):
            return np.concatenate([X[:, :3, 3], Rotation.from_matrix(X[:, :3, :3]).as_euler("xyz")], axis=1)
        fam = {"fk": to6(M), "golden": g["goal_pose"], "named": named}
        fam.update(E.euler_families(arm))
    out = {}
    for name, P in fam.items():
        P = np.ascontiguousarray(P, dtype=np.float64)
        cj = q if name == "fk" else fk.sample_fk_joints(len(P), rng)
        out[name] = (P, np.ascontiguousarray(cj))
    return out


def near_shortcut(j_pref, rng):
    """Current joints at joint distance 0, just below and just above 0.01 from the joints at the preferred angle:
    (exact (N,7), below (N,7), above (N,7)).  The offset is along a random unit direction; 1e-4 relative keeps the
    distance clear of 0.01 by far more than rounding."""
    u = rng.normal(size=j_pref.shape)
    u /= np.linalg.norm(u, axis=1, keepdims=True)
    return j_pref, j_pref + u * (SHORTCUT * (1 - 1e-4)), j_pref + u * (SHORTCUT * (1 + 1e-4))


class Mismatches:
    """The comparison rule of the module docstring, accumulated over calls; `report()` returns the summary line."""

    def __init__(self, name):
        self.name = name
        self.n = 0
        self.tie = 0
        self.lines = []

    def check(self, what, got, want):
        """got = (state, theta, joints) of the build under test; want = oracle_best_theta's tuple."""
        g_state, g_theta, g_joints = got
        w_state, w_theta, w_joints, cmp_m, short_m = want[:5]
        np.testing.assert_array_equal(g_state, w_state, err_msg=f"{self.name} {what}: states")
        ok = w_state == 0
        assert np.isnan(g_theta[~ok]).all() and np.isnan(g_joints[~ok]).all(), f"{self.name} {what}: NaN rows"
        same = (g_theta == w_theta) | ~ok
        margin = np.minimum(cmp_m, short_m)
        genuine = ~same & (margin > THETA_MARGIN)
        self.n += int(ok.sum())
        self.tie += int((~same).sum())
        if (~same).any():
            self.lines.append(f"{what}: {int((~same).sum())} angles differ, margins {np.sort(margin[~same])[:5]}")
        assert not genuine.any(), (f"{self.name} {what}: {int(genuine.sum())} angles differ where every decision margin "
                                   f"exceeds {THETA_MARGIN:.2e}: indices {np.nonzero(genuine)[0][:10]}, "
                                   f"got {g_theta[genuine][:5]} want {w_theta[genuine][:5]}")
        return same & ok

    def report(self):
        msg = f"[{self.name}] {self.n} reachable poses, {self.tie} angles decided differently within rounding of a tie"
        return "\n  ".join([msg] + self.lines)
