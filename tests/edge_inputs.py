"""Seeded extreme inputs for the solver's C ABI, shared by the GPU tests (test_gpu_edges.py) and the host harness tests
(test_hostsim_parity.py).  Every family is a batch of goal poses; the expected values come from the CPU oracle.

Families (``mat4_families(arm)``, (N,4,4) homogeneous matrices, and ``euler_families(arm)``, (N,2,3) goal poses):
  far            goal at 10^k m from the shoulder, k = -300 .. 200: inside the arm, on the reach sphere's side of it, and
                 past 1.3e154 m, where the squared distance overflows to inf
  near_shoulder  wrist within 10^-k m of the shoulder, k = 0 .. 300 (pushed out to the minimum distance)
  scaled         rotation blocks times 10^k, k = -100 .. 100 (scipy projects them back onto a rotation; beyond that
                 range the determinant whose sign decides validity under- or overflows, and whether it does depends
                 on how it is evaluated -- numpy's LU against the closed form -- not on the rotation)
  axis           exact axis rotations with signed zeros, and single subnormal / signed-zero entries in them
  rmfv           poses whose elbow-circle normal or wrist direction is +-e_x exactly, or sits on the np.isclose edges
                 of rotation_matrix_from_vector (utl:59-81)
  float32, five_digits  non-orthonormal blocks: float32-rounded, or printed with 5 digits
  big_euler      euler angles of 1e3 .. 1e15 rad (euler families only), and the same magnitudes as theta (``big_thetas``)
"""
from __future__ import annotations

import numpy as np

from reachy2_symbolic_ik_b200 import _abi, fk

SEED = 20261020


def _shoulder(arm):
    return np.asarray(_abi.DEFAULT_IK_PARAMETERS[f"{arm[0]}_shoulder_position"], dtype=np.float64)


def _wrist_offset(arm):
    """wo: the wrist in the goal frame (sik:422), for the default tip."""
    tip = np.asarray(_abi.DEFAULT_IK_PARAMETERS[f"{arm[0]}_tip_position"], dtype=np.float64)
    return np.array([-tip[0], tip[1], tip[2]])


def _units(rng, n):
    v = rng.normal(size=(n, 3))
    return v / np.linalg.norm(v, axis=1, keepdims=True)


def _with_rot(R, p):
    M = np.tile(np.eye(4), (len(R), 1, 1))
    M[:, :3, :3] = R
    M[:, :3, 3] = p
    return M


def _axis_rotations():
    """All 24 proper rotations with entries in {0, -0, 1, -1}, in both signs of their zeros."""
    out = []
    import itertools

    for perm in itertools.permutations(range(3)):
        for signs in itertools.product((1.0, -1.0), repeat=3):
            R = np.zeros((3, 3))
            for i, j in enumerate(perm):
                R[i, j] = signs[i]
            if np.linalg.det(R) > 0:
                out.append(R)
                out.append(np.where(R == 0, -0.0, R))
    return np.array(out)


def mat4_families(arm: str, seed: int = SEED) -> dict[str, np.ndarray]:
    rng = np.random.default_rng(seed + (arm == "l_arm"))
    s, wo = _shoulder(arm), _wrist_offset(arm)
    base = fk.sample_fk_poses(4000, arm, seed=seed % 1000)
    R0 = base[:, :3, :3]
    fam = {}

    k = np.repeat(np.arange(-300, 201, dtype=np.float64), 3)
    d = 10.0 ** k * rng.choice([1.0, 1.0 + 1e-9, 0.5], len(k))
    fam["far"] = _with_rot(R0[rng.integers(0, len(R0), len(k))], s + _units(rng, len(k)) * d[:, None])

    k = np.repeat(np.arange(0, 301, dtype=np.float64), 2)
    R = R0[rng.integers(0, len(R0), len(k))]
    w = s + _units(rng, len(k)) * (10.0 ** -k)[:, None]
    fam["near_shoulder"] = _with_rot(R, w - np.einsum("nij,j->ni", R, wo))

    k = np.arange(-100, 101, 2, dtype=np.float64)
    pick = rng.integers(0, len(base), len(k))
    M = base[pick].copy()
    M[:, :3, :3] *= (10.0 ** k)[:, None, None]
    fam["scaled"] = M

    A = _axis_rotations()
    reps = 6
    R = np.repeat(A, reps, axis=0)
    p = s + _units(rng, len(R)) * rng.uniform(0.15, 0.5, (len(R), 1))
    p[:, 0] = np.abs(p[:, 0]) + 0.05
    M = _with_rot(R, p)
    tweak = M[::3].copy()                 # one entry of the block replaced by a subnormal / signed zero / tiny number
    i, j = rng.integers(0, 3, len(tweak)), rng.integers(0, 3, len(tweak))
    tweak[np.arange(len(tweak)), i, j] += rng.choice([5e-324, -5e-324, 1e-310, -0.0, 1e-17], len(tweak))
    fam["axis"] = np.concatenate([M, tweak])

    # rmfv: the elbow-circle normal n = (w - s) / |w - s| = +-e_x, or (cos a, sin a, 0) with sin a on the isclose edge
    # 1e-8 of utl:66-70; the wrist-limit normal (w - p) / |w - p| = R wo / |wo| likewise (exact axis rotations)
    eps = np.array([0.0, -0.0, 1e-8 * (1 - 1e-3), 1e-8, 1e-8 * (1 + 1e-3), 1e-8 * (1 + 1e-5), 2e-8, 1e-7])
    dist = np.array([0.3, 0.45, 0.52])
    sign = np.array([1.0, -1.0])
    E, D, S = (a.ravel() for a in np.meshgrid(eps, dist, sign, indexing="ij"))
    n = np.stack([S * np.sqrt(1 - E * E), E, np.where(np.arange(len(E)) % 2 == 0, 0.0, E)], axis=1)
    R = np.repeat(A[:4], len(E) // 4 + 1, axis=0)[: len(E)]
    w = s + n * D[:, None]
    fam["rmfv"] = _with_rot(R, w - np.einsum("nij,j->ni", R, wo))

    X = fk.sample_fk_poses(3000, arm, seed=seed % 1000 + 1)
    fam["float32"] = X.astype(np.float32).astype(np.float64)
    fam["five_digits"] = np.round(X, 5)
    return fam


def undetermined_wrist_direction(arm: str, M: np.ndarray) -> np.ndarray:
    """(N,) bool: the wrist lies within 1e-7 m of the shoulder, where the rounding of w = p + R wo (~1e-17 m) turns the
    direction (w - s) / |w - s| that the minimum-distance push-out follows by more than 1e-10 rad."""
    w = M[:, :3, 3] + np.einsum("nij,j->ni", M[:, :3, :3], _wrist_offset(arm))
    return np.linalg.norm(w - _shoulder(arm), axis=1) < 1e-7


def euler_families(arm: str, seed: int = SEED) -> dict[str, np.ndarray]:
    rng = np.random.default_rng(seed + 10 + (arm == "l_arm"))
    s = _shoulder(arm)
    n = 3000
    P = np.empty((n, 2, 3))
    P[:, 0] = s + _units(rng, n) * rng.uniform(0.1, 0.7, (n, 1))
    P[:, 0, 0] = np.abs(P[:, 0, 0])
    mag = 10.0 ** rng.uniform(3, 15, (n, 3)) * rng.choice([-1.0, 1.0], (n, 3))
    keep = rng.random((n, 3)) < 0.3                     # some axes stay ordinary
    P[:, 1] = np.where(keep, rng.uniform(-np.pi, np.pi, (n, 3)), mag)
    fam = {"big_euler": P}
    far = P[:600].copy()
    far[:, 0] = s + _units(rng, 600) * (10.0 ** rng.uniform(-300, 200, 600))[:, None]
    fam["far_euler"] = far
    return fam


def big_thetas(n: int, seed: int = SEED) -> np.ndarray:
    rng = np.random.default_rng(seed + 20)
    return 10.0 ** rng.uniform(3, 15, n) * rng.choice([-1.0, 1.0], n)
