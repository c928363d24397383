"""Seeded trajectory families for continuous mode (ControlIK.symbolic_inverse_kinematics_batch(..., "continuous")), shared by
the host harness tests (test_continuous_edges_host.py) and the GPU tests (test_gpu_continuous_edges.py).  Every family is a
(T, W, 4, 4) batch of goal matrices; the expected values come from the CPU oracle.

A trajectory is a recursion with a continuity check: the first waypoint that jumps latches the emergency stop, and every
later waypoint returns the frozen previous solution.  So the extreme poses of edge_inputs.py, dropped into a trajectory,
test almost nothing after the first of them.  Two kinds of family follow from that.

Live families (``live_families``) reach the fragile arithmetic through transforms that keep the trajectory continuous, and
must not latch (the tests cap the latched share of each at LIVE_MAX_LATCHED, 0 unless listed there):
  scaled_ramp   the rotation block times 10^k, k from -100 to 100 along the trajectory
  float32       rounded to float32
  five_digits   rounded to 5 digits
  slow_rmfv     the elbow-circle normal (even trajectories) or the wrist direction (odd ones) sweeps through +-e_x and across
                the 1e-8 np.isclose band of rotation_matrix_from_vector (utl:59-81), 3e-10 per waypoint
  straight_arm  the elbow pitch goes to 0 (the fully stretched arm) and back
  slow_shoulder the wrist approaches the shoulder from 0.3 m to SHOULDER_MIN m, geometrically
  slow_far      the goal recedes from 0.4 m to 0.8 m from the shoulder in 100 waypoints, then geometrically to FAR_MAX m;
                past the reach sphere every waypoint is unreachable, so the stretch crosses the 127-waypoint blocks of the
                joints kernel

Latching and irregular families (``event_families``): one event per trajectory, at a waypoint of EVENT_AT (the edges of the
phased kernels' 127-waypoint blocks, 128-waypoint code tiles and 8-waypoint theta tiles), cycling through the EVENTS:
  invalid       det < 0 at that waypoint only (irregular, does not latch)
  flip          half a turn about the tool axis from that waypoint on (latches)
  far, near_shoulder, scaled, axis   one pose of the edge_inputs family of that name at that waypoint
The tests resume each trajectory after its event with "unfreeze" (parity.run_with_unfreeze).

Both are built at the largest shape, T_MAX x W_MAX; a shape (T, W) of SHAPES is the prefix [:T, :W] (a trajectory's
outputs at waypoints < W depend on those waypoints only).
"""
from __future__ import annotations

import numpy as np

import edge_inputs as E
from reachy2_symbolic_ik_b200 import fk

SEED = 20261022
T_MAX, W_MAX = 129, 256
# W: around the 127 / 128 block edge, the 128-waypoint code tile, the 8-waypoint theta tile and the W % 8 vector path;
# T: around the 64-trajectory blocks of the scans
SHAPES = [(1, 1), (63, 2), (65, 7), (64, 8), (129, 9), (1, 126), (65, 127), (63, 128), (64, 129), (129, 254), (1, 255),
          (129, 256)]
EVENT_AT = (0, 1, 7, 8, 126, 127, 128, 129, 253, 254, 255, W_MAX - 1)
EVENTS = ("invalid", "flip", "far", "near_shoulder", "scaled", "axis")
SHOULDER_MIN = 1e-6   # m: below ~1e-7 m the rounding of w = p + R wo (~1e-17 m) turns the wrist direction by > 1e-10 rad
FAR_MAX = 1e150       # m: below the 1.3e154 m at which the squared distance overflows (the goal then snaps to the shoulder)
# latched share of a live family's trajectories, and its ill-conditioned share of waypoints, that the tests accept
# slow_far: 4 of 129 per arm (the goal leaves the reach sphere faster than the elbow angle may follow); slow_shoulder: none
# of 129, 1.8 % / 2.9 % of 4 096 x 1 000 (r / l arm, B200), where the wrist is pushed out to the minimum distance
LIVE_MAX_LATCHED = {"slow_far": 0.05, "slow_shoulder": 0.04}
MAX_ILL = {"straight_arm": 0.2, "events": 0.1}  # the stretched arm's elbow circle degenerates; every other family <= 0.07
MAX_ILL_DEFAULT = 0.07


def _sinusoids(arm, T, W, seed):
    return fk.sinusoidal_trajectories(T, W, arm, seed=seed)


def _place_wrist(arm, M, w):
    """M with its translations moved so that the wrist (p + R wo) sits at w (..., 3)."""
    M = M.copy()
    M[..., :3, 3] = w - np.einsum("...ij,j->...i", M[..., :3, :3], E._wrist_offset(arm))
    return M


def _align(u, n):
    """Rotations (N,3,3) taking the unit vector u to the unit vectors n (N,3) (Rodrigues; n never equals -u here)."""
    v = np.cross(u, n)
    c = n @ u
    K = np.zeros((len(n), 3, 3))
    K[:, 0, 1], K[:, 0, 2], K[:, 1, 2] = -v[:, 2], v[:, 1], -v[:, 0]
    K = K - K.transpose(0, 2, 1)
    return np.eye(3) + K + K @ K / (1.0 + c)[:, None, None]


def _axis_angle(u, a):
    """Rotations (N,3,3) about the unit vector u by the angles a (N,)."""
    K = np.array([[0, -u[2], u[1]], [u[2], 0, -u[0]], [-u[1], u[0], 0]])
    return np.eye(3) + np.sin(a)[:, None, None] * K + (1 - np.cos(a))[:, None, None] * (K @ K)


def _rmfv(arm, T, W, seed):
    rng = np.random.default_rng(seed)
    s, wo = E._shoulder(arm), E._wrist_offset(arm)
    M = _sinusoids(arm, T, W, seed)[0]
    eps = np.linspace(-3e-8, 3e-8, W) * (W > 1)
    for k in (0.5, 0.25, 0.75):                # exact 0, -0.0 and the band edges at fixed waypoints
        eps[int(k * (W - 1))] = {0.5: 0.0, 0.25: -1e-8, 0.75: 1e-8}[k]
    for t in range(T):
        sign = 1.0 if t % 4 < 2 else -1.0
        third = eps if t % 3 else 0.0 * eps    # n = (+-sqrt(1 - e^2), e, e or 0)
        n = np.stack([sign * np.sqrt(1 - eps * eps), eps, third], axis=1)
        n /= np.linalg.norm(n, axis=1, keepdims=True)
        if t % 2 == 0:                          # elbow-circle normal (w - s) / |w - s| = n
            M[t] = _place_wrist(arm, M[t], s + n * rng.uniform(0.3, 0.5))
        else:                                   # wrist direction R wo / |wo| = n, slowly spinning about it
            u = wo / np.linalg.norm(wo)
            R = _align(u, n) @ _axis_angle(u, rng.uniform(-np.pi, np.pi) + np.linspace(0, 0.3, W))
            M[t, :, :3, :3] = R
            M[t] = _place_wrist(arm, M[t], s + np.array([0.25, 0.0, -0.2]) + rng.uniform(-0.05, 0.05, 3))
    return M


def live_families(arm: str, T: int = T_MAX, W: int = W_MAX, seed: int = SEED, only=None) -> dict[str, np.ndarray]:
    """The live families at T x W; `only`: the names to build (all by default)."""
    seed = seed + (arm == "l_arm")
    rng = np.random.default_rng(seed)
    s = E._shoulder(arm)
    M0, q0 = _sinusoids(arm, T, W, seed)
    u_near, u_far = E._units(rng, T)[:, None, :], E._units(rng, T)[:, None, :]
    u_near[..., 0], u_far[..., 0] = np.abs(u_near[..., 0]), np.abs(u_far[..., 0])     # in front of the shoulder

    def scaled_ramp():
        M = M0.copy()
        M[:, :, :3, :3] *= (10.0 ** np.linspace(-100, 100, W))[None, :, None, None]
        return M

    def straight_arm():                        # elbow pitch -0.5 s^2, s = -1 .. 1: exactly 0 at the middle waypoint
        q = q0.copy()
        q[:, :, 3] = -0.5 * np.linspace(-1, 1, W) ** 2 if W > 1 else 0.0
        return fk.forward_kinematics(q, arm)

    def slow_far():                            # across the reach sphere at 4 mm per waypoint, then geometrically
        n1 = min(W, 100)
        d = np.concatenate([np.linspace(0.4, 0.8, n1), np.geomspace(0.8, FAR_MAX, W - n1 + 1)[1:]])[None, :, None]
        M = M0.copy()
        M[:, :, :3, 3] = s + u_far * d
        return M

    make = {
        "scaled_ramp": scaled_ramp,
        "float32": lambda: M0.astype(np.float32).astype(np.float64),
        "five_digits": lambda: np.round(M0, 5),
        "slow_rmfv": lambda: _rmfv(arm, T, W, seed + 2),
        "straight_arm": straight_arm,
        "slow_shoulder": lambda: _place_wrist(arm, M0, s + u_near * np.geomspace(0.3, SHOULDER_MIN, W)[None, :, None]),
        "slow_far": slow_far,
    }
    return {name: f() for name, f in make.items() if only is None or name in only}


def event_families(arm: str, T: int = T_MAX, W: int = W_MAX, seed: int = SEED) -> tuple[dict[str, np.ndarray], np.ndarray]:
    """{"events": (T, W, 4, 4)} and the event waypoint of every trajectory (T,).  Trajectory t has its event at
    EVENT_AT[t % 12] (W_MAX - 1 when W is smaller), of kind event_kind(t): over 72 trajectories every event meets every edge."""
    seed = seed + 10 + (arm == "l_arm")
    rng = np.random.default_rng(seed)
    M = _sinusoids(arm, T, W, seed)[0].copy()
    edges = E.mat4_families(arm)
    at = np.empty(T, np.int64)
    for t in range(T):
        w = min(EVENT_AT[t % len(EVENT_AT)], W - 1)
        kind = event_kind(t)
        at[t] = w
        if kind == "invalid":
            M[t, w, :3, :3] = np.diag([1.0, -1.0, 1.0])
        elif kind == "flip":
            M[t, w:, :3, :3] = M[t, w:, :3, :3] @ np.diag([-1.0, -1.0, 1.0])
        else:
            P = edges[kind]
            M[t, w] = P[rng.integers(0, len(P))]
    return {"events": M}, at


def event_kind(t: int) -> str:
    return EVENTS[(t + t // len(EVENT_AT)) % len(EVENTS)]    # the shift by t // 12 walks each event across the edges


def perturbed_trajectories(M: np.ndarray, seed: int, amplitude: float) -> np.ndarray:
    """M with every entry of the top 3 x 4 moved by a uniform relative amount: the rotation block by amplitude times its
    scale (|R|_F / sqrt 3, which a scaled block carries), the translation by amplitude times max(1, |p|)."""
    rng = np.random.default_rng(seed)
    out = M.copy()
    R = M[..., :3, :3]
    sr = np.linalg.norm(R.reshape(*R.shape[:-2], 9), axis=-1) / np.sqrt(3)
    sp = np.maximum(1.0, np.linalg.norm(M[..., :3, 3], axis=-1))
    out[..., :3, :3] += rng.uniform(-amplitude, amplitude, R.shape) * sr[..., None, None]
    out[..., :3, 3] += rng.uniform(-amplitude, amplitude, M[..., :3, 3].shape) * sp[..., None]
    return out


# ------------------------------------------------------------------------------------------------- oracle and checks
def oracle_config(oracle, arm):
    """The controller's solver (URDF parameters, no elbow projection) and default ControlParams, as ControlIK builds them."""
    from parity import load

    u = load("symik_urdf.npz")
    params = {k[len("param_"):]: u[k] for k in u.files if k.startswith("param_")}
    return oracle.arm_config(arm, ik_parameters=params, singularity_offset=-1.01), oracle.ControlParams(arm=arm)


_REFERENCE = {}


def reference(oracle, arm, name):
    """(M, oracle outputs, ill) of family `name` at T_MAX x W_MAX.  ill (T, W): the waypoints whose oracle joints move by
    more than COND_TOL, or whose flag / state / NaN pattern changes, when the whole trajectory is perturbed by PERTURB
    (relative, 3 draws): a trajectory is a recursion, so one ill-conditioned waypoint can carry into its tail."""
    from parity import COND_TOL, PERTURB

    key = (arm, name)
    if key not in _REFERENCE:
        fams = live_families(arm)
        M = fams[name] if name in fams else event_families(arm)[0][name]
        ocfg, opar = oracle_config(oracle, arm)
        want = oracle.ctl_continuous_batch(ocfg, opar, M)
        ill = np.zeros(M.shape[:2], bool)
        for k in range(3):
            pj, pr, ps, _ = oracle.ctl_continuous_batch(ocfg, opar, perturbed_trajectories(M, 1000 + k, PERTURB))
            nan_a, nan_b = np.isnan(want[0]), np.isnan(pj)
            moved = np.where(nan_a | nan_b, 0.0, np.abs(pj - want[0])).max(axis=2)
            ill |= (moved > COND_TOL) | (nan_a != nan_b).any(axis=2) | (pr != want[1]) | (ps != want[2])
        _REFERENCE[key] = (M, want, ill)
    return _REFERENCE[key]


def compare_with_oracle(what, got, want, ill):
    """got / want = (joints, reachable, state, states) of the same trajectories: flags, states and the controller's integer
    state identical; joints within TOL and the same NaN pattern, except at ill-conditioned waypoints.  Returns the largest
    joint error among the well-conditioned waypoints."""
    from parity import TOL

    np.testing.assert_array_equal(got[1], want[1], err_msg=f"{what}: reachable")
    np.testing.assert_array_equal(got[2], want[2], err_msg=f"{what}: state")
    for f in ("emergency_stop", "emergency_bits", "init", "has_previous_sol"):
        np.testing.assert_array_equal(got[3][f], want[3][f], err_msg=f"{what}: controller {f}")
    nan_g, nan_w = np.isnan(got[0]), np.isnan(want[0])
    err = np.where(nan_g | nan_w, 0.0, np.abs(got[0] - want[0])).max(axis=2)
    bad = ((err > TOL) | (nan_g != nan_w).any(axis=2)) & ~ill
    assert not bad.any(), (f"{what}: {int(bad.sum())} well-conditioned waypoints off the oracle, first (t, w) "
                           f"{np.argwhere(bad)[:5].tolist()}, max|err| {err[bad].max():.3e}")
    return float(np.where(ill, 0.0, err).max(initial=0.0))


def assert_same_trajectories(a, b, what, atol=1e-12):
    """Two forms of the controller on the same trajectories: flags, states and the integer controller state identical,
    joints / previous_sol / previous_theta equal to atol (0: bit for bit)."""
    for i, name in ((1, "reachable"), (2, "state")):
        np.testing.assert_array_equal(a[i], b[i], err_msg=f"{what}: {name}")
    for f in ("has_previous_sol", "init", "emergency_stop", "emergency_bits"):
        np.testing.assert_array_equal(a[3][f], b[3][f], err_msg=f"{what}: controller {f}")
    for x, y, name in ((a[0], b[0], "joints"), (a[3]["previous_sol"], b[3]["previous_sol"], "previous_sol"),
                       (a[3]["previous_theta"], b[3]["previous_theta"], "previous_theta")):
        if atol == 0:
            np.testing.assert_array_equal(x, y, err_msg=f"{what}: {name}")
        else:
            np.testing.assert_allclose(x, y, rtol=0, atol=atol, err_msg=f"{what}: {name}")


def split_run(run, M, cuts):
    """run(M, states) -> (joints, reachable, state, states) over the waypoint segments cut at `cuts`, each resumed from the
    states the previous one returned; the pieces concatenated."""
    edges = [0, *cuts, M.shape[1]]
    parts, st = [], None
    for lo, hi in zip(edges[:-1], edges[1:]):
        j, r, s, st = run(np.ascontiguousarray(M[:, lo:hi]), st)
        parts.append((j, r, s))
    return (np.concatenate([p[0] for p in parts], axis=1), np.concatenate([p[1] for p in parts], axis=1),
            np.concatenate([p[2] for p in parts], axis=1), st)


SPLITS = (5, 61, 131, 250)    # resume points that are multiples of neither 8 nor 127


def unfreeze_run(run, oracle, Mt, at):
    """One trajectory Mt (W,4,4) with control_type "unfreeze" right after its event at waypoint `at`
    (parity.run_with_unfreeze), through run(M (1,w,4,4), states) -> (joints, reachable, state, states); returned with a
    leading trajectory axis."""
    from parity import run_with_unfreeze

    st0 = np.zeros(1, dtype=oracle.CTL_STATE_DTYPE)
    st0["init"] = 1
    j, r, s, st = run_with_unfreeze(run, Mt, [at + 1] if at + 1 < len(Mt) else [], st0)
    return j[None], r[None], s[None], st


_UNFREEZE = {}


def unfreeze_references(oracle, arm):
    """[(t, oracle outputs of unfreeze_run, ill (1, W))] for every trajectory of the event family; ill as in reference(),
    from the unfreeze runs of the perturbed trajectory."""
    from parity import COND_TOL, PERTURB

    if arm not in _UNFREEZE:
        M, _, _ = reference(oracle, arm, "events")
        at = event_families(arm)[1]
        ocfg, opar = oracle_config(oracle, arm)
        orc = lambda m, st: oracle.ctl_continuous_batch(ocfg, opar, m, states=st)  # noqa: E731
        perturbed = [perturbed_trajectories(M, 1000 + k, PERTURB) for k in range(3)]
        out = []
        for t in range(len(M)):
            want = unfreeze_run(orc, oracle, M[t], at[t])
            ill = np.zeros((1, M.shape[1]), bool)
            for Mp in perturbed:
                alt = unfreeze_run(orc, oracle, Mp[t], at[t])
                nan_a, nan_b = np.isnan(want[0]), np.isnan(alt[0])
                moved = np.where(nan_a | nan_b, 0.0, np.abs(alt[0] - want[0])).max(axis=2)
                ill |= (moved > COND_TOL) | (nan_a != nan_b).any(axis=2) | (alt[1] != want[1]) | (alt[2] != want[2])
            out.append((t, want, ill))
        _UNFREEZE[arm] = out
    return _UNFREEZE[arm]
