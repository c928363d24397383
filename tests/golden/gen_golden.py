"""Generate the golden fixtures under tests/golden/ by running the UNMODIFIED reference.

Runs only in the build container, where the reference checkout is mounted read-only at
/root/reference (it does not exist on the GPU box).  The fixtures pin (a) the CPU oracle
(oracle/r2ik_oracle.c) and (b) the CUDA library, to the reference's own outputs:

    PYTHONDONTWRITEBYTECODE=1 python tests/golden/gen_golden.py

Oracle of record = reference source + this container's numpy / scipy (versions are stored
in every file; the reference pins scipy == 1.8.0, this container has scipy 1.18.1).

Every file stays below 1 MB: symik_random_<arm>.npz, symik_ctor.npz and symik_elbow.npz keep a fixed, seeded subset
of the poses solved here (golden_subset.py says which rows and why the tests still find their blocks).

Reference quirk handled here (SURVEY.md A.6.1): ``get_joints`` mutates the solver when the
elbow projection fires, so every ``get_joints`` below is preceded by a fresh ``is_reachable``.
"""
from __future__ import annotations

import os
import sys
import time
import warnings

import numpy as np
import scipy

HERE = os.path.dirname(os.path.abspath(__file__))
REPO = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, "/root/reference/src")
sys.path.insert(0, REPO)
sys.dont_write_bytecode = True
warnings.filterwarnings("ignore", message="Gimbal lock detected")

from scipy.spatial.transform import Rotation as R  # noqa: E402

import reachy2_symbolic_ik.control_ik as ref_control  # noqa: E402
from reachy2_symbolic_ik.control_ik import ControlIK  # noqa: E402
from reachy2_symbolic_ik.symbolic_ik import SymbolicIK  # noqa: E402
from reachy2_symbolic_ik.utils import get_ik_parameters_from_urdf  # noqa: E402

from reachy2_symbolic_ik_b200 import fk  # noqa: E402
import golden_subset  # noqa: E402  (this directory: sys.path[0] when run as a script)

STATE_CODES = {
    "reachable": 0,
    "Pose out of reach": 1,
    "Backward pose": 2,
    "wrist out of range": 3,
    "limited by wrist": 4,
    "out of reach - should not happen": 5,
    "limited by shoulder": 6,
    "": 7,
}
META = dict(numpy_version=np.__version__, scipy_version=scipy.__version__, reference="pollen-robotics/reachy2_symbolic_ik")
URDF_PATH = "/root/reference/src/config_files/reachy2.urdf"


class _Quiet:
    def __enter__(self):
        self._o = sys.stdout
        sys.stdout = open(os.devnull, "w")

    def __exit__(self, *a):
        sys.stdout.close()
        sys.stdout = self._o


def state_code(s: str) -> int:
    if s.startswith("\nEMERGENCY") or "EMERGENCY" in s:
        return 8
    return STATE_CODES[s]


def euler_pose_from_matrix(M):
    return np.array([M[:3, 3], R.from_matrix(M[:3, :3]).as_euler("xyz")])


def run_symik(ik: SymbolicIK, goal_poses, thetas=None):
    """goal_poses: (N,2,3).  Returns flag, state, interval, joints@theta(or interval[0]), elbow."""
    n = len(goal_poses)
    flag = np.zeros(n, bool)
    state = np.zeros(n, np.uint8)
    interval = np.full((n, 2), np.nan)
    joints = np.full((n, 7), np.nan)
    elbow = np.full((n, 3), np.nan)
    for i, gp in enumerate(goal_poses):
        ok, itv, fn, st = ik.is_reachable(np.array(gp))
        flag[i] = ok
        state[i] = state_code(st)
        if ok:
            interval[i] = itv
            th = itv[0] if thetas is None else thetas[i]
            j, e = fn(th)
            joints[i] = j
            elbow[i] = np.asarray(e)[:3]
    return flag, state, interval, joints, elbow


def named_poses():
    """Poses named in the reference's tests / docs / examples (euler format), per arm."""
    rad = np.radians
    r = [
        # tests/test_ik.py:15-79
        [[0.4, 0.2, 0.1], [rad(-60), rad(-90), rad(20)]],
        [[0.3, -0.2, -0.3], [rad(0), rad(-90), rad(0)]],
        [[0.02, -0.2, -0.65], [0.0, 0.0, 0.0]],
        [[0.0, -0.2, -0.65], [0.0, 0.0, 0.0]],
        [[0.87, -0.2, -0.0], [0.0, -np.pi / 2, 0.0]],
        [[0.35, -0.2, -0.28], [0.0, -np.pi / 2, 0.0]],
        # README.md:73-75
        [[0.55, -0.3, -0.15], [0.0, -np.pi / 2, 0.0]],
        # src/benchmark/ik_benchmarks.py:13-14
        [[0.3, -0.1, 0.1], [rad(20), rad(-50), rad(20)]],
        # src/example/test_go_to.py:169-187
        [[0.0001, -0.2, -0.6599], [0, 0, 0]],
        [[0.38, -0.2, -0.28], [0, -np.pi / 2, 0]],
        [[0.66, -0.2, -0.0], [0, -np.pi / 2, 0]],
        [[0.30, -0.2, -0.28], [0.0, 0.0, np.pi / 3]],
        [[0.0, -0.85, -0.0], [-np.pi / 2, 0, 0]],
        [[0.0, -0.58, -0.28], [-np.pi / 2, -np.pi / 2, 0]],
        [[0.15, 0.35, -0.10], [np.pi / 3, -np.pi / 2, 0]],
        [[0.10, 0.20, -0.22], [np.pi / 3, -np.pi / 2, 0]],
        [[0.0, -0.2, -0.66], [0.0, 0.0, -np.pi / 3]],
        [[0.001, -0.2, -0.68], [0.0, 0.0, -np.pi / 3]],
        [[0.001, -0.2, -0.659], [0.0, np.pi / 2, 0.0]],
        [[0.38, -0.2, -0.28], [0.0, np.pi / 2, 0.0]],
        [[0.1, -0.2, 0.0], [0.0, np.pi, 0.0]],
        [[0.38, -0.2, -0.28], [0.0, 0.0, 0.0]],
        [[0.1, 0.2, -0.1], [0.0, -np.pi / 2, np.pi / 2]],
        [[0.0, -0.2, -0.66], [0, 0, 0]],
    ]
    r = np.array(r, dtype=np.float64)
    # left arm: the reference's own l_goal_poses (test_go_to.py:189-209) are the y / roll / yaw mirror
    l = r.copy()
    l[:, 0, 1] *= -1
    l[:, 1, 0] *= -1
    l[:, 1, 2] *= -1
    return {"r_arm": r, "l_arm": l}


def gen_symik_named():
    out = dict(META)
    for arm, poses in named_poses().items():
        with _Quiet():
            ik = SymbolicIK(arm=arm)
        flag, state, interval, joints, elbow = run_symik(ik, poses)
        th0 = np.zeros(len(poses))
        _, _, _, joints0, elbow0 = run_symik(ik, poses, th0)
        out.update({
            f"{arm}_poses": poses, f"{arm}_reachable": flag, f"{arm}_state": state, f"{arm}_interval": interval,
            f"{arm}_joints": joints, f"{arm}_elbow": elbow, f"{arm}_joints_theta0": joints0, f"{arm}_elbow_theta0": elbow0,
        })
    np.savez_compressed(os.path.join(HERE, "symik_named.npz"), **out)


def gen_symik_random(n_fk=3000, n_task=3000):
    for arm, seed in (("r_arm", 0), ("l_arm", 1)):
        M = np.concatenate([
            fk.sample_fk_poses(n_fk // 2, arm, seed=10 + seed, min_x=None),
            fk.sample_fk_poses(n_fk - n_fk // 2, arm, seed=20 + seed, min_x=0.05),
            fk.sample_task_space_poses(n_task, arm, seed=30 + seed),
        ])
        gp = np.array([euler_pose_from_matrix(m) for m in M])
        with _Quiet():
            ik = SymbolicIK(arm=arm)
        flag, state, interval, joints, elbow = run_symik(ik, gp)
        # a second theta per pose: a deterministic point inside the interval (or anywhere if unreachable)
        rng = np.random.default_rng(100 + seed)
        u = rng.uniform(0, 1, len(M))
        width = np.where(interval[:, 0] <= interval[:, 1], interval[:, 1] - interval[:, 0],
                         interval[:, 1] + 2 * np.pi - interval[:, 0])
        theta2 = np.where(flag, interval[:, 0] + u * width, 0.0)
        _, _, _, joints2, elbow2 = run_symik(ik, gp, theta2)
        out = dict(META, M=M, goal_pose=gp, reachable=flag, state=state, interval=interval, joints=joints, elbow=elbow,
                   theta2=theta2, joints_theta2=joints2, elbow_theta2=elbow2, n_fk=n_fk, n_task=n_task)
        np.savez_compressed(os.path.join(HERE, f"symik_random_{arm}.npz"), **golden_subset.symik_random(out, seed))
        print(arm, "symik_random: reachable", flag.mean(), "states", np.bincount(state, minlength=8))


GEOMETRY_PARAMETERS = {                    # an arm that is not Reachy's: unequal links, offset tip, tilted shoulder
    "r_shoulder_position": np.array([0.02, -0.22, 0.05]), "r_shoulder_orientation": [-12, 3, 8],
    "r_upper_arm_size": np.float64(0.30), "r_forearm_size": np.float64(0.25), "r_tip_position": np.array([0.01, -0.005, 0.12]),
    "l_shoulder_position": np.array([0.02, 0.22, 0.05]), "l_shoulder_orientation": [12, 3, -8],
    "l_upper_arm_size": np.float64(0.30), "l_forearm_size": np.float64(0.25), "l_tip_position": np.array([0.01, 0.005, 0.12]),
}
CTOR_VARIANTS = {                          # non-default SymbolicIK constructor arguments (symbolic_ik.py:26-37)
    "geometry": dict(ik_parameters=GEOMETRY_PARAMETERS),
    "limits": dict(elbow_limit=110, wrist_limit=np.float64(30.0)),
    "margins": dict(backward_limit=0.10, projection_margin=1e-6, normal_vector_margin=1e-3),
    "singularity": dict(singularity_offset=0.08, singularity_limit_coeff=0.7),
    "wide": dict(elbow_limit=140, wrist_limit=np.float64(55.0), backward_limit=-0.05, singularity_offset=-0.02,
                 singularity_limit_coeff=1.4),
}


def gen_symik_ctor(n_fk=900, n_task=900):
    """SymbolicIK with non-default limits / margins / singularity plane: flags, states, intervals, joints at
    theta_interval[0] and at a second theta inside the interval."""
    out = dict(META, variants=np.array(list(CTOR_VARIANTS)))
    for arm, seed in (("r_arm", 0), ("l_arm", 1)):
        M = np.concatenate([fk.sample_fk_poses(n_fk, arm, seed=110 + seed, min_x=0.0),
                            fk.sample_task_space_poses(n_task, arm, seed=120 + seed)])
        gp = np.array([euler_pose_from_matrix(m) for m in M])
        out.update({f"{arm}_M": M, f"{arm}_goal_pose": gp})
        for name, kw in CTOR_VARIANTS.items():
            with _Quiet():
                ik = SymbolicIK(arm=arm, **kw)
            flag, state, interval, joints, elbow = run_symik(ik, gp)
            rng = np.random.default_rng(130 + seed)
            u = rng.uniform(0, 1, len(M))
            width = np.where(interval[:, 0] <= interval[:, 1], interval[:, 1] - interval[:, 0],
                             interval[:, 1] + 2 * np.pi - interval[:, 0])
            theta2 = np.where(flag, interval[:, 0] + u * width, 0.0)
            _, _, _, joints2, elbow2 = run_symik(ik, gp, theta2)
            pre = f"{arm}_{name}_"
            # is_reachable_no_limits + get_joints(theta) on the first n_nl poses (symbolic_ik.py:85-119)
            n_nl = 500
            nl_th = np.random.default_rng(135 + seed).uniform(-np.pi, np.pi, n_nl)
            nl_j = np.full((n_nl, 7), np.nan); nl_e = np.full((n_nl, 3), np.nan)
            with _Quiet():
                for i in list(range(n_nl // 2)) + list(range(len(M) - n_nl // 2, len(M))):
                    k = i if i < n_nl // 2 else i - (len(M) - n_nl)
                    ok, _, fn = ik.is_reachable_no_limits(np.array(gp[i]))
                    assert ok
                    j, e = fn(nl_th[k])
                    nl_j[k], nl_e[k] = j, np.asarray(e)[:3]
            out.update({pre + "nl_theta": nl_th, pre + "nl_joints": nl_j, pre + "nl_elbow": nl_e})
            out.update({pre + "reachable": flag, pre + "state": state, pre + "interval": interval, pre + "joints": joints,
                        pre + "elbow": elbow, pre + "theta2": theta2, pre + "joints_theta2": joints2,
                        pre + "elbow_theta2": elbow2})
            print(arm, "symik_ctor", name, "reachable", flag.mean(), "states", np.bincount(state, minlength=8))
    np.savez_compressed(os.path.join(HERE, "symik_ctor.npz"), **golden_subset.symik_ctor(out))


def gen_symik_big_euler(n=800):
    """Goal orientations given as large euler angles (the same rotations shifted by multiples of 2 pi, and angles drawn
    in +-15 rad): the reference goes through scipy's from_euler, the kernels through their argument reduction."""
    out = dict(META)
    for arm, seed in (("r_arm", 0), ("l_arm", 1)):
        rng = np.random.default_rng(140 + seed)
        M = fk.sample_fk_poses(n, arm, seed=142 + seed, min_x=0.05)
        gp = np.array([euler_pose_from_matrix(m) for m in M])
        gp[:, 1, :] += 2 * np.pi * rng.integers(-3, 4, (n, 3))
        gp[n // 2:, 1, :] = rng.uniform(-15, 15, (n - n // 2, 3))
        with _Quiet():
            ik = SymbolicIK(arm=arm)
        flag, state, interval, joints, elbow = run_symik(ik, gp)
        out.update({f"{arm}_goal_pose": gp, f"{arm}_reachable": flag, f"{arm}_state": state, f"{arm}_interval": interval,
                    f"{arm}_joints": joints, f"{arm}_elbow": elbow})
        print(arm, "symik_big_euler: reachable", flag.mean(), "states", np.bincount(state, minlength=8))
    np.savez_compressed(os.path.join(HERE, "symik_big_euler.npz"), **out)


def gen_symik_elbow(n_fk=400, n_task=400, K=4):
    """get_elbow_position(theta) (symbolic_ik.py:684-695, returns [x, y, z, 1]) for K thetas per pose after is_reachable
    (whenever the intersection circle was stored, :197 -- also for "limited by wrist") AND after is_reachable_no_limits
    (:85-119, circle stored at :114-116); get_joints(theta, previous_joints) after is_reachable_no_limits with a non-zero
    previous_joints; the SHAPE of the elbow that get_joints returns: (4,) = get_elbow_position's homogeneous point, (3,)
    once make_elbow_projection fired (:708-714, returned at :863); and the solver attributes the calls leave behind
    (goal_pose / wrist_position after is_reachable, :143-171; after get_joints, :711-716)."""
    out = dict(META)
    named = named_poses()
    for arm, seed in (("r_arm", 0), ("l_arm", 1)):
        M = np.concatenate([fk.sample_fk_poses(n_fk, arm, seed=310 + seed, min_x=0.05),
                            fk.sample_task_space_poses(n_task, arm, seed=320 + seed)])
        gp = np.concatenate([np.array([euler_pose_from_matrix(m) for m in M]), named[arm]])
        n = len(gp)
        rng = np.random.default_rng(330 + seed)
        flag = np.zeros(n, bool)
        state = np.zeros(n, np.uint8)
        thetas = rng.uniform(-np.pi, np.pi, (n, K))
        thetas[:, K - 1] = rng.uniform(-9.0, 9.0, n)
        el_pos = np.full((n, K, 4), np.nan)          # get_elbow_position after is_reachable
        ir_goal = np.full((n, 3), np.nan)            # goal_pose[0] / wrist_position left by is_reachable
        ir_wrist = np.full((n, 3), np.nan)
        gj_joints = np.full((n, K, 7), np.nan)       # get_joints(theta_k) after a fresh is_reachable
        gj_elbow = np.full((n, K, 3), np.nan)
        gj_elbow_len = np.zeros((n, K), np.uint8)
        gj_goal = np.full((n, K, 3), np.nan)         # goal_pose[0] / wrist_position left by get_joints
        gj_wrist = np.full((n, K, 3), np.nan)
        nl_thetas = rng.uniform(-np.pi, np.pi, (n, K))
        nl_thetas[:, K - 1] = rng.uniform(-9.0, 9.0, n)
        nl_el_pos = np.full((n, K, 4), np.nan)       # get_elbow_position after is_reachable_no_limits
        nl_prev = rng.uniform(-2.0, 2.0, (n, 7))
        nl_joints = np.full((n, K, 7), np.nan)       # get_joints(theta_k, nl_prev) after a fresh is_reachable_no_limits
        nl_elbow = np.full((n, K, 3), np.nan)
        nl_elbow_len = np.zeros((n, K), np.uint8)
        with _Quiet():
            for i in range(n):
                g = np.array(gp[i])
                ik = SymbolicIK(arm=arm)             # fresh: attributes below are those THIS call set
                ok, itv, fn, st = ik.is_reachable(g.copy())
                flag[i] = ok
                state[i] = state_code(st)
                if st in ("reachable", "limited by wrist", "wrist out of range"):
                    ir_goal[i] = ik.goal_pose[0]
                    ir_wrist[i] = ik.wrist_position
                if st in ("reachable", "limited by wrist"):
                    if ok:
                        width = itv[1] - itv[0] if itv[0] <= itv[1] else itv[1] + 2 * np.pi - itv[0]
                        thetas[i, 0] = itv[0]
                        thetas[i, 1] = itv[0] + rng.uniform(0, 1) * width
                    for k in range(K):
                        e = ik.get_elbow_position(thetas[i, k])
                        assert e.shape == (4,)
                        el_pos[i, k] = e
                if ok:
                    for k in range(K):
                        ok2, _, fn2, _ = ik.is_reachable(g.copy())
                        j, e = fn2(thetas[i, k])
                        gj_joints[i, k] = j
                        gj_elbow[i, k] = np.asarray(e)[:3]
                        gj_elbow_len[i, k] = len(e)
                        gj_goal[i, k] = ik.goal_pose[0]
                        gj_wrist[i, k] = ik.wrist_position
                ok, _, fn = ik.is_reachable_no_limits(g.copy())
                assert ok
                for k in range(K):
                    nl_el_pos[i, k] = ik.get_elbow_position(nl_thetas[i, k])
                for k in range(K):
                    ok, _, fn = ik.is_reachable_no_limits(g.copy())
                    j, e = fn(nl_thetas[i, k], list(nl_prev[i]))
                    nl_joints[i, k] = j
                    nl_elbow[i, k] = np.asarray(e)[:3]
                    nl_elbow_len[i, k] = len(e)
        pre = arm + "_"
        out.update({pre + "goal_pose": gp, pre + "reachable": flag, pre + "state": state, pre + "thetas": thetas,
                    pre + "elbow_position": el_pos, pre + "ir_goal": ir_goal, pre + "ir_wrist": ir_wrist,
                    pre + "gj_joints": gj_joints, pre + "gj_elbow": gj_elbow, pre + "gj_elbow_len": gj_elbow_len,
                    pre + "gj_goal": gj_goal, pre + "gj_wrist": gj_wrist,
                    pre + "nl_thetas": nl_thetas, pre + "nl_elbow_position": nl_el_pos, pre + "nl_prev": nl_prev,
                    pre + "nl_joints": nl_joints, pre + "nl_elbow": nl_elbow, pre + "nl_elbow_len": nl_elbow_len})
        print(arm, "symik_elbow: reachable", flag.mean(), "projection fired (limits)", (gj_elbow_len[flag] == 3).mean(),
              "(no limits)", (nl_elbow_len == 3).mean(), "limited by wrist", (state == 4).mean())
    np.savez_compressed(os.path.join(HERE, "symik_elbow.npz"), **golden_subset.symik_elbow(out, n_fk, n_task))


def gen_ctl_ctor(n_variants=6):
    """ControlIK.previous_theta right after construction (control_ik.py:142-159): default arguments and random
    current_joints / current_pose, standard and DVT."""
    out = dict(META, n_variants=n_variants)
    rng = np.random.default_rng(400)
    variants = []
    for v in range(n_variants):
        cj = np.array([fk.sample_fk_joints(1, np.random.default_rng(410 + v))[0], fk.sample_fk_joints(1, np.random.default_rng(420 + v))[0]])
        cp = np.array([fk.forward_kinematics(cj[0][None], "r_arm")[0], fk.forward_kinematics(cj[1][None], "l_arm")[0]])
        if v == 0:                                  # identity rotations: the np.allclose snap of control_ik.py:142
            cp[:, :3, :3] = np.eye(3)
        variants.append((cj, cp))
        out[f"v{v}_current_joints"] = cj
        out[f"v{v}_current_pose"] = cp
    for tag, dvt in (("std", False), ("dvt", True)):
        with _Quiet():
            ctl = new_control(is_dvt=dvt)
        for arm in ("r_arm", "l_arm"):
            out[f"{tag}_default_{arm}"] = ctl.previous_theta[arm]
        for v, (cj, cp) in enumerate(variants):
            with _Quiet():
                ctl = ControlIK(current_joints=[list(cj[0]), list(cj[1])], current_pose=[cp[0], cp[1]], urdf_path="../config_files/reachy2.urdf",
                                is_dvt=dvt)
            for arm in ("r_arm", "l_arm"):
                out[f"{tag}_v{v}_{arm}"] = ctl.previous_theta[arm]
        print("ctl_ctor", tag, {k: float(out[k]) for k in out if k.startswith(tag)})
    np.savez_compressed(os.path.join(HERE, "ctl_ctor.npz"), **out)


def gen_api_surface():
    """Names, parameter names and defaults of the public methods of the reference's two classes (the drop-in boundary,
    SURVEY.md 8(b)) -> api_surface.json."""
    import inspect
    import json

    def describe(cls):
        out = {}
        for name, fn in inspect.getmembers(cls, predicate=inspect.isfunction):
            if name.startswith("_") and name != "__init__":
                continue
            sig = inspect.signature(fn)
            out[name] = [[p.name, None if p.default is inspect.Parameter.empty else repr(p.default)]
                         for p in sig.parameters.values()]
        return out

    with _Quiet():
        ik = SymbolicIK()
        ctl = new_control()
    surface = {"SymbolicIK": describe(SymbolicIK), "ControlIK": describe(ControlIK),
               "SymbolicIK_attributes": sorted(k for k in vars(ik) if not k.startswith("_")),
               "ControlIK_attributes": sorted(k for k in vars(ctl) if not k.startswith("_"))}
    with open(os.path.join(HERE, "api_surface.json"), "w") as f:
        json.dump(surface, f, indent=1, sort_keys=True)
    print("api_surface:", {k: len(v) for k, v in surface.items()})


def urdf_params():
    with open(URDF_PATH) as f:
        urdf = f.read()
    return get_ik_parameters_from_urdf(urdf, ["r", "l"])


def gen_symik_urdf(n=1500):
    """SymbolicIK as ControlIK configures it (URDF parameters, singularity_offset=-1.01) + no-limits path."""
    params = urdf_params()
    out = dict(META)
    for k, v in params.items():
        out["param_" + k] = np.asarray(v, dtype=np.float64)
    for arm, seed in (("r_arm", 0), ("l_arm", 1)):
        M = np.concatenate([fk.sample_fk_poses(n // 2, arm, seed=40 + seed, min_x=None),
                            fk.sample_task_space_poses(n - n // 2, arm, seed=50 + seed)])
        gp = np.array([euler_pose_from_matrix(m) for m in M])
        ik = SymbolicIK(arm=arm, ik_parameters=params, singularity_offset=-1.01, singularity_limit_coeff=1.0)
        flag, state, interval, joints, elbow = run_symik(ik, gp)
        # is_reachable_no_limits + get_joints(theta) for every pose (symbolic_ik.py:85-119)
        rng = np.random.default_rng(200 + seed)
        th = rng.uniform(-np.pi, np.pi, len(M))
        nl_joints = np.full((len(M), 7), np.nan)
        nl_elbow = np.full((len(M), 3), np.nan)
        for i, g in enumerate(gp):
            ok, _, fn = ik.is_reachable_no_limits(np.array(g))
            assert ok
            j, e = fn(th[i])
            nl_joints[i] = j
            nl_elbow[i] = np.asarray(e)[:3]
        out.update({f"{arm}_M": M, f"{arm}_goal_pose": gp, f"{arm}_reachable": flag, f"{arm}_state": state,
                    f"{arm}_interval": interval, f"{arm}_joints": joints, f"{arm}_elbow": elbow,
                    f"{arm}_nl_theta": th, f"{arm}_nl_joints": nl_joints, f"{arm}_nl_elbow": nl_elbow})
    np.savez_compressed(os.path.join(HERE, "symik_urdf.npz"), **out)


def new_control(is_dvt=False):
    with _Quiet():
        return ControlIK(urdf_path="../config_files/reachy2.urdf", is_dvt=is_dvt)


def run_discrete(ctl, arm, M, constrained_mode="unconstrained"):
    n = len(M)
    joints = np.zeros((n, 7))
    flag = np.zeros(n, bool)
    state = np.zeros(n, np.uint8)
    for i in range(n):
        j, ok, st = ctl.symbolic_inverse_kinematics(arm, M[i], "discrete", constrained_mode=constrained_mode)
        joints[i] = j
        flag[i] = ok
        state[i] = state_code(st)
        assert not ctl.emergency_stop
    return joints, flag, state


def gen_ctl_discrete(n_fk=1500, n_task=1000, n_k360=600, n_low=500, n_dvt=500):
    for arm, seed in (("r_arm", 0), ("l_arm", 1)):
        M = np.concatenate([fk.sample_fk_poses(n_fk, arm, seed=60 + seed, min_x=0.0),
                            fk.sample_task_space_poses(n_task, arm, seed=70 + seed)])
        # sprinkle identity / near-identity rotations to exercise the allclose() snap (control_ik.py:212)
        rng = np.random.default_rng(300 + seed)
        for k in range(0, 40):
            eps = 10.0 ** rng.uniform(-10, -4)
            e = rng.normal(size=3) * eps
            M[k, :3, :3] = R.from_euler("xyz", e).as_matrix() if k % 4 else np.eye(3)
        out = dict(META, M=M)
        ctl = new_control()
        j, f, s = run_discrete(ctl, arm, M)
        out.update(joints_k20=j, reachable_k20=f, state_k20=s)
        ctl = new_control()
        ctl.nb_search_points = 360
        j, f, s = run_discrete(ctl, arm, M[:n_k360])
        out.update(joints_k360=j, reachable_k360=f, state_k360=s)
        ctl = new_control()
        j, f, s = run_discrete(ctl, arm, M[:n_low], constrained_mode="low_elbow")
        out.update(joints_low=j, reachable_low=f, state_low=s)
        ctl = new_control(is_dvt=True)
        j, f, s = run_discrete(ctl, arm, M[:n_dvt])
        out.update(joints_dvt=j, reachable_dvt=f, state_dvt=s)
        np.savez_compressed(os.path.join(HERE, f"ctl_discrete_{arm}.npz"), **out)
        print(arm, "ctl_discrete: reachable", out["reachable_k20"].mean(), np.bincount(out["state_k20"], minlength=9))


class FakeTime:
    """Deterministic clock for control_ik.time: 1/120 s per call, starting far from 0 so that
    the first call sees the timeout (control_ik.py:296-304) and later calls never do."""

    def __init__(self):
        self.t = 1000.0

    def time(self):
        self.t += 1.0 / 120.0
        return self.t


def run_continuous(arm, Mtraj, is_dvt=False, current_joints=None, current_pose=None):
    """One fresh ControlIK per trajectory.  Returns joints (W,7), flag (W,), state (W,), emergency flag."""
    ctl = new_control(is_dvt=is_dvt)
    W = len(Mtraj)
    joints = np.zeros((W, 7))
    flag = np.zeros(W, bool)
    state = np.zeros(W, np.uint8)
    kw = {}
    if current_joints is not None:
        kw["current_joints"] = list(current_joints)
        kw["current_pose"] = np.array(current_pose)
    with _Quiet():
        for w in range(W):
            j, ok, st = ctl.symbolic_inverse_kinematics(arm, Mtraj[w], "continuous", **kw)
            joints[w] = j
            flag[w] = ok
            state[w] = state_code(st)
    return joints, flag, state, ctl.emergency_stop, ctl.previous_theta[arm]


def gen_ctl_continuous(T_sin=6, W=300):
    ref_control.time = FakeTime()
    for arm, seed in (("r_arm", 0), ("l_arm", 1)):
        Ms, q = fk.sinusoidal_trajectories(T_sin, W, arm, seed=80 + seed)
        trajs = [Ms[t] for t in range(T_sin)]
        kinds = ["sin"] * T_sin
        # trajectories that leave the workspace and come back (unreachable branch, control_ik.py:368-388)
        side = 1.0 if arm == "r_arm" else -1.0
        for k in range(2):
            s = np.linspace(0, 1, W)
            Mo = np.tile(np.eye(4), (W, 1, 1))
            ang = np.array([0.0, -np.pi / 2, 0.0]) + np.array([0.3 * side, 0.2, 0.4 * side]) * k
            Mo[:, :3, :3] = R.from_euler("xyz", ang).as_matrix()
            Mo[:, 0, 3] = 0.35 + 0.45 * np.sin(np.pi * s) ** 2
            Mo[:, 1, 3] = -0.25 * side + 0.1 * side * np.sin(2 * np.pi * s)
            Mo[:, 2, 3] = -0.25 + 0.15 * np.cos(2 * np.pi * s) * (k + 1)
            trajs.append(Mo)
            kinds.append("outreach")
        # a trajectory with a jump (continuity_check -> emergency stop, control_ik.py:395-400)
        Mj = Ms[0].copy()
        Mj[W // 2:] = Ms[1][W // 2:][::-1][: W - W // 2] if T_sin > 1 else Mj[W // 2:]
        Mj[W // 2:, :3, 3] += np.array([0.0, 0.25 * side, 0.3])
        trajs.append(Mj)
        kinds.append("jump")
        trajs = np.array(trajs)
        T = len(trajs)
        out = dict(META, M=trajs, kinds=np.array(kinds))
        J = np.zeros((T, W, 7)); F = np.zeros((T, W), bool); S = np.zeros((T, W), np.uint8)
        E = np.zeros(T, bool); TH = np.zeros(T)
        for t in range(T):
            J[t], F[t], S[t], E[t], TH[t] = run_continuous(arm, trajs[t])
        out.update(joints=J, reachable=F, state=S, emergency=E, final_theta=TH)
        # explicit current joints / pose on the (re)initialising call: start from the trajectory's own first sample
        J2 = np.zeros((T_sin, W, 7)); F2 = np.zeros((T_sin, W), bool); S2 = np.zeros((T_sin, W), np.uint8)
        E2 = np.zeros(T_sin, bool); TH2 = np.zeros(T_sin)
        for t in range(T_sin):
            J2[t], F2[t], S2[t], E2[t], TH2[t] = run_continuous(arm, trajs[t], current_joints=q[t, 0], current_pose=Ms[t, 0])
        out.update(cj_joints=J2, cj_reachable=F2, cj_state=S2, cj_emergency=E2, cj_final_theta=TH2,
                   cj_current_joints=q[:, 0], cj_current_pose=Ms[:, 0])
        # DVT mode (singularity_offset = 0.03: elbow projection + state leak inside the ternary search)
        nd = 3
        J3 = np.zeros((nd, W, 7)); F3 = np.zeros((nd, W), bool); S3 = np.zeros((nd, W), np.uint8)
        E3 = np.zeros(nd, bool); TH3 = np.zeros(nd)
        for t in range(nd):
            J3[t], F3[t], S3[t], E3[t], TH3[t] = run_continuous(arm, trajs[t], is_dvt=True)
        out.update(dvt_joints=J3, dvt_reachable=F3, dvt_state=S3, dvt_emergency=E3, dvt_final_theta=TH3)
        np.savez_compressed(os.path.join(HERE, f"ctl_continuous_{arm}.npz"), **out)
        print(arm, "ctl_continuous: emergency", E, "reachable frac", F.mean(axis=1))
    ref_control.time = time


OVERRIDE_VARIANTS = {                      # per-call keyword overrides of symbolic_inverse_kinematics (control_ik.py:162-172)
    "dth_big": dict(d_theta_max=0.05),
    "dth_small": dict(d_theta_max=0.002),
    "pref": dict(preferred_theta=-np.pi / 2),
    "low": dict(constrained_mode="low_elbow"),
    "low_pref_dth": dict(constrained_mode="low_elbow", preferred_theta=-5 * np.pi / 6, d_theta_max=0.03),
}
UNFREEZE_AT = (120, 125)                   # waypoints at which the "unfreeze" control type is sent


def gen_ctl_overrides(T=3, W=160, n_dis=600):
    """Per-call overrides (d_theta_max, preferred_theta, constrained_mode) in continuous and discrete mode, and the
    "unfreeze" control type after an emergency latch (control_ik.py:198-212, :262)."""
    ref_control.time = FakeTime()
    for arm, seed in (("r_arm", 0), ("l_arm", 1)):
        side = 1.0 if arm == "r_arm" else -1.0
        Ms, q = fk.sinusoidal_trajectories(T, W, arm, seed=90 + seed)
        # a trajectory that leaves the workspace and comes back: the unreachable branch uses the per-call preferred
        # theta (control_ik.py:373-379), the reachable branch the constructor's (:348)
        s = np.linspace(0, 1, W)
        Mo = np.tile(np.eye(4), (W, 1, 1))
        Mo[:, :3, :3] = R.from_euler("xyz", [0.2 * side, -np.pi / 2 + 0.1, 0.3 * side]).as_matrix()
        Mo[:, 0, 3] = 0.35 + 0.45 * np.sin(np.pi * s) ** 2
        Mo[:, 1, 3] = -0.25 * side + 0.1 * side * np.sin(2 * np.pi * s)
        Mo[:, 2, 3] = -0.25 + 0.15 * np.cos(2 * np.pi * s)
        trajs = np.concatenate([Ms, Mo[None]])
        Tn = len(trajs)
        out = dict(META, M=trajs, variants=np.array(list(OVERRIDE_VARIANTS)))
        for name, kw in OVERRIDE_VARIANTS.items():
            J = np.zeros((Tn, W, 7)); F = np.zeros((Tn, W), bool); S = np.zeros((Tn, W), np.uint8)
            E = np.zeros(Tn, bool); TH = np.zeros(Tn)
            for t in range(Tn):
                ctl = new_control()
                with _Quiet():
                    for w in range(W):
                        j, ok, st = ctl.symbolic_inverse_kinematics(arm, trajs[t, w], "continuous", **kw)
                        J[t, w], F[t, w], S[t, w] = j, ok, state_code(st)
                E[t], TH[t] = ctl.emergency_stop, ctl.previous_theta[arm]
            out.update({f"con_{name}_joints": J, f"con_{name}_reachable": F, f"con_{name}_state": S,
                        f"con_{name}_emergency": E, f"con_{name}_final_theta": TH})
            print(arm, "overrides continuous", name, "reachable", F.mean(axis=1), "emergency", E)
        # discrete mode with a per-call preferred theta
        Md = np.concatenate([fk.sample_fk_poses(n_dis - 200, arm, seed=94 + seed, min_x=0.0),
                             fk.sample_task_space_poses(200, arm, seed=96 + seed)])
        for name, kw in (("pref", dict(preferred_theta=-np.pi / 3)),
                         ("low_pref", dict(preferred_theta=-np.pi / 4, constrained_mode="low_elbow"))):
            ctl = new_control()
            J = np.zeros((n_dis, 7)); F = np.zeros(n_dis, bool); S = np.zeros(n_dis, np.uint8)
            with _Quiet():
                for i in range(n_dis):
                    j, ok, st = ctl.symbolic_inverse_kinematics(arm, Md[i], "discrete", **kw)
                    J[i], F[i], S[i] = j, ok, state_code(st)
            assert not ctl.emergency_stop
            out.update({f"dis_{name}_joints": J, f"dis_{name}_reachable": F, f"dis_{name}_state": S})
            print(arm, "overrides discrete", name, "reachable", F.mean())
        out["dis_M"] = Md
        # discrete mode from a multi-turn previous solution (allow_multiturn + the +-6 pi clamp / emergency of
        # multiturn_safety_check, utils.py:493-568) and explicit current_joints (returned for unreachable poses)
        prevs = np.array([[4 * np.pi + 0.3, 0.2 * side, -5.9 * np.pi, -1.0, 0.1, 0.1, 5.95 * np.pi],
                          [-5.97 * np.pi, -0.1 * side, 5.99 * np.pi, -0.5, -0.2, 0.3, -5.98 * np.pi]])
        cur = np.array([0.4, 0.3 * side, -0.2, -1.2, 0.05, -0.05, 7.0])
        nm = 300
        J = np.zeros((2, nm, 7)); F = np.zeros((2, nm), bool); S = np.zeros((2, nm), np.uint8); B = np.zeros((2, nm), np.uint8)
        for k in range(2):
            ctl = new_control()
            with _Quiet():
                for i in range(nm):
                    ctl.previous_sol[arm] = prevs[k].copy()
                    ctl.emergency_stop, ctl.emergency_state = False, ""
                    j, ok, st = ctl.symbolic_inverse_kinematics(arm, Md[i], "discrete", current_joints=cur.tolist())
                    J[k, i], F[k, i], S[k, i] = j, ok, state_code(st)
                    es = ctl.emergency_state
                    B[k, i] = (1 * ("shoulder pitch" in es)) | (2 * ("elbow yaw" in es)) | (4 * ("wrist yaw" in es))
                    assert ctl.emergency_stop == bool(B[k, i])
        out.update(dis_mt_prev=prevs, dis_mt_current=cur, dis_mt_joints=J, dis_mt_reachable=F, dis_mt_state=S, dis_mt_bits=B)
        print(arm, "overrides discrete multiturn: emergency bits", np.bincount(B.ravel(), minlength=8), "max |j|/pi",
              np.abs(J).max() / np.pi)
        # multi-turn trajectories: joint-space ramps of wrist yaw / elbow yaw / shoulder pitch through several turns
        # (allow_multiturn unwrapping; the +-6 pi clamp of multiturn_safety_check latches the emergency at the end)
        Wm = 260
        u = np.linspace(0.0, 1.0, Wm)[:, None]
        q0 = np.radians([-25.0, -40.0 * side, 0.0, -70.0, 0.0, 0.0, 0.0])
        ramps = np.array([[0, 0, 0, 0, 0, 0, 6.4 * np.pi],                        # wrist yaw up: clamp at +6 pi
                          [0, 0, -3.0 * np.pi * side, 0, 0, 0, -4.5 * np.pi],     # elbow yaw and wrist yaw, opposite senses
                          [2.5 * np.pi, 0, 0, 0, 0, 0, 3.0 * np.pi],              # shoulder pitch circles
                          [0, 0, 6.3 * np.pi * side, 0, 0, 0, 0]])                # elbow yaw to its clamp
        qm = q0[None, None, :] + u[None, :, :] * ramps[:, None, :]
        qm[..., 4] += 0.2 * np.sin(9 * u[None, :, 0]); qm[..., 5] += 0.15 * np.cos(7 * u[None, :, 0])
        Mm = fk.forward_kinematics(qm.reshape(-1, 7), arm).reshape(len(ramps), Wm, 4, 4)
        J = np.zeros((len(ramps), Wm, 7)); F = np.zeros((len(ramps), Wm), bool); S = np.zeros((len(ramps), Wm), np.uint8)
        E = np.zeros(len(ramps), bool); TH = np.zeros(len(ramps)); EW = np.full(len(ramps), -1)
        for t in range(len(ramps)):
            ctl = new_control()
            with _Quiet():
                for w in range(Wm):
                    j, ok, st = ctl.symbolic_inverse_kinematics(arm, Mm[t, w], "continuous")
                    J[t, w], F[t, w], S[t, w] = j, ok, state_code(st)
                    if ctl.emergency_stop and EW[t] < 0:
                        EW[t] = w
            E[t], TH[t] = ctl.emergency_stop, ctl.previous_theta[arm]
        out.update(mt_M=Mm, mt_q=qm, mt_joints=J, mt_reachable=F, mt_state=S, mt_emergency=E, mt_final_theta=TH,
                   mt_emergency_waypoint=EW)
        print(arm, "multi-turn continuous: max |j|/pi per joint", np.round(np.abs(J).max(axis=(0, 1)) / np.pi, 2),
              "emergency", E, "at", EW, "reachable", F.mean(axis=1))
        # emergency latch, then "unfreeze" (twice: the second one while not latched)
        Mj = Ms[0].copy()
        Mj[W // 2:, :3, :3] = Mj[W // 2:, :3, :3] @ np.diag([-1.0, -1.0, 1.0])   # half a turn about the tool axis
        ctl = new_control()
        J = np.zeros((W, 7)); F = np.zeros(W, bool); S = np.zeros(W, np.uint8); EM = np.zeros(W, bool)
        with _Quiet():
            for w in range(W):
                j, ok, st = ctl.symbolic_inverse_kinematics(arm, Mj[w], "unfreeze" if w in UNFREEZE_AT else "continuous")
                J[w], F[w], S[w], EM[w] = j, ok, state_code(st), ctl.emergency_stop
        out.update(unf_M=Mj, unf_joints=J, unf_reachable=F, unf_state=S, unf_emergency_after=EM,
                   unf_at=np.array(UNFREEZE_AT), unf_final_theta=ctl.previous_theta[arm])
        print(arm, "unfreeze: latched waypoints", int(EM.sum()), "first", int(np.argmax(EM)), "states", np.bincount(S, minlength=9))
        np.savez_compressed(os.path.join(HERE, f"ctl_overrides_{arm}.npz"), **out)
    ref_control.time = time


def example_matrices():
    """4x4 goal matrices that appear verbatim in the reference's examples (truncated decimals: not orthonormal)."""
    M_r = np.array([[-0.34159004, -0.90910326, -0.23842717, 0.15009035], [0.92063745, -0.3746924, 0.10969179, -0.36832501],
                    [-0.18905801, -0.18203536, 0.9649457, 0.05864802], [0.0, 0.0, 0.0, 1.0]])   # test_continuous_ik.py:345-357
    M_l = np.array([[-0.34159004, 0.90910326, -0.23842717, 0.15009035], [-0.92063745, -0.3746924, -0.10969179, 0.36832501],
                    [-0.18905801, 0.18203536, 0.9649457, 0.05864802], [0.0, 0.0, 0.0, 1.0]])    # test_continuous_ik.py:358-370
    M_g = np.array([[0.36861, 0.089736, -0.92524, 0.37213], [-0.068392, 0.99525, 0.069279, -0.028012],
                    [0.92706, 0.037742, 0.373, -0.38572], [0, 0, 0, 1.0]])                       # test_go_to.py:250-257
    M_g_r = M_g.copy()
    M_g_r[1, 3] *= -1; M_g_r[0, 1] *= -1; M_g_r[1, 0] *= -1; M_g_r[1, 2] *= -1; M_g_r[2, 1] *= -1   # its y-mirror for the r_arm
    return {"r_arm": np.array([M_r, M_g_r]), "l_arm": np.array([M_l, M_g])}


def gen_ctl_examples(W=40):
    """The debug matrices of src/example through SymbolicIK, ControlIK discrete and ControlIK continuous (the matrix held
    for W calls: the rate-limited theta walks from the initial theta toward its target)."""
    out = dict(META)
    for arm, Ms in example_matrices().items():
        gp = np.array([euler_pose_from_matrix(m) for m in Ms])
        with _Quiet():
            ik = SymbolicIK(arm=arm)
        flag, state, interval, joints, elbow = run_symik(ik, gp)
        out.update({f"{arm}_M": Ms, f"{arm}_goal_pose": gp, f"{arm}_sym_reachable": flag, f"{arm}_sym_state": state,
                    f"{arm}_sym_interval": interval, f"{arm}_sym_joints": joints, f"{arm}_sym_elbow": elbow})
        dj, df, ds = [], [], []
        for m in Ms:
            with _Quiet():
                j, f, st = run_discrete(new_control(), arm, m[None])
            dj.append(j[0]); df.append(f[0]); ds.append(st[0])
        out.update({f"{arm}_dis_joints": np.array(dj), f"{arm}_dis_reachable": np.array(df), f"{arm}_dis_state": np.array(ds)})
        cj, cf, cs, ce = [], [], [], []
        for m in Ms:
            j, f, st, emg, _ = run_continuous(arm, np.repeat(m[None], W, axis=0))
            cj.append(j); cf.append(f); cs.append(st); ce.append(emg)
        out.update({f"{arm}_con_joints": np.array(cj), f"{arm}_con_reachable": np.array(cf), f"{arm}_con_state": np.array(cs),
                    f"{arm}_con_emergency": np.array(ce)})
        print(arm, "examples: sym", state, "dis", ds, "con states", [np.unique(x).tolist() for x in cs], "emergency", ce)
    np.savez_compressed(os.path.join(HERE, "ctl_examples.npz"), **out)


def gen_task_space():
    """The reference's task_space_test sweep (src/benchmark/ik_comparison.py:137-181, default steps): flags and states
    of SymbolicIK.is_reachable on its 37 376 goal poses; the grid itself is rebuilt by workspace.task_space_grid."""
    from reachy2_symbolic_ik_b200 import workspace

    with _Quiet():
        ik = SymbolicIK()
    poses = workspace.task_space_grid(ik.shoulder_position)
    flag = np.zeros(len(poses), bool)
    state = np.zeros(len(poses), np.uint8)
    for i, gp in enumerate(poses):
        ok, _, _, st = ik.is_reachable(np.array(gp))
        flag[i] = ok
        state[i] = state_code(st)
    print("task space:", len(poses), "poses,", int(flag.sum()), "reachable, states", np.bincount(state, minlength=8))
    np.savez_compressed(os.path.join(HERE, "task_space.npz"), **META, n_poses=len(poses), reachable_packed=np.packbits(flag),
                        state=state, reachable_count=int(flag.sum()))


def gen_helpers(n=2000):
    """Pins of the scipy / utils helpers the kernels restate."""
    from reachy2_symbolic_ik.utils import (angle_diff, limit_orbita3d_joints, limit_theta_to_interval,
                                            rotation_matrix_from_vector)
    rng = np.random.default_rng(7)
    # matrix -> euler xyz (incl. gimbal lock and truncated / non-orthonormal matrices)
    e = rng.uniform(-np.pi, np.pi, (n, 3))
    e[:50, 1] = np.pi / 2
    e[50:100, 1] = -np.pi / 2
    e[100:150, 1] = np.pi / 2 - 10.0 ** rng.uniform(-12, -5, 50)
    Rm = R.from_euler("xyz", e).as_matrix()
    Rm[150:400] = np.round(Rm[150:400], 5)  # truncated like src/example/test_go_to.py:250-257
    Rm[400:500] += rng.normal(size=(100, 3, 3)) * 1e-9
    eul = R.from_matrix(Rm).as_euler("xyz")
    # orbita3d limit
    w = rng.uniform(-np.pi, np.pi, (n, 3))
    w[:100] *= 0.1
    w[100:120, 1] = 0.0
    w[120:125] = 0.0
    orb = np.array([limit_orbita3d_joints(list(x), np.deg2rad(42.5)) for x in w])
    # angle_diff / limit_theta_to_interval
    a = rng.uniform(-20, 20, n); b = rng.uniform(-20, 20, n)
    ad = np.array([angle_diff(x, y) for x, y in zip(a, b)])
    itv = rng.uniform(-np.pi, np.pi, (n, 2))
    th = rng.uniform(-10, 10, n)
    lt = np.array([limit_theta_to_interval(t, 0.0, i)[0] for t, i in zip(th, itv)])
    # rotation_matrix_from_vector incl. the isclose branches
    v = rng.normal(size=(n, 3))
    v[:20] = [1, 0, 0]; v[20:40] = [-1, 0, 0]
    v[40:80] = np.array([1, 0, 0]) + rng.normal(size=(40, 3)) * 10.0 ** rng.uniform(-10, -6, (40, 1))
    v[80:120] = np.array([-2, 0, 0]) + rng.normal(size=(40, 3)) * 10.0 ** rng.uniform(-10, -6, (40, 1))
    rm = np.array([rotation_matrix_from_vector(x) for x in v])
    np.savez_compressed(os.path.join(HERE, "helpers.npz"), **META, mat=Rm, mat_euler=eul, wrist_in=w, wrist_out=orb,
                        ad_a=a, ad_b=b, ad=ad, lt_theta=th, lt_interval=itv, lt_out=lt, rmfv_v=v, rmfv=rm)


def gen_legacy_theta(n_fk=120, n_task=60):
    """get_best_continuous_theta, the first version of the continuous policy (utils.py:130-217, still imported by
    src/example/placo/movement_memory.py:51 and test_limits.py:31), and tend_to_preferred_theta (utils.py:115-127):
    flag, theta and the debug text for reachable poses x previous thetas x step limits, with the solver's own
    get_elbow_position as the callback."""
    from reachy2_symbolic_ik.utils import get_best_continuous_theta, tend_to_preferred_theta
    out = dict(META)
    for arm, seed in (("r_arm", 0), ("l_arm", 1)):
        rng = np.random.default_rng(910 + seed)
        M = np.concatenate([fk.sample_fk_poses(n_fk, arm, seed=900 + seed, min_x=0.05), fk.sample_task_space_poses(n_task, arm, seed=905 + seed)])
        ik = SymbolicIK(arm=arm)
        preferred = -4 * np.pi / 6 if arm == "r_arm" else -np.pi + 4 * np.pi / 6
        rows, texts = [], []
        for m in M:
            gp = euler_pose_from_matrix(m)
            ok, interval, _, _ = ik.is_reachable(gp)
            if not ok:
                continue
            for prev, d in ((rng.uniform(-np.pi, np.pi), 0.01), (rng.uniform(-np.pi, np.pi), 0.6), (preferred + rng.uniform(-0.005, 0.005), 0.01),
                            ((interval[0] + interval[1]) / 2 + rng.uniform(-0.3, 0.3), 0.2)):
                flag, theta, text = get_best_continuous_theta(prev, interval, ik.get_elbow_position, d, preferred, arm, ik.singularity_offset,
                                                              ik.singularity_limit_coeff, ik.elbow_singularity_position)
                t_flag, t_theta = tend_to_preferred_theta(prev, interval, None, d, preferred)
                rows.append([*np.concatenate(gp), interval[0], interval[1], prev, d, preferred, float(flag), theta, float(t_flag), t_theta])
                texts.append(text)
        out[f"{arm}_rows"] = np.array(rows)
        out[f"{arm}_text"] = np.array(texts)
        out[f"{arm}_elbow_singularity_position"] = np.array(ik.elbow_singularity_position, dtype=np.float64)
        out[f"{arm}_singularity"] = np.array([ik.singularity_offset, ik.singularity_limit_coeff])
    out["columns"] = np.array(["x", "y", "z", "roll", "pitch", "yaw", "interval0", "interval1", "previous_theta", "d_theta_max", "preferred_theta",
                               "flag", "theta", "tend_flag", "tend_theta"])
    np.savez_compressed(os.path.join(HERE, "legacy_theta.npz"), **out)
    print("legacy_theta", {k: v.shape for k, v in out.items() if hasattr(v, "shape") and v.ndim})


if __name__ == "__main__":
    t0 = time.time()
    which = sys.argv[1:] or ["named", "random", "urdf", "discrete", "continuous", "helpers", "examples", "task_space", "overrides", "ctor", "big_euler", "elbow", "ctl_ctor", "api", "legacy"]
    if "named" in which:
        gen_symik_named()
    if "helpers" in which:
        gen_helpers()
    if "random" in which:
        gen_symik_random()
    if "urdf" in which:
        gen_symik_urdf()
    if "discrete" in which:
        gen_ctl_discrete()
    if "continuous" in which:
        gen_ctl_continuous()
    if "examples" in which:
        gen_ctl_examples()
    if "overrides" in which:
        gen_ctl_overrides()
    if "ctor" in which:
        gen_symik_ctor()
    if "big_euler" in which:
        gen_symik_big_euler()
    if "elbow" in which:
        gen_symik_elbow()
    if "ctl_ctor" in which:
        gen_ctl_ctor()
    if "api" in which:
        gen_api_surface()
    if "legacy" in which:
        gen_legacy_theta()
    if "task_space" in which:
        gen_task_space()
    print(f"done in {time.time() - t0:.1f}s")
