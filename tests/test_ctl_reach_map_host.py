"""The controller's workspace map (r2ik_ctl_reach_map_u32) on the host: tests/hostsim/ctl_reach_map.cpp loops the item
functions of k_ctl_reach_map (ctl_map_rotation per orientation, ctl_reach_pair per pair) over a grid and an orientation
set, and this file holds it to the CPU oracle's discrete mode (oracle.ctl_discrete_batch) on the materialised poses
M(v, o) = [R_o | origin + (ix, iy, iz) * step]: accepted = the oracle's `reachable`, reachable = its state in
{REACHABLE, LIMITED_BY_SHOULDER}, pair by pair and summed per voxel.  The argument checks of the C entry are exercised
on libr2ik.so without a device."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from parity import REPO, Report, ill_conditioned_mask, load
from reachy2_symbolic_ik_b200 import _abi
from reachy2_symbolic_ik_b200.fk import fibonacci_orientations
from reachy2_symbolic_ik_b200.workspace import reach_grid, rpy_matrices

HS_DIR = os.path.join(REPO, "tests", "hostsim")
STANDARD, DVT = -1.01, 0.03   # ControlIK's singularity_offset without / with is_dvt
STATE_REACHABLE, STATE_LIMITED_BY_SHOULDER = 0, 6


@pytest.fixture(scope="module")
def cm(tmp_path_factory):
    """tests/hostsim/ctl_reach_map.cpp built with the harness's flags (tests/hostsim/Makefile) into a temporary directory."""
    out = str(tmp_path_factory.mktemp("hostsim_ctl_reach_map") / "libr2ik_hostsim_ctl_reach_map.so")
    subprocess.run(["g++", "-O2", "-fPIC", "-std=c++17", "-ffp-contract=off", "-Wall", "-Wno-unknown-pragmas", "-shared",
                    "-o", out, os.path.join(HS_DIR, "ctl_reach_map.cpp"), "-lm"], check=True, capture_output=True)
    return C.CDLL(out)


def urdf_params():
    u = load("symik_urdf.npz")
    return {k[len("param_"):]: u[k] for k in u.files if k.startswith("param_")}


def cfg_for(arm, singularity_offset):
    return _abi.make_arm_config(arm, urdf_params(), 127, 42.5, 1e-8, 0.02, 1e-7, singularity_offset, 1.0)


def ctl_params(oracle, arm, **kw):
    """R2ikCtlParams has the oracle's field layout; fill it from the oracle's ControlParams."""
    op = oracle.ControlParams(arm=arm, **kw)._c
    p = _abi.CtlParams()
    C.memmove(C.byref(p), C.byref(op), C.sizeof(p))
    return p


def orientation_set(n_fib=36):
    """Fibonacci orientations as matrices, plus the rotation routes of the controller's pose intake: exact identity, a
    rotation within np.allclose of identity (the snap), pitch +-pi/2 (the literal as_euler route) and a det < 0 block."""
    eps = 1e-9
    near = np.array([[1.0, 0.0, 0.0], [0.0, np.cos(eps), -np.sin(eps)], [0.0, np.sin(eps), np.cos(eps)]])
    extra = [np.eye(3), near, rpy_matrices([[0.3, np.pi / 2, -0.7]])[0], rpy_matrices([[-1.1, -np.pi / 2, 0.4]])[0],
             np.diag([1.0, 1.0, -1.0])]
    return np.concatenate([rpy_matrices(fibonacci_orientations(n_fib)), np.stack(extra)])


def grid_for(cm, cfg, n):
    pub = _abi.ArmConstants()
    cm.hs_arm_constants(C.byref(cfg), C.byref(pub))
    shoulder = np.array(cfg.shoulder_position[:])
    return reach_grid(shoulder, pub.max_arm_length, n)


def hs_map(cm, cfg, par, origin, step, dims, ori):
    dp = C.POINTER(C.c_double)
    nv = int(np.prod(dims))
    acc = np.zeros(nv, np.uint32); rea = np.zeros(nv, np.uint32); pairs = np.zeros((nv, len(ori)), np.uint8)
    o = np.ascontiguousarray(ori, dtype=np.float64).reshape(-1, 9)
    cm.hs_ctl_reach_map(C.byref(cfg), C.byref(par), origin.ctypes.data_as(dp), step.ctypes.data_as(dp),
                        dims.ctypes.data_as(C.POINTER(C.c_int32)), o.ctypes.data_as(dp), C.c_int32(len(o)),
                        acc.ctypes.data_as(C.POINTER(C.c_uint32)), rea.ctypes.data_as(C.POINTER(C.c_uint32)),
                        pairs.ctypes.data_as(C.POINTER(C.c_uint8)))
    return acc, rea, pairs


def materialise(origin, step, dims, ori):
    """M(v, o) as (nv * n_ori, 4, 4): positions as a multiply then an add, like the kernel."""
    ix, iy, iz = np.meshgrid(*(np.arange(int(d)) for d in dims), indexing="ij")
    idx = np.stack([ix, iy, iz], axis=-1).reshape(-1, 3).astype(np.float64)
    p = origin + idx * step
    nv, no = len(p), len(ori)
    M = np.zeros((nv, no, 4, 4))
    M[:, :, :3, :3] = ori[None]
    M[:, :, :3, 3] = p[:, None, :]
    M[:, :, 3, 3] = 1.0
    return M.reshape(nv * no, 4, 4)


CASES = [   # arm, singularity_offset, grid n, ControlParams overrides
    ("r_arm", STANDARD, 24, {}),
    ("l_arm", STANDARD, 16, {}),
    ("r_arm", DVT, 16, {}),
    ("l_arm", DVT, 24, {}),
    ("r_arm", STANDARD, 16, {"nb_search_points": 360}),
    ("l_arm", DVT, 16, {"nb_search_points": 360}),
    ("r_arm", DVT, 16, {"nb_search_points": 5}),
    ("l_arm", STANDARD, 16, {"nb_search_points": 5}),
    ("r_arm", STANDARD, 16, {"preferred_theta": -np.pi / 3}),
    ("l_arm", DVT, 16, {"preferred_theta": -np.pi / 3, "nb_search_points": 360}),
]


@pytest.mark.parametrize("arm,offset,n,kw", CASES,
                         ids=[f"{a}-{'dvt' if o == DVT else 'std'}-{n}-" + ("_".join(f"{k}{v:.3g}" for k, v in kw.items()) or "default")
                              for a, o, n, kw in CASES])
def test_ctl_reach_map_host_vs_oracle(cm, oracle, arm, offset, n, kw):
    cfg = cfg_for(arm, offset)
    par = ctl_params(oracle, arm, **kw)
    origin, step, dims = grid_for(cm, cfg, n)
    ori = orientation_set()
    acc, rea, pairs = hs_map(cm, cfg, par, origin, step, dims, ori)
    got_r, got_a = (pairs & 1).astype(bool), (pairs & 2).astype(bool)
    # the counts are the per-voxel sums of the pair verdicts, and accepted <= reachable pair by pair
    assert np.array_equal(acc, got_a.sum(axis=1)) and np.array_equal(rea, got_r.sum(axis=1))
    assert not (got_a & ~got_r).any()
    # the det < 0 block and the pairs whose pre-checks fail count nowhere; the special rotations are in the set
    assert not pairs[:, -1].any()
    assert got_r[:, -5:-1].any(), "no voxel reaches the identity / snap / gimbal-lock orientations"

    ocfg = oracle.arm_config(arm, ik_parameters=urdf_params(), singularity_offset=offset)
    opar = oracle.ControlParams(arm=arm, **kw)
    M = materialise(origin, step, dims, ori)
    _, want_a, want_s, _ = oracle.ctl_discrete_batch(ocfg, opar, M)
    want_r = (want_s == STATE_REACHABLE) | (want_s == STATE_LIMITED_BY_SHOULDER)
    want_a = want_a.reshape(pairs.shape); want_r = want_r.reshape(pairs.shape)
    mism = ((got_a != want_a) | (got_r != want_r)).reshape(-1)
    # exact except pairs the existing perturbation criterion classes ill-conditioned (only the mismatches are classed)
    ill = np.zeros(len(mism), bool)
    if mism.any():
        sub = M[mism]
        ill[mism] = ill_conditioned_mask(lambda p: oracle.ctl_discrete_batch(ocfg, opar, p.reshape(-1, 4, 4))[1:3],
                                         sub.reshape(len(sub), -1))
    rep = Report(f"hostsim ctl reach map {arm} off={offset} n={n} {kw}", len(mism), ill)
    rep.exact("accepted (pairs)", got_a.reshape(-1), want_a.reshape(-1))
    rep.exact("reachable (pairs)", got_r.reshape(-1), want_r.reshape(-1))
    rep.check(max_ill_fraction=0.02)
    ok_vox = ~ill.reshape(pairs.shape).any(axis=1)
    assert np.array_equal(acc[ok_vox], want_a.sum(axis=1)[ok_vox])
    assert np.array_equal(rea[ok_vox], want_r.sum(axis=1)[ok_vox])
    print(f"accepted {int(acc.sum())} / reachable {int(rea.sum())} of {pairs.size} pairs")
