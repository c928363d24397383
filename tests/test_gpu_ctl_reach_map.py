"""GPU tests of the controller's workspace map (k_ctl_reach_map, r2ik_ctl_reach_map_u32, ControlIK.reach_map) against
ControlIK's discrete entry on the materialised poses M(v, o) = [R_o | origin + (ix, iy, iz) * step].  The two run the
same device functions on the same inputs, so no mismatch is allowed: accepted[v] = sum over o of the entry's
`reachable`, reachable[v] = sum over o of its state in {REACHABLE, LIMITED_BY_SHOULDER}."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ARMS = ("r_arm", "l_arm")
STATE_REACHABLE, STATE_LIMITED_BY_SHOULDER = 0, 6


@pytest.fixture(scope="module")
def controls():
    from reachy2_symbolic_ik_b200 import ControlIK

    return {False: ControlIK(urdf_path="../config_files/reachy2.urdf"),
            True: ControlIK(urdf_path="../config_files/reachy2.urdf", is_dvt=True)}


def grid(ctl, arm, n):
    from reachy2_symbolic_ik_b200 import workspace

    sv = ctl.symbolic_ik_solver[arm]
    return workspace.reach_grid(sv.shoulder_position, sv.max_arm_length, n)


def positions(origin, step, dims):
    """Voxel centres (nv, 3) as a multiply then an add, in the kernel's voxel order."""
    ix, iy, iz = np.meshgrid(*(np.arange(int(d)) for d in dims), indexing="ij")
    idx = np.stack([ix, iy, iz], axis=-1).reshape(-1, 3).astype(np.float64)
    return origin + idx * step


def materialise(P, R):
    """(nv * n_ori, 4, 4) CUDA tensor of [R_o | p_v], voxel-major."""
    import torch

    nv, no = len(P), len(R)
    M = torch.zeros((nv, no, 4, 4), dtype=torch.float64, device="cuda")
    M[:, :, :3, :3] = torch.from_numpy(np.ascontiguousarray(R)).cuda()[None]
    M[:, :, :3, 3] = torch.from_numpy(np.ascontiguousarray(P)).cuda()[:, None, :]
    M[:, :, 3, 3] = 1.0
    return M.reshape(nv * no, 4, 4)


def discrete_flags(ctl, arm, M, no, compact=None, **kw):
    """The discrete entry's (accepted, reachable) flags on M, shaped (nv, n_ori)."""
    _, reach, state, _ = ctl.symbolic_inverse_kinematics_batch(arm, M, "discrete", compact=compact, **kw)
    r = (state == STATE_REACHABLE) | (state == STATE_LIMITED_BY_SHOULDER)
    return reach.reshape(-1, no), r.reshape(-1, no)


def live_mask(ctl, arm, P):
    """Voxels some orientation could reach, with a margin: outside it both counts must be 0."""
    sv = ctl.symbolic_ik_solver[arm]
    d = np.linalg.norm(P - np.asarray(sv.shoulder_position), axis=1)
    return (d <= float(sv.max_arm_length) * (1 + 1e-9)) & (P[:, 0] >= sv.backward_limit - 1e-12)


def special_rotations():
    from reachy2_symbolic_ik_b200.workspace import rpy_matrices

    eps = 1e-9
    near = np.array([[1.0, 0.0, 0.0], [0.0, np.cos(eps), -np.sin(eps)], [0.0, np.sin(eps), np.cos(eps)]])
    return np.stack([np.eye(3), near, rpy_matrices([[0.3, np.pi / 2, -0.7]])[0], np.diag([1.0, 1.0, -1.0])])


@pytest.mark.parametrize("arm", ARMS)
@pytest.mark.parametrize("compact", [False, True])
def test_one_orientation_equals_discrete_entry(controls, arm, compact):
    """One orientation at a time: the volumes are the discrete entry's flags on the materialised poses, reshaped."""
    from reachy2_symbolic_ik_b200 import fk, workspace

    ctl = controls[False]
    origin, step, dims = grid(ctl, arm, 24)
    P = positions(origin, step, dims)
    R_all = np.concatenate([special_rotations(), workspace.rpy_matrices(fk.fibonacci_orientations(64)[[5, 40]])])
    for R in R_all:
        acc, rea = ctl.reach_map(arm, orientations=R[None], origin=origin, step=step, dims=dims, with_reachable=True)
        wa, wr = discrete_flags(ctl, arm, materialise(P, R[None]), 1, compact=compact)
        assert torch_equal(acc.reshape(-1), wa[:, 0]) and torch_equal(rea.reshape(-1), wr[:, 0])
        assert tuple(acc.shape) == tuple(int(d) for d in dims)
    # the det < 0 block counts nowhere
    acc, rea = ctl.reach_map(arm, orientations=R_all[3:4], origin=origin, step=step, dims=dims, with_reachable=True)
    assert int(acc.sum()) == 0 and int(rea.sum()) == 0


def torch_equal(counts, flags):
    return bool((counts.long() == flags.long()).all())


CASES = [(arm, dvt, K, pt) for arm in ARMS for dvt in (False, True) for K in (20, 360) for pt in (None,)] + \
        [("r_arm", False, 20, -np.pi / 3), ("l_arm", True, 360, -np.pi / 2)]


@pytest.mark.parametrize("arm,dvt,K,pt", CASES)
def test_volume_equals_summed_discrete_entry(controls, arm, dvt, K, pt):
    """32^3 voxels x 40 orientations: each volume is the per-voxel sum of the discrete entry's flags; accepted <=
    reachable everywhere and both are 0 outside the live voxels."""
    from reachy2_symbolic_ik_b200 import fk, workspace

    ctl = controls[dvt]
    kw = {} if pt is None else {"preferred_theta": pt}
    origin, step, dims = grid(ctl, arm, 32)
    P = positions(origin, step, dims)
    R = np.concatenate([workspace.rpy_matrices(fk.fibonacci_orientations(36)), special_rotations()])
    old = ctl.nb_search_points
    ctl.nb_search_points = K
    try:
        acc, rea = ctl.reach_map(arm, orientations=R, origin=origin, step=step, dims=dims, with_reachable=True, **kw)
        wa, wr = discrete_flags(ctl, arm, materialise(P, R), len(R), **kw)
        only_acc = ctl.reach_map(arm, orientations=R, origin=origin, step=step, dims=dims, **kw)
    finally:
        ctl.nb_search_points = old
    acc, rea = acc.reshape(-1), rea.reshape(-1)
    assert bool((acc.long() == wa.sum(dim=1)).all()), f"accepted: {int((acc.long() != wa.sum(dim=1)).sum())} voxels differ"
    assert bool((rea.long() == wr.sum(dim=1)).all()), f"reachable: {int((rea.long() != wr.sum(dim=1)).sum())} voxels differ"
    assert bool((only_acc.reshape(-1) == acc).all())
    assert bool((acc <= rea).all())
    dead = ~live_mask(ctl, arm, P)
    assert int(acc.cpu().numpy()[dead].sum()) == 0 and int(rea.cpu().numpy()[dead].sum()) == 0
    assert int(acc.sum()) > 0 and int(acc.sum()) < int(rea.sum())


def test_orientation_slices_add_up(controls):
    """Launches over slices of the orientation set (what each rank runs with dist=) add up to the whole set's volume."""
    import torch

    from reachy2_symbolic_ik_b200 import fk, workspace

    ctl = controls[True]
    arm = "l_arm"
    sv = ctl.symbolic_ik_solver[arm]
    origin, step, dims = grid(ctl, arm, 28)
    R = workspace.rpy_matrices(fk.fibonacci_orientations(45))
    whole_a, whole_r = ctl.reach_map(arm, orientations=R, origin=origin, step=step, dims=dims, with_reachable=True)
    ori = torch.from_numpy(R.reshape(-1, 9)).cuda()
    par = ctl._ctl_params(arm, "unconstrained", -4 * np.pi / 6, 0.01)
    dp = C.POINTER(C.c_double)
    dims32 = np.ascontiguousarray(dims, dtype=np.int32)
    tot_a = torch.zeros_like(whole_a); tot_r = torch.zeros_like(whole_r)
    for b, e in ((0, 7), (7, 7), (7, 30), (30, 45)):
        a = torch.full_like(whole_a, -1); r = torch.full_like(whole_r, -1)      # overwritten, not accumulated
        rc = sv._handle.lib.r2ik_ctl_reach_map_u32(
            sv._handle.h, C.byref(par), origin.ctypes.data_as(dp), step.ctypes.data_as(dp),
            dims32.ctypes.data_as(C.POINTER(C.c_int32)), C.c_void_p(ori.data_ptr()), C.c_int32(b), C.c_int32(e),
            C.c_void_p(a.data_ptr()), C.c_void_p(r.data_ptr()), C.c_void_p(torch.cuda.current_stream().cuda_stream))
        assert rc == 0
        if b == e:
            assert int(a.abs().sum()) == 0 and int(r.abs().sum()) == 0
        tot_a += a; tot_r += r
    assert torch.equal(tot_a, whole_a) and torch.equal(tot_r, whole_r)


def test_full_size_r_arm(controls):
    """256^3 voxels x 512 orientations (the default map): accepted <= reachable everywhere, and one x-plane (65 536
    voxels x 512 = 33.5 M poses) equals the discrete entry on its materialised poses."""
    import torch

    from reachy2_symbolic_ik_b200 import fk, workspace

    ctl = controls[False]
    arm = "r_arm"
    acc, rea = ctl.reach_map(arm, with_reachable=True)
    assert tuple(acc.shape) == (256, 256, 256)
    assert bool((acc <= rea).all()) and int(acc.sum()) > 0
    origin, step, dims = grid(ctl, arm, 256)
    R = workspace.rpy_matrices(fk.fibonacci_orientations(512))
    ix = 150
    x = origin[0] + float(ix) * step[0]
    ys = origin[1] + np.arange(256, dtype=np.float64) * step[1]
    zs = origin[2] + np.arange(256, dtype=np.float64) * step[2]
    P = np.stack([np.full(256 * 256, x), np.repeat(ys, 256), np.tile(zs, 256)], axis=1)
    wa, wr = discrete_flags(ctl, arm, materialise(P, R), 512)
    ga, gr = acc[ix].reshape(-1).long(), rea[ix].reshape(-1).long()
    assert int(ga.sum()) > 0
    assert bool((ga == wa.sum(dim=1)).all()), f"accepted: {int((ga != wa.sum(dim=1)).sum())} voxels differ"
    assert bool((gr == wr.sum(dim=1)).all()), f"reachable: {int((gr != wr.sum(dim=1)).sum())} voxels differ"
    del wa, wr
    torch.cuda.empty_cache()


def _sharded_worker(rank, world, port, tmp):
    import os
    import sys

    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    import torch
    import torch.distributed as dist

    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        from reachy2_symbolic_ik_b200 import ControlIK, fk

        ctl = ControlIK(urdf_path="../config_files/reachy2.urdf", device=rank)
        for n, n_ori in ((40, 37), (33, 64)):
            ori = fk.fibonacci_orientations(n_ori)
            single = ctl.reach_map("l_arm", n=n, orientations=ori, with_reachable=True)
            sharded = ctl.reach_map("l_arm", n=n, orientations=ori, with_reachable=True, dist=dist)
            assert torch.equal(sharded[0], single[0]) and torch.equal(sharded[1], single[1]), (n, n_ori)
            assert torch.equal(ctl.reach_map("l_arm", n=n, orientations=ori, dist=dist), single[0]), (n, n_ori)
        open(os.path.join(tmp, f"ok{rank}"), "w").write("ok")
    finally:
        dist.destroy_process_group()


def test_ctl_reach_map_two_gpus(tmp_path):
    """dist=torch.distributed over NCCL: orientation slices per rank, one int32 all-reduce -- equal to the single-GPU
    volumes on every rank."""
    import socket

    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp

    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    mp.spawn(_sharded_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    assert all((tmp_path / f"ok{r}").exists() for r in range(2))


def test_out_and_orientation_forms(controls):
    """Euler angles equal their matrices (rpy_matrices); `out` is reused; a bad orientation shape is refused."""
    import torch

    from reachy2_symbolic_ik_b200 import fk, workspace

    ctl = controls[False]
    e = fk.fibonacci_orientations(20)
    a = ctl.reach_map("r_arm", n=20, orientations=e)
    b = ctl.reach_map("r_arm", n=20, orientations=workspace.rpy_matrices(e))
    assert torch.equal(a, b)
    out = torch.empty((2, 20, 20, 20), dtype=torch.int32, device="cuda")
    acc, rea = ctl.reach_map("r_arm", n=20, orientations=e, with_reachable=True, out=out)
    assert acc.data_ptr() == out.data_ptr() and torch.equal(acc, a) and bool((acc <= rea).all())
    with pytest.raises(ValueError):
        ctl.reach_map("r_arm", n=20, orientations=np.zeros((4, 2)))
