"""Workspace reachability map (BASELINE.json configs[4]) and the multi-GPU partitioning helpers.

The reference has no such component; its closest code is the task-space grid sweep of
``src/benchmark/ik_comparison.py:137-181`` (``is_reachable`` over a position grid).  Here a
voxel grid x orientation set is swept by the K4 kernel (``r2ik_reach_map_u32``): counts[v] =
number of orientations for which ``SymbolicIK.is_reachable(voxel centre, orientation)`` is True.

``ctl_reach_map`` is the same sweep for ``ControlIK``'s discrete mode (``r2ik_ctl_reach_map_u32``): counts[v] = number
of orientations for which the controller accepts the pose, i.e. is_reachable holds AND an elbow angle passes
``is_elbow_ok`` (the preferred one or a sample of the search).

Multi-GPU: poses / trajectories are independent, so batches are cut into contiguous slices
(``shard_range``) with no exchange.  The reach map shards the ORIENTATION set; every rank counts its
shard for every voxel and the volumes are summed by an all-reduce (NCCL over NVLink / NVSwitch) -- the
only collective of the whole path.  Three things keep it off the critical path (``reach_map_sharded``):
only the x-range of the volume that can hold a reachable voxel is exchanged (the torso plane and the
reach sphere do not depend on the orientation, so the rest is zero on every rank), counts are 16 bits
on the wire, and the range is produced slab by slab so that the all-reduce of one slab overlaps the
kernel of the next.
"""
from __future__ import annotations

import ctypes as C
from typing import Callable, Optional, Tuple

import numpy as np

from . import _native
from .fk import fibonacci_orientations


def shard_range(n_items: int, rank: int, world: int) -> Tuple[int, int]:
    """Contiguous balanced slice [begin, end) of ``n_items`` owned by ``rank`` (first ``n % world``
    ranks get one extra item)."""
    if world <= 0 or not (0 <= rank < world):
        raise ValueError(f"bad rank/world {rank}/{world}")
    base, extra = divmod(int(n_items), world)
    begin = rank * base + min(rank, extra)
    return begin, begin + base + (1 if rank < extra else 0)


def reach_grid(shoulder_position, max_arm_length: float, n: int):
    """Cell-centred n^3 grid over the bounding cube of the reach sphere (shoulder +- max_arm_length)."""
    step = 2.0 * float(max_arm_length) / n
    origin = np.asarray(shoulder_position, dtype=np.float64) - float(max_arm_length) + step / 2
    return origin, np.array([step, step, step]), np.array([n, n, n], dtype=np.int32)


def sharded_sum(launch: Callable[[int, int], "object"], n_orientations: int, dist=None, group=None, mark=None):
    """Run ``launch(ori_begin, ori_end)`` on this rank's orientation slice and sum the returned
    count tensor over the ranks in place.  ``dist`` is ``torch.distributed`` (initialised) or None.
    ``mark``: optional callable invoked between the kernel and the collective (benchmarks record an event there)."""
    rank, world = 0, 1
    if dist is not None and dist.is_initialized():
        rank, world = dist.get_rank(group), dist.get_world_size(group)
    b, e = shard_range(n_orientations, rank, world)
    counts = launch(b, e)
    if mark is not None:
        mark()
    if world > 1:
        dist.all_reduce(counts, op=dist.ReduceOp.SUM, group=group)
    return counts


def live_x_range(solver, origin, step, dims, margin: int = 1) -> Tuple[int, int]:
    """Index range [lo, hi) along x outside which no voxel can be reachable for ANY orientation: the pre-checks of
    ``is_reachable`` (symbolic_ik.py:284-307) reject goals behind ``backward_limit`` and outside the reach sphere before
    the orientation is looked at.  ``margin`` indices are added on both sides (the device evaluates the same
    comparisons on ox + ix * sx; the margin makes the host-side range a superset whatever the rounding)."""
    x = origin[0] + np.arange(int(dims[0])) * step[0]
    sx = float(np.asarray(solver.shoulder_position, dtype=np.float64)[0])
    ok = (x >= solver.backward_limit) & (np.abs(x - sx) <= float(solver.max_arm_length))
    idx = np.nonzero(ok)[0]
    if len(idx) == 0:
        return 0, 0
    return max(0, int(idx[0]) - margin), min(int(dims[0]), int(idx[-1]) + 1 + margin)


def allreduce_u16_pairs(c16, v0: int, v1: int, dist, group=None):
    """Sum the 16-bit counts c16[v0:v1] (an int16 tensor; v0 even) over the ranks, two counts per int32 lane of the
    all-reduce: exact as long as no total exceeds 65 535 (no carry from the low half into the high one; the sign bit of
    the int16 storage is just the top count bit).  An odd tail takes the following (padding) element along.  Returns
    the async work handle."""
    v1e = v1 + (v1 - v0) % 2
    import torch

    lanes = c16[v0:v1e].view(torch.int32)
    return dist.all_reduce(lanes, op=dist.ReduceOp.SUM, group=group, async_op=True)


def reach_map_sharded(solver, ori, origin, step, dims, dist, group=None, out=None, n_slabs: int = 4, timing=None,
                      shard: str = "orientations"):
    """The map over several GPUs.  Returns the int32 volume (every rank holds the full map).

    Only the x-range of the volume that can hold a reachable voxel takes part (the rest is zero on every rank), counts are
    16 bits on the wire (two per int32 lane of the all-reduce) and the work is launched slab by slab so that the all-reduce
    of one slab overlaps the kernel of the next.  shard="orientations" (default, BASELINE.json's wording): each rank
    counts its slice of the orientation set for every voxel.  shard="voxels": each rank counts ALL orientations for every
    world-th row (ix, iy, :) of the volume and the all-reduce adds the disjoint pieces -- the per-voxel pre-checks are
    then divided by the number of ranks too, but the ranks end up less evenly loaded (the cost of a row depends on how
    many of its voxels and orientations pass the early range tests) and the step is the slowest rank's: measured
    5.66 / 3.07 / 1.90 ms against 5.59 / 2.99 / 1.75 ms for orientation shards on 2 / 4 / 8 GPUs (contiguous voxel
    ranges of equal chord length were 12 % out of balance).
    ``timing``: optional dict that receives CUDA events (``k``: per slab kernel, ``t0`` / ``t1`` around the call)."""
    torch = solver._torch
    dev = solver._device
    rank, world = dist.get_rank(group), dist.get_world_size(group)
    d0, d1, d2 = (int(d) for d in dims)
    plane = d1 * d2
    lo, hi = live_x_range(solver, origin, step, dims)
    if d2 % 2:               # two 16-bit counts per int32 lane: slab boundaries must sit on even element offsets
        lo, hi, n_slabs, shard = 0, d0, 1, "orientations"
    c16 = solver.__dict__.get("_reach_c16")
    if c16 is None or c16.numel() != d0 * plane + (d0 * plane) % 2 or c16.device != dev:
        c16 = solver._reach_c16 = torch.zeros(d0 * plane + (d0 * plane) % 2, dtype=torch.int16, device=dev)
    stream = torch.cuda.current_stream(dev)
    if timing is not None:
        timing["t0"] = torch.cuda.Event(enable_timing=True); timing["t0"].record(stream)
        timing["k"] = []
    if shard == "voxels":
        c16.zero_()                                   # the other ranks' rows (and the dead ranges) are zero here
        b, e, row_mod, row_rem = 0, ori.shape[0], world, rank
    else:
        b, e = shard_range(ori.shape[0], rank, world)
        row_mod, row_rem = 1, 0
        c16[:lo * plane].zero_()
        c16[hi * plane:].zero_()
    xe = [lo + (hi - lo) * k // n_slabs for k in range(n_slabs + 1)]
    slabs = [(x0 * plane, x1 * plane, x0 * plane, x1 * plane) for x0, x1 in zip(xe[:-1], xe[1:]) if x1 > x0]
    works = []
    dp = C.POINTER(C.c_double)
    for g0, g1, v0, v1 in slabs:
        if v1 > v0:
            if timing is not None:
                k0 = torch.cuda.Event(enable_timing=True); k0.record(stream)
            rc = solver._handle.lib.r2ik_reach_map_range_u16(
                solver._handle.h, origin.ctypes.data_as(dp), step.ctypes.data_as(dp), dims.ctypes.data_as(C.POINTER(C.c_int32)),
                C.c_void_p(ori.data_ptr()), C.c_int32(b), C.c_int32(e), C.c_int64(v0), C.c_int64(v1), C.c_int32(row_mod),
                C.c_int32(row_rem), C.c_void_p(c16.data_ptr()), C.c_void_p(stream.cuda_stream))
            _native.check(rc, "r2ik_reach_map_range_u16")
            if timing is not None:
                k1 = torch.cuda.Event(enable_timing=True); k1.record(stream)
                timing["k"].append((k0, k1))
        works.append(allreduce_u16_pairs(c16, g0, g1, dist, group))
    for w in works:
        w.wait()                                 # the current stream waits for the collective
    if out is None:
        out = torch.empty((d0, d1, d2), dtype=torch.int32, device=dev)
    out.view(-1).copy_(c16[:d0 * plane])
    if timing is not None:
        timing["t1"] = torch.cuda.Event(enable_timing=True); timing["t1"].record(stream)
        timing["exchanged_bytes"] = 2 * (hi - lo) * plane
        timing["shard"] = shard
    return out


def reach_map(solver, n: int = 256, orientations_euler=None, n_orientations: int = 512, origin=None, step=None,
              dims=None, dist=None, group=None, out=None, all_fp64: bool = False, mark=None, plain_allreduce: bool = False,
              timing=None, shard: str = "orientations"):
    """Reachability count volume of ``solver`` (a ``SymbolicIK``): int32 CUDA tensor (d0, d1, d2).

    orientations_euler: (n_ori, 3) xyz Euler angles (default: ``fibonacci_orientations(n_orientations)``).
    With an initialised ``torch.distributed`` passed as ``dist`` the orientation set is sharded over the
    ranks and the volume is all-reduced; every rank returns the full map.
    all_fp64: decide every (voxel, orientation) pair with the FP64 flag solve instead of the mixed-precision test with
    FP64 escalation (identical counts, slower: the cross-check).
    plain_allreduce: sum the full int32 volumes with one all-reduce after the kernel (the base form, kept as the
    cross-check of ``reach_map_sharded``)."""
    torch = solver._torch
    if orientations_euler is None:
        orientations_euler = fibonacci_orientations(n_orientations)
    if origin is None or step is None or dims is None:
        origin, step, dims = reach_grid(solver.shoulder_position, solver.max_arm_length, n)
    origin = np.ascontiguousarray(origin, dtype=np.float64)
    step = np.ascontiguousarray(step, dtype=np.float64)
    dims = np.ascontiguousarray(dims, dtype=np.int32)
    dev = solver._device
    with torch.cuda.device(dev):
        if hasattr(orientations_euler, "is_cuda"):
            ori = orientations_euler.to(dev, torch.float64).contiguous()
        else:
            ori = torch.from_numpy(np.ascontiguousarray(orientations_euler, dtype=np.float64)).to(dev)
        n_ori = ori.shape[0]
        sharded = dist is not None and dist.is_initialized() and dist.get_world_size(group) > 1
        if sharded and not all_fp64 and not plain_allreduce and n_ori <= 65535:
            return reach_map_sharded(solver, ori, origin, step, dims, dist, group, out, timing=timing, shard=shard)
        if out is None:
            out = torch.empty(tuple(int(d) for d in dims), dtype=torch.int32, device=dev)

        def launch(b: int, e: int):
            s = torch.cuda.current_stream(dev).cuda_stream
            entry = solver._handle.lib.r2ik_reach_map_f64_u32 if all_fp64 else solver._handle.lib.r2ik_reach_map_u32
            rc = entry(
                solver._handle.h, origin.ctypes.data_as(C.POINTER(C.c_double)), step.ctypes.data_as(C.POINTER(C.c_double)),
                dims.ctypes.data_as(C.POINTER(C.c_int32)), C.c_void_p(ori.data_ptr()), C.c_int32(b), C.c_int32(e),
                C.c_void_p(out.data_ptr()), C.c_void_p(s))
            _native.check(rc, "r2ik_reach_map_u32")
            return out

        return sharded_sum(launch, n_ori, dist, group, mark)


def rpy_matrices(euler) -> np.ndarray:
    """(n, 3) xyz Euler angles (roll, pitch, yaw) -> (n, 3, 3) rotation matrices Rz(yaw) Ry(pitch) Rx(roll): the
    vectorised ``fk._rpy_matrix``."""
    e = np.asarray(euler, dtype=np.float64).reshape(-1, 3)
    cr, sr = np.cos(e[:, 0]), np.sin(e[:, 0])
    cp, sp = np.cos(e[:, 1]), np.sin(e[:, 1])
    cy, sy = np.cos(e[:, 2]), np.sin(e[:, 2])
    R = np.empty((len(e), 3, 3))
    R[:, 0, 0] = cy * cp; R[:, 0, 1] = cy * sp * sr - sy * cr; R[:, 0, 2] = cy * sp * cr + sy * sr
    R[:, 1, 0] = sy * cp; R[:, 1, 1] = sy * sp * sr + cy * cr; R[:, 1, 2] = sy * sp * cr - cy * sr
    R[:, 2, 0] = -sp; R[:, 2, 1] = cp * sr; R[:, 2, 2] = cp * cr
    return R


def orientation_matrices(orientations) -> np.ndarray:
    """An orientation set as (n, 3, 3) float64 rotation matrices: (n, 3, 3) matrices are taken as given, (n, 3) xyz
    Euler angles go through ``rpy_matrices``."""
    o = orientations.detach().cpu().numpy() if hasattr(orientations, "detach") else np.asarray(orientations)
    o = np.asarray(o, dtype=np.float64)
    if o.ndim == 3 and o.shape[1:] == (3, 3):
        return np.ascontiguousarray(o)
    if o.ndim == 2 and o.shape[1] == 3:
        return rpy_matrices(o)
    raise ValueError(f"orientations must be (n, 3, 3) rotation matrices or (n, 3) xyz Euler angles, got {o.shape}")


def ctl_reach_map(controller, name: str, n: int = 256, orientations=None, n_orientations: int = 512,
                  preferred_theta: float = -4 * np.pi / 6, origin=None, step=None, dims=None, with_reachable: bool = False,
                  dist=None, group=None, out=None, mark=None):
    """The controller's workspace map (``r2ik_ctl_reach_map_u32``): for ``controller`` (a ``ControlIK``) and arm ``name``,
    the int32 CUDA volume (d0, d1, d2) of per-voxel counts of the orientations for which
    ``controller.symbolic_inverse_kinematics_batch(name, M, "discrete", preferred_theta=preferred_theta)`` returns
    reachable = True, M = [R_o | voxel centre].  Voxel centres are origin + (ix, iy, iz) * step (a multiply then an add,
    no fused multiply-add); the default grid is ``reach_grid`` with n cells per side.

    orientations: (n_ori, 3, 3) rotation matrices, or (n_ori, 3) xyz Euler angles (``rpy_matrices``); default
    ``fibonacci_orientations(n_orientations)``.  A block with det <= 0 counts nowhere.
    with_reachable: return (accepted, reachable), where reachable counts the orientations for which ``is_reachable``
    holds on the rotation the controller solves with (discrete state REACHABLE or LIMITED_BY_SHOULDER); reachable -
    accepted is the per-voxel "limited by shoulder" count.  Both come out of the same pass.
    The counts depend on the arm, the controller's solver (``is_dvt``), ``controller.nb_search_points`` and
    ``preferred_theta`` (mirrored for l_arm as in the batched call).  They do not depend on ``constrained_mode``,
    ``d_theta_max``, ``previous_joints`` or ``current_joints``, which in discrete mode only change the joints and the
    emergency bits, so they are not parameters here; the map describes a controller that is not latched by
    ``emergency_stop``.  Continuous mode never rejects a reachable pose and has no map of its own.
    dist: an initialised ``torch.distributed``; each rank counts its slice of the orientation set and one int32
    all-reduce sums the volumes (both at once when ``with_reachable``); every rank returns the full map.
    out: int32 CUDA tensor (2, d0, d1, d2) with ``with_reachable``, else (d0, d1, d2), reused for the result."""
    torch = controller._torch
    solver = controller.symbolic_ik_solver[name]
    par = controller._ctl_params(name, "unconstrained", preferred_theta, 0.01)
    if orientations is None:
        orientations = fibonacci_orientations(n_orientations)
    if origin is None or step is None or dims is None:
        origin, step, dims = reach_grid(solver.shoulder_position, solver.max_arm_length, n)
    origin = np.ascontiguousarray(origin, dtype=np.float64)
    step = np.ascontiguousarray(step, dtype=np.float64)
    dims = np.ascontiguousarray(dims, dtype=np.int32)
    shape = tuple(int(d) for d in dims)
    dev = solver._device
    with torch.cuda.device(dev):
        ori = torch.from_numpy(orientation_matrices(orientations).reshape(-1, 9)).to(dev)
        n_ori = ori.shape[0]
        want = (2,) + shape if with_reachable else shape
        if out is None:
            out = torch.empty(want, dtype=torch.int32, device=dev)
        elif tuple(out.shape) != want or out.dtype != torch.int32 or not out.is_contiguous() or out.device != dev:
            raise ValueError(f"out must be a contiguous int32 tensor of shape {want} on {dev}")
        acc = out[0] if with_reachable else out
        reach = out[1] if with_reachable else None
        dp = C.POINTER(C.c_double)

        def launch(b: int, e: int):
            s = torch.cuda.current_stream(dev).cuda_stream
            rc = solver._handle.lib.r2ik_ctl_reach_map_u32(
                solver._handle.h, C.byref(par), origin.ctypes.data_as(dp), step.ctypes.data_as(dp),
                dims.ctypes.data_as(C.POINTER(C.c_int32)), C.c_void_p(ori.data_ptr()), C.c_int32(b), C.c_int32(e),
                C.c_void_p(acc.data_ptr()), C.c_void_p(reach.data_ptr() if reach is not None else None), C.c_void_p(s))
            _native.check(rc, "r2ik_ctl_reach_map_u32")
            return out

        sharded_sum(launch, n_ori, dist, group, mark)
    return (acc, reach) if with_reachable else acc


def task_space_grid(shoulder_position, arm_length: float = 0.5, x_step: float = 0.15, y_step: float = 0.15,
                    z_step: float = 0.15, roll_step: int = 45, pitch_step: int = 45, yaw_step: int = 45) -> np.ndarray:
    """The goal poses of the reference's ``task_space_test`` (``src/benchmark/ik_comparison.py:137-170``): a position
    grid over the cube shoulder +- arm_length, kept where it lies inside the sphere of that radius and in front of the
    robot (x >= 0), crossed with an Euler-angle grid in degrees.  Returns (N, 2, 3) ``[[x, y, z], [roll, pitch, yaw]]``
    in the reference's loop order."""
    s = np.asarray(shoulder_position, dtype=np.float64)
    xs = np.arange(s[0] - arm_length, s[0] + arm_length + x_step, x_step)
    ys = np.arange(s[1] - arm_length, s[1] + arm_length + y_step, y_step)
    zs = np.arange(s[2] - arm_length, s[2] + arm_length + z_step, z_step)
    P = np.stack(np.meshgrid(xs, ys, zs, indexing="ij"), axis=-1).reshape(-1, 3)
    keep = ~((np.linalg.norm(P - s, axis=1) > arm_length) | (P[:, 0] < 0))
    P = P[keep]
    ang = [np.radians(np.arange(0, 360, st)) for st in (roll_step, pitch_step, yaw_step)]
    E = np.stack(np.meshgrid(*ang, indexing="ij"), axis=-1).reshape(-1, 3)
    out = np.empty((len(P), len(E), 2, 3))
    out[:, :, 0, :] = P[:, None, :]
    out[:, :, 1, :] = E[None, :, :]
    return out.reshape(-1, 2, 3)


def task_space_test(solver, arm_length: float = 0.5, precision: str = "fp64", **steps):
    """Batched ``task_space_test`` (``ik_comparison.py:137-181``): ``is_reachable`` on every pose of ``task_space_grid``
    in one launch.  Returns (goal_poses (N,2,3), BatchResult); ``int(result.reachable.sum())`` is the reference's
    "reachable poses" count."""
    poses = task_space_grid(solver.shoulder_position, arm_length, **steps)
    return poses, solver.is_reachable_batch(poses, want_joints=False, precision=precision)


def save_reach_map(path: str, counts, origin, step, orientations_euler, arm: str = "") -> None:
    """Write a reachability count volume with its grid (cell centres = origin + index * step) and orientation set to a
    compressed ``.npz``."""
    c = counts.cpu().numpy() if hasattr(counts, "cpu") else np.asarray(counts)
    np.savez_compressed(path, counts=c.astype(np.uint32), origin=np.asarray(origin, dtype=np.float64),
                        step=np.asarray(step, dtype=np.float64), orientations_euler=np.asarray(orientations_euler, dtype=np.float64),
                        arm=np.array(arm))


def load_reach_map(path: str) -> dict:
    """Read a volume written by ``save_reach_map``; adds ``fraction`` = counts / number of orientations."""
    with np.load(path, allow_pickle=False) as z:
        d = {k: z[k] for k in z.files}
    d["arm"] = str(d["arm"])
    d["fraction"] = d["counts"].astype(np.float64) / max(len(d["orientations_euler"]), 1)
    return d
