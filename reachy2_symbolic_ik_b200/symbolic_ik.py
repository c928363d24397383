"""``SymbolicIK`` -- drop-in for ``reachy2_symbolic_ik.symbolic_ik.SymbolicIK`` whose geometry
runs in the sm_100a CUDA library (``libr2ik.so``), plus batched entry points.

Reference interface mirrored here: constructor ``symbolic_ik.py:26-83``; ``is_reachable``
``:121-282``; ``is_reachable_no_limits`` ``:85-119``; ``get_joints`` ``:697-863``;
``get_elbow_position`` ``:684-695``.  A scalar call is ONE launch of a one-thread kernel
(``r2ik_symik_scalar_f64``: the query travels as a kernel parameter, the result record lands in mapped pinned
host memory) plus one stream synchronisation; there is no CPU code path.

Semantics that differ from the reference on purpose (SURVEY.md A.6.1): ``get_joints`` of the
reference mutates the solver when the elbow projection fires, so a second call on the same
solved pose returns different joints.  Here every ``get_joints`` / closure call is a fresh
solve of the last pose (the value the reference returns on its *first* call).
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import Any, NamedTuple, Optional, Tuple

import numpy as np

from . import _abi, _native
from .states import STATE_REACHABLE, STATE_STRINGS

_ZERO7 = [0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0]


@dataclass
class BatchResult:
    """Outputs of a batched solve.  Arrays are torch CUDA tensors when the input was a CUDA
    tensor, NumPy arrays otherwise."""

    reachable: Any        # (N,) bool
    theta_interval: Any   # (N, 2) float64, NaN when unreachable; [0] > [1] means wrapped
    state: Any            # (N,) uint8, see states.STATE_STRINGS
    joints: Any           # (N, 7) float64, NaN when unreachable
    elbow: Any            # (N, 3) float64
    n_escalated: Any = None   # precision="fp32" only: poses re-solved by the FP64 solver (int, or a CUDA int32 tensor)

    def state_strings(self):
        s = self.state
        if hasattr(s, "cpu"):
            s = s.cpu().numpy()
        return [STATE_STRINGS[int(c)] for c in s]


@dataclass
class SweepResult:
    """Outputs of ``SymbolicIK.get_joints_sweep_batch``: K elbow angles per pose.  torch CUDA tensors when the poses
    were a CUDA tensor, NumPy arrays otherwise."""

    reachable: Any        # (N,) bool
    state: Any            # (N,) uint8, see states.STATE_STRINGS
    theta_interval: Any   # (N, 2) float64, NaN when unreachable; [0] > [1] means wrapped
    thetas: Any           # (N, K) float64, the angles used; NaN when unreachable
    joints: Any           # (N, K, 7) float64, NaN when unreachable
    elbow: Any            # (N, K, 3) float64
    projected: Any        # (N, K) bool: make_elbow_projection fired at that angle


class BestThetaResult(NamedTuple):
    """Outputs of ``SymbolicIK.get_best_theta_to_current_joints_batch``.  torch CUDA tensors when the poses were a CUDA
    tensor, NumPy arrays otherwise."""

    reachable: Any        # (N,) bool
    state: Any            # (N,) uint8, see states.STATE_STRINGS
    theta: Any            # (N,) float64, NaN when unreachable
    joints: Any           # (N, 7) float64 (None without want_joints), NaN when unreachable


def _ptr(t) -> C.c_void_p:
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(None)


def _precision_dtype(torch, precision: str):
    if precision == "fp64":
        return torch.float64
    if precision == "fp32":
        return torch.float32
    raise ValueError(f"precision must be 'fp64' or 'fp32', got {precision!r}")


def normalise_poses(torch, poses, device, dtype=None):
    """Accept (N,4,4) / (N,16) homogeneous matrices or (N,2,3) / (N,6) reference goal poses, as
    NumPy, CPU tensor or CUDA tensor.  Returns (device tensor (N,k) of ``dtype`` (default float64), kind,
    was_cuda)."""
    dtype = torch.float64 if dtype is None else dtype
    was_cuda = hasattr(poses, "is_cuda") and poses.is_cuda
    if not hasattr(poses, "is_cuda"):
        poses = torch.from_numpy(np.ascontiguousarray(poses))
    if poses.dtype != dtype:
        poses = poses.to(dtype)
    shp = tuple(poses.shape)
    if len(shp) == 3 and shp[1:] == (4, 4) or len(shp) == 2 and shp[1] == 16:
        kind, k = _abi.POSE_MAT4, 16
    elif len(shp) == 3 and shp[1:] == (2, 3) or len(shp) == 2 and shp[1] == 6:
        kind, k = _abi.POSE_EULER6, 6
    elif (len(shp) == 3 and shp[1:] == (3, 4) or len(shp) == 2 and shp[1] == 12) and dtype == torch.float64:
        kind, k = _abi.POSE_MAT34, 12       # the 3x4 top of the homogeneous matrix: 96 useful bytes of its 128
    else:
        raise ValueError(f"poses must be (N,4,4), (N,16), (N,3,4), (N,12), (N,2,3) or (N,6); got {shp}")
    poses = poses.reshape(shp[0], k).contiguous()
    if not was_cuda:
        poses = poses.to(device, non_blocking=True)
    elif poses.data_ptr() % 16:
        poses = poses.clone()   # the C ABI reads poses with 128-bit loads
    return poses, kind, was_cuda


class SymbolicIK:
    def __init__(
        self,
        arm: str = "r_arm",
        ik_parameters: dict[str, Any] = {},
        elbow_limit: int = 127,
        wrist_limit: np.float64 = np.float64(42.5),
        projection_margin: float = 1e-8,
        backward_limit: float = 0.02,
        normal_vector_margin: float = 1e-7,
        singularity_offset: float = 0.03,
        singularity_limit_coeff: float = 1.0,
        device: Optional[int] = None,
    ) -> None:
        if ik_parameters == {}:
            print("Using default parameters")
            ik_parameters = _abi.DEFAULT_IK_PARAMETERS
        if arm not in ["r_arm", "l_arm"]:
            raise ValueError("arm should be either 'r_arm' or 'l_arm'")
        self.arm = arm
        n = arm[0]
        self.shoulder_position = ik_parameters[f"{n}_shoulder_position"]
        self.shoulder_orientation_offset = ik_parameters[f"{n}_shoulder_orientation"]
        self.upper_arm_size = ik_parameters[f"{n}_upper_arm_size"]
        self.forearm_size = ik_parameters[f"{n}_forearm_size"]
        self.tip_position = ik_parameters[f"{n}_tip_position"]
        self.torso_pose = np.array([0.0, 0.0, 0.0])
        self.projection_margin = projection_margin
        self.normal_vector_margin = normal_vector_margin
        self.backward_limit = backward_limit
        self.elbow_limit = elbow_limit
        self.wrist_limit = wrist_limit
        self.singularity_offset = singularity_offset
        self.singularity_limit_coeff = singularity_limit_coeff

        cfg = _abi.make_arm_config(arm, ik_parameters, elbow_limit, wrist_limit, projection_margin, backward_limit,
                                   normal_vector_margin, singularity_offset, singularity_limit_coeff)
        self._torch = _native.require_cuda()
        self._handle = _native.Handle(cfg, device)
        self._device = self._torch.device("cuda", self._handle.device)
        k = self._handle.constants
        self.gripper_size = np.float64(k.gripper_size)
        self.max_arm_length = np.float64(k.max_arm_length)
        self.shoulder_wrist_min_distance = np.float64(k.shoulder_wrist_min_distance)
        self.elbow_singularity_position = np.array(k.elbow_singularity_position[:])
        self.wrist_singularity_position = np.array(k.wrist_singularity_position[:])

        self._ctor = dict(arm=arm, ik_parameters=ik_parameters, elbow_limit=elbow_limit, wrist_limit=wrist_limit,
                          projection_margin=projection_margin, backward_limit=backward_limit,
                          normal_vector_margin=normal_vector_margin, singularity_offset=singularity_offset,
                          singularity_limit_coeff=singularity_limit_coeff)
        self._replicas: dict = {self._handle.device: self}

        # state of the scalar API: the last pose handed to is_reachable / is_reachable_no_limits (the reference
        # keeps the solved pose on the instance; here every later call re-solves from the pose as it was given)
        self.goal_pose: Optional[np.ndarray] = None
        self.wrist_position: Optional[np.ndarray] = None
        self.elbow_position: Optional[np.ndarray] = None
        self._pose_in: Optional[np.ndarray] = None
        self._no_limits = False
        self._scalar_query = _abi.ScalarQuery()
        self._scalar_pinned = None   # pinned (mapped) host record the scalar kernel writes, allocated on first use

    def replica(self, device: int) -> "SymbolicIK":
        """The same solver (same constructor arguments) bound to another CUDA device of this process; cached."""
        device = int(device)
        if device not in self._replicas:
            import contextlib
            import io

            with contextlib.redirect_stdout(io.StringIO()):   # the constructor prints like the reference's
                r = SymbolicIK(device=device, **self._ctor)
            r._replicas = self._replicas
            self._replicas[device] = r
        return self._replicas[device]

    # ------------------------------------------------------------------ batched API
    def is_reachable_batch(self, poses, theta=None, previous_joints=None, want_joints: bool = True,
                           precision: str = "fp64", devices=None) -> BatchResult:
        """``is_reachable`` + ``theta_to_joints_func(theta)`` for N poses in one launch.

        poses: (N,4,4) homogeneous matrices (converted like the reference's ControlIK front
        end, ``R.from_matrix(M[:3,:3]).as_euler("xyz")``) or (N,2,3)/(N,6) reference goal poses
        ``[[x,y,z],[roll,pitch,yaw]]``.  theta: None -> ``theta_interval[0]``; else (N,).
        precision: "fp64" (the correctness reference, 1e-9 rad) or "fp32" (the fast path: float32 poses in,
        float32 results out, within 1e-4 rad for >= 99.99 % of the poses and 3e-4 rad for all (include/r2ik.h); states are the FP64 path's because poses
        FP32 cannot decide are re-solved in FP64 -- their count is ``n_escalated``).
        devices: CUDA ordinals of this node to spread a HOST batch over -- contiguous slices of the batch, one
        H2D -> K1 -> D2H pipeline per device, no inter-GPU traffic (``is_reachable_batch_host``); results are NumPy arrays.
        """
        torch = self._torch
        dt = _precision_dtype(torch, precision)
        if devices is not None:
            if hasattr(poses, "is_cuda") and poses.is_cuda:
                raise ValueError("devices=[...] spreads a host batch; a CUDA tensor already lives on one device")
            if theta is not None or previous_joints is not None:
                raise ValueError("devices=[...] solves at theta_interval[0] with the default previous_joints")
            want = self.HOST_FIELDS if want_joints else ("reachable", "state", "interval")
            o = self.is_reachable_batch_host(poses, precision=precision, want=want, devices=devices)
            npy = lambda t: None if t is None else t.numpy()   # noqa: E731
            return BatchResult(o.reachable.numpy().astype(bool), npy(o.theta_interval), o.state.numpy(), npy(o.joints), npy(o.elbow))
        with torch.cuda.device(self._device):
            P, kind, was_cuda = normalise_poses(torch, poses, self._device, dt)
            n = P.shape[0]
            th = None
            if theta is not None:
                th = torch.as_tensor(theta).to(self._device, dt).reshape(n).contiguous()
            pj = None
            if previous_joints is not None:
                pj = torch.as_tensor(previous_joints).to(self._device, dt).reshape(7).contiguous()
            reach = torch.empty(n, dtype=torch.uint8, device=self._device)
            state = torch.empty(n, dtype=torch.uint8, device=self._device)
            interval = torch.empty((n, 2), dtype=dt, device=self._device)
            joints = torch.empty((n, 7), dtype=dt, device=self._device) if want_joints else None
            elbow = torch.empty((n, 3), dtype=dt, device=self._device) if want_joints else None
            n_esc = None
            if precision == "fp32":
                n_esc = torch.empty(1, dtype=torch.int32, device=self._device)
                self.solve_into_f32(P, kind, th, pj, reach, state, interval, joints, elbow, n_esc)
            else:
                self.solve_into(P, kind, th, pj, reach, state, interval, joints, elbow)
            res = BatchResult(reach.bool(), interval, state, joints, elbow, n_esc)
            if was_cuda:
                return res
            out = [None if x is None else x.cpu().numpy() for x in
                   (res.reachable, res.theta_interval, res.state, res.joints, res.elbow)]
            return BatchResult(*out, None if n_esc is None else int(n_esc.item()))

    def solve_into(self, poses_dev, kind, theta_dev, prev_dev, reach, state, interval, joints, elbow, stream=None):
        """Raw launch on device tensors (no allocation, asynchronous): the C-ABI call itself."""
        torch = self._torch
        s = torch.cuda.current_stream(self._device).cuda_stream if stream is None else stream
        rc = self._handle.lib.r2ik_symik_solve_f64(
            self._handle.h, kind, _ptr(poses_dev), _ptr(theta_dev), _ptr(prev_dev), C.c_int64(poses_dev.shape[0]),
            _ptr(reach), _ptr(state), _ptr(interval), _ptr(joints), _ptr(elbow), C.c_void_p(s))
        _native.check(rc, "r2ik_symik_solve_f64")

    def solve_into_f32(self, poses_dev, kind, theta_dev, prev_dev, reach, state, interval, joints, elbow, n_escalated=None,
                       stream=None, scratch=None):
        """Raw launch of the FP32 fast path on float32 device tensors (``r2ik_symik_solve_f32``).  ``n_escalated``: int32
        device tensor (1,) the call sets to the number of poses re-solved in FP64; ``scratch``: int32 device tensor of
        at least N entries (the list of those poses); both are allocated / cached here when omitted."""
        torch = self._torch
        n = poses_dev.shape[0]
        s = torch.cuda.current_stream(self._device).cuda_stream if stream is None else stream
        if scratch is None:   # one cached list per stream: calls on one stream are ordered, calls on two may overlap
            cache = self.__dict__.setdefault("_esc_scratch", {})
            scratch = cache.get(s)
            if scratch is None or scratch.numel() < n:
                scratch = cache[s] = torch.empty(max(n, 1), dtype=torch.int32, device=self._device)
        if n_escalated is None:
            n_escalated = torch.empty(1, dtype=torch.int32, device=self._device)
        rc = self._handle.lib.r2ik_symik_solve_f32(
            self._handle.h, kind, _ptr(poses_dev), _ptr(theta_dev), _ptr(prev_dev), C.c_int64(n),
            _ptr(reach), _ptr(state), _ptr(interval), _ptr(joints), _ptr(elbow), _ptr(scratch), _ptr(n_escalated),
            C.c_void_p(s))
        _native.check(rc, "r2ik_symik_solve_f32")

    # ------------------------------------------------------------------ host-buffer pipeline
    HOST_FIELDS = ("reachable", "state", "interval", "joints", "elbow")
    LEAN = ("state", "joints")   # 57 bytes per pose back: state == 0 <=> reachable (states.STATE_STRINGS)

    def alloc_host_outputs(self, n: int, precision: str = "fp64", want=None) -> BatchResult:
        """Pinned host output buffers for ``is_reachable_batch_host`` (reusable across calls); fields not in ``want``
        (default: all five) are None."""
        torch = self._torch
        dt = _precision_dtype(torch, precision)
        want = self.HOST_FIELDS if want is None else tuple(want)
        pin = lambda *shape, dtype: torch.empty(shape, dtype=dtype).pin_memory()   # noqa: E731
        return BatchResult(
            reachable=pin(n, dtype=torch.uint8) if "reachable" in want else None,
            theta_interval=pin(n, 2, dtype=dt) if "interval" in want else None,
            state=pin(n, dtype=torch.uint8),
            joints=pin(n, 7, dtype=dt) if "joints" in want else None,
            elbow=pin(n, 3, dtype=dt) if "elbow" in want else None)

    def is_reachable_batch_host(self, poses_host, out: Optional[BatchResult] = None, chunk: Optional[int] = None,
                                n_streams: int = 3, precision: str = "fp64", want=None, devices=None,
                                wait: bool = True) -> BatchResult:
        """Host-to-host batched solve: ``poses_host`` is a CPU tensor (N,16)/(N,4,4)/(N,6)/(N,2,3),
        ideally pinned; results land in ``out`` (pinned CPU tensors; ``reachable`` is uint8 0/1).
        The batch is cut into chunks that flow H2D -> K1 -> D2H on ``n_streams`` CUDA streams so the
        PCIe copies in both directions overlap the kernel.  Synchronous on return.

        precision="fp32": float32 poses and outputs (half the PCIe bytes), the FP32 fast path of K1.
        want: which of ("reachable", "state", "interval", "joints", "elbow") to compute and bring back (``state`` always
        is); the link is the bound of this call, so bytes are throughput: the reference's own input format (N,6) =
        48 B / pose with ``want=SymbolicIK.LEAN`` (state + joints = 57 B / pose) moves 105 B where (N,4,4) + all
        five outputs moves 226 B.
        devices: CUDA ordinals to spread the batch over (contiguous slices, one pipeline per device, no exchange);
        default = this solver's device only.
        wait=False: enqueue and return at once; ``out`` is complete after ``wait_host()`` (several calls -- both arms, the
        next batch -- can then share the link without a pipeline fill / drain gap between them)."""
        torch = self._torch
        dt = _precision_dtype(torch, precision)
        want = self.HOST_FIELDS if want is None else tuple(want)
        unknown = set(want) - set(self.HOST_FIELDS)
        if unknown:
            raise ValueError(f"unknown output fields {sorted(unknown)}; choose from {self.HOST_FIELDS}")
        if precision == "fp32" and "reachable" not in want:
            want = want + ("reachable",)     # r2ik_symik_solve_f32 always writes it
        chunk_auto = chunk is None
        if not hasattr(poses_host, "is_cuda"):
            poses_host = torch.from_numpy(np.ascontiguousarray(poses_host))
        if poses_host.is_cuda:
            raise ValueError("is_reachable_batch_host takes host poses; use is_reachable_batch for CUDA tensors")
        if poses_host.dtype != dt:
            poses_host = poses_host.to(dt)
        shp = tuple(poses_host.shape)
        k = 16 if shp[1:] in ((4, 4), (16,)) else 12 if shp[1:] in ((3, 4), (12,)) else 6
        if k == 6 and shp[1:] not in ((2, 3), (6,)) or k == 12 and precision != "fp64":
            raise ValueError(f"poses must be (N,4,4), (N,16), (N,2,3) or (N,6) -- or (N,3,4) / (N,12) in FP64; got {shp}")
        kind = {16: _abi.POSE_MAT4, 12: _abi.POSE_MAT34, 6: _abi.POSE_EULER6}[k]
        if chunk_auto:
            # measured on B200 / PCIe 5 (profiles/r2_experiments.md): when the results outweigh the poses the D2H stream is
            # the critical one and the first, exposed H2D copy should be short (64 k poses); otherwise 128 k-pose chunks
            out_cols = 2 * ("interval" in want) + 7 * ("joints" in want) + 3 * ("elbow" in want)
            chunk = (1 << 16 if out_cols > k else 1 << 17) * (1 if precision == "fp64" else 2)
        P = poses_host.reshape(shp[0], k)
        if not P.is_contiguous():
            P = P.contiguous()
        n = shp[0]
        if out is None:
            out = self.alloc_host_outputs(n, precision, want)
        else:   # the native pipeline addresses raw rows of these buffers
            for name, t, cols, tdt in (("reachable", out.reachable, 1, torch.uint8), ("state", out.state, 1, torch.uint8),
                                       ("interval", out.theta_interval, 2, dt), ("joints", out.joints, 7, dt), ("elbow", out.elbow, 3, dt)):
                if name != "state" and name not in want:
                    continue
                if (t is None or not hasattr(t, "is_cuda") or t.is_cuda or t.dtype != tdt or not t.is_contiguous()
                        or t.numel() != n * cols):
                    raise ValueError(f"out.{name} must be a contiguous CPU tensor of {n} x {cols} {tdt} (see alloc_host_outputs)")
        devices = [self._handle.device] if devices is None else [int(d) for d in devices]
        self._keep_alive = P          # the copies read it until wait_host()
        if len(devices) == 1 and devices[0] == self._handle.device:
            self._host_pipeline(P, kind, k, dt, precision, want, out, 0, n, chunk, n_streams, sync=wait)
            if not wait:
                self._pending = [(self, (chunk, n_streams, k, dt))]
            return out
        # one pipeline per device on its contiguous slice; everything is enqueued before anything is waited for
        from .workspace import shard_range

        solvers = [self.replica(d) for d in devices]
        for r, sv in enumerate(solvers):
            lo, hi = shard_range(n, r, len(solvers))
            sv._host_pipeline(P, kind, k, dt, precision, want, out, lo, hi, chunk, n_streams, sync=False)
        self._pending = [(sv, (chunk, n_streams, k, dt)) for sv in solvers]
        if wait:
            self.wait_host()
        return out

    def wait_host(self) -> None:
        """Block until the last ``is_reachable_batch_host(..., wait=False)`` has delivered its results."""
        for sv, key in self.__dict__.pop("_pending", []):
            sv._host_pipeline_wait(*key)
        self.__dict__.pop("_keep_alive", None)

    def _host_pipeline(self, P, kind, k, dt, precision, want, out, begin, end, chunk, n_streams, sync):
        """Enqueue rows [begin, end) on this solver's native pipeline (r2ik_pipeline_*: the chunk loop, the three
        streams and the staging buffers live in libr2ik.so)."""
        pipe = self._pipeline(chunk, n_streams, k, dt)
        esz = P.element_size()

        def at(t, cols):
            return C.c_void_p(None) if t is None else C.c_void_p(t.data_ptr() + begin * cols * t.element_size())

        w = set(want)
        args = (pipe.p, kind, C.c_void_p(P.data_ptr() + begin * k * esz), C.c_int64(end - begin),
                at(out.reachable if "reachable" in w else None, 1), at(out.state, 1),
                at(out.theta_interval if "interval" in w else None, 2), at(out.joints if "joints" in w else None, 7),
                at(out.elbow if "elbow" in w else None, 3))
        if precision == "fp32":
            _native.check_pipeline(pipe.lib.r2ik_pipeline_symik_f32(*args), "r2ik_pipeline_symik_f32")
        else:
            _native.check_pipeline(pipe.lib.r2ik_pipeline_symik_f64(*args), "r2ik_pipeline_symik_f64")
        if sync:
            pipe.wait()

    def _host_pipeline_wait(self, chunk, n_streams, k, dt):
        self._pipeline(chunk, n_streams, k, dt).wait()

    _PIPE_CACHE_MAX = 4   # distinct (chunk, slots) pipelines kept per solver (each owns device staging buffers)

    def _pipeline(self, chunk: int, n_streams: int, k: int = 16, dt=None):
        key = (int(chunk), int(n_streams))
        cache = getattr(self, "_pipe_cache", None)
        if cache is None:
            cache = self._pipe_cache = {}
        if key not in cache:
            while len(cache) >= self._PIPE_CACHE_MAX:      # bounded: the oldest pipeline's buffers are freed
                cache.pop(next(iter(cache)))
            cache[key] = _native.Pipeline(self._handle, chunk, max(2, n_streams))
        return cache[key]

    def clear_caches(self) -> None:
        """Drop the cached host-pipeline device buffers and FP32 scratch lists."""
        self.__dict__.pop("_pipe_cache", None)
        self.__dict__.pop("_esc_scratch", None)

    def is_reachable_no_limits_batch(self, poses, theta, previous_joints=None, with_projected: bool = False):
        """``is_reachable_no_limits`` + ``get_joints(theta, previous_joints)``: returns (joints (N,7), elbow (N,3)) and,
        with ``with_projected``, the (N,) bool "make_elbow_projection fired" (the reference's get_joints then returns a
        3-vector elbow instead of [x, y, z, 1]).  previous_joints: None (zeros), (7,) broadcast or (N,7)."""
        torch = self._torch
        with torch.cuda.device(self._device):
            P, kind, was_cuda = normalise_poses(torch, poses, self._device)
            n = P.shape[0]
            th = torch.as_tensor(theta, dtype=torch.float64).to(self._device).reshape(n).contiguous()
            pj, stride = None, 0
            if previous_joints is not None:
                pj = torch.as_tensor(previous_joints, dtype=torch.float64).to(self._device).contiguous()
                if pj.numel() == 7:
                    pj = pj.reshape(7)
                else:
                    pj, stride = pj.reshape(n, 7), 7
            joints = torch.empty((n, 7), dtype=torch.float64, device=self._device)
            elbow = torch.empty((n, 3), dtype=torch.float64, device=self._device)
            proj = torch.empty(n, dtype=torch.uint8, device=self._device) if with_projected else None
            s = torch.cuda.current_stream(self._device).cuda_stream
            rc = self._handle.lib.r2ik_symik_no_limits_f64(self._handle.h, kind, _ptr(P), _ptr(th), _ptr(pj), C.c_int32(stride),
                                                           C.c_int64(n), _ptr(joints), _ptr(elbow), _ptr(proj), C.c_void_p(s))
            _native.check(rc, "r2ik_symik_no_limits_f64")
            res = (joints, elbow) + ((proj.bool(),) if with_projected else ())
            return res if was_cuda else tuple(x.cpu().numpy() for x in res)

    def get_joints_sweep_batch(self, poses, thetas=None, n_samples: Optional[int] = None, previous_joints=None,
                               no_limits: bool = False) -> SweepResult:
        """``is_reachable`` (``is_reachable_no_limits`` with ``no_limits``) of each pose, then ``theta_to_joints_func`` at K
        elbow angles per pose, each as the first call on that solve -- the pose is solved once for its K angles.

        thetas: (N,K) angles per pose, or (1,K) one row shared by all poses.  n_samples: K angles per pose placed on its
        own theta_interval as ``get_best_discrete_theta`` places them (utils.py:366-375).  Give exactly one of the two.
        previous_joints: None (zeros) or (7,) broadcast.  A pose that is not reachable gets NaN angles, joints and
        elbows."""
        if (thetas is None) == (n_samples is None):
            raise ValueError("give either thetas (N,K) / (1,K) or n_samples, not both")
        torch = self._torch
        with torch.cuda.device(self._device):
            P, kind, was_cuda = normalise_poses(torch, poses, self._device)
            n = P.shape[0]
            th, stride = None, 0
            if thetas is not None:
                th = torch.as_tensor(thetas).to(self._device, torch.float64)
                if th.dim() != 2 or th.shape[0] not in (1, n) or th.shape[1] < 1:
                    raise ValueError(f"thetas must be (N,K) or (1,K) with N = {n}; got {tuple(th.shape)}")
                th = th.contiguous()
                K = th.shape[1]
                stride = K if th.shape[0] == n and n != 1 else 0
            else:
                K = int(n_samples)
                if K < 1:
                    raise ValueError(f"n_samples must be >= 1; got {n_samples}")
            pj = None
            if previous_joints is not None:
                pj = torch.as_tensor(previous_joints).to(self._device, torch.float64).reshape(7).contiguous()
            state = torch.empty(n, dtype=torch.uint8, device=self._device)
            interval = torch.empty((n, 2), dtype=torch.float64, device=self._device)
            used = torch.empty((n, K), dtype=torch.float64, device=self._device)
            joints = torch.empty((n, K, 7), dtype=torch.float64, device=self._device)
            elbow = torch.empty((n, K, 3), dtype=torch.float64, device=self._device)
            proj = torch.empty((n, K), dtype=torch.uint8, device=self._device)
            s = torch.cuda.current_stream(self._device).cuda_stream
            rc = self._handle.lib.r2ik_symik_sweep_f64(
                self._handle.h, kind, _ptr(P), C.c_int64(n), _ptr(th), C.c_int32(stride), C.c_int32(K),
                C.c_int32(int(bool(no_limits))), _ptr(pj), _ptr(state), _ptr(interval), _ptr(used), _ptr(joints),
                _ptr(elbow), _ptr(proj), C.c_void_p(s))
            _native.check(rc, "r2ik_symik_sweep_f64")
            res = SweepResult(state == STATE_REACHABLE, state, interval, used, joints, elbow, proj.bool())
            if was_cuda:
                return res
            return SweepResult(*(x.cpu().numpy() for x in (res.reachable, res.state, res.theta_interval, res.thetas,
                                                           res.joints, res.elbow, res.projected)))

    def get_best_theta_to_current_joints_batch(self, poses, current_joints, preferred_theta: Optional[float] = None,
                                               no_limits: bool = False, want_joints: bool = True) -> BestThetaResult:
        """``get_best_theta_to_current_joints`` (utils.py:267-331) for N poses: ``is_reachable`` (``is_reachable_no_limits``
        with ``no_limits``) of each pose, then the reference's search for the elbow angle whose joints are closest to that
        pose's current joints, on that solve and in the reference's order (so the state that ``get_joints`` leaks from
        one evaluation to the next when the elbow projection fires is part of the answer, as in the reference).

        current_joints: (7,) shared by all poses, or (N,7).  preferred_theta: the angle tried first; default ControlIK's
        for this arm (-2 pi / 3 for r_arm, -pi / 3 for l_arm).  joints: get_joints(theta) as the first call on a fresh
        solve of the pose, what ``is_reachable_batch(poses, theta)`` returns.  A pose that is not reachable gets NaN
        theta and joints."""
        if preferred_theta is None:
            preferred_theta = -4 * np.pi / 6 if self.arm == "r_arm" else -np.pi - (-4 * np.pi / 6)
        torch = self._torch
        with torch.cuda.device(self._device):
            P, kind, was_cuda = normalise_poses(torch, poses, self._device)
            n = P.shape[0]
            cj = torch.as_tensor(current_joints).to(self._device, torch.float64)
            if cj.shape == (7,) or cj.shape == (1, 7):
                stride = 0
            elif cj.dim() == 2 and cj.shape == (n, 7):
                stride = 7
            else:
                raise ValueError(f"current_joints must be (7,) or (N,7) with N = {n}; got {tuple(cj.shape)}")
            cj = cj.contiguous()
            state = torch.empty(n, dtype=torch.uint8, device=self._device)
            theta = torch.empty(n, dtype=torch.float64, device=self._device)
            joints = torch.empty((n, 7), dtype=torch.float64, device=self._device) if want_joints else None
            s = torch.cuda.current_stream(self._device).cuda_stream
            rc = self._handle.lib.r2ik_symik_best_theta_f64(
                self._handle.h, kind, _ptr(P), C.c_int64(n), _ptr(cj), C.c_int32(stride), C.c_double(float(preferred_theta)),
                C.c_int32(int(bool(no_limits))), _ptr(state), _ptr(theta), _ptr(joints), C.c_void_p(s))
            _native.check(rc, "r2ik_symik_best_theta_f64")
            res = BestThetaResult(state == STATE_REACHABLE, state, theta, joints)
            if was_cuda:
                return res
            return BestThetaResult(*(None if x is None else x.cpu().numpy() for x in res))

    def get_elbow_position_batch(self, poses, thetas, no_limits: bool = False, with_projected: bool = False):
        """``get_elbow_position`` for K thetas per pose after ``is_reachable`` (or ``is_reachable_no_limits``): (N,K,3),
        NaN where the reference would have stored no intersection circle (symbolic_ik.py:197, :114-116)."""
        torch = self._torch
        with torch.cuda.device(self._device):
            P, kind, was_cuda = normalise_poses(torch, poses, self._device)
            n = P.shape[0]
            th = torch.as_tensor(thetas, dtype=torch.float64).to(self._device).reshape(n, -1).contiguous()
            K = th.shape[1]
            out = torch.empty((n, K, 3), dtype=torch.float64, device=self._device)
            proj = torch.empty((n, K), dtype=torch.uint8, device=self._device) if with_projected else None
            s = torch.cuda.current_stream(self._device).cuda_stream
            rc = self._handle.lib.r2ik_elbow_positions_f64(self._handle.h, kind, _ptr(P), _ptr(th), C.c_int32(K), C.c_int64(n),
                                                           C.c_int32(int(bool(no_limits))), _ptr(out), _ptr(proj), C.c_void_p(s))
            _native.check(rc, "r2ik_elbow_positions_f64")
            res = (out, proj.bool()) if with_projected else (out,)
            res = res if was_cuda else tuple(x.cpu().numpy() for x in res)
            return res if with_projected else res[0]

    def reach_map(self, n: int = 256, orientations_euler=None, n_orientations: int = 512, **kw):
        """Workspace reachability map: int32 CUDA tensor (n,n,n) of per-voxel reachable-orientation
        counts (see ``workspace.reach_map``; all-reduced over ranks when ``dist=torch.distributed``)."""
        from . import workspace

        return workspace.reach_map(self, n=n, orientations_euler=orientations_euler, n_orientations=n_orientations, **kw)

    def task_space_test(self, arm_length: float = 0.5, precision: str = "fp64", **steps):
        """Batched form of the reference's ``task_space_test`` sweep (``src/benchmark/ik_comparison.py:137-181``):
        returns (goal_poses, BatchResult) for the position x Euler-angle grid (see ``workspace.task_space_grid``)."""
        from . import workspace

        return workspace.task_space_test(self, arm_length=arm_length, precision=precision, **steps)

    # ------------------------------------------------------------------ scalar API (reference signatures)
    def _scalar(self, no_limits: bool, theta=None, previous_joints=_ZERO7) -> np.void:
        """One launch of the one-thread kernel on the stored pose: query by value, record into mapped pinned memory."""
        torch = self._torch
        if self._scalar_pinned is None:
            self._scalar_pinned = torch.zeros(_abi.SCALAR_RESULT_DTYPE.itemsize, dtype=torch.uint8).pin_memory()
            self._scalar_view = self._scalar_pinned.numpy().view(_abi.SCALAR_RESULT_DTYPE)
        q = self._scalar_query
        q.goal_pose[:] = self._pose_in
        q.no_limits = int(no_limits)
        q.has_theta = int(theta is not None)
        q.theta = 0.0 if theta is None else float(theta)
        q.previous_joints[:] = [float(x) for x in previous_joints]
        lib = self._handle.lib
        stream = C.c_void_p(torch.cuda.current_stream(self._device).cuda_stream)
        _native.check(lib.r2ik_symik_scalar_f64(self._handle.h, C.byref(q), C.c_void_p(self._scalar_pinned.data_ptr()), stream),
                      "r2ik_symik_scalar_f64")
        _native.check(lib.r2ik_stream_synchronize(stream), "r2ik_stream_synchronize")
        return self._scalar_view[0].copy()

    def _store_pose(self, goal_pose, no_limits: bool) -> None:
        self._pose_in = np.concatenate([np.asarray(goal_pose[0], dtype=np.float64).reshape(3),
                                        np.asarray(goal_pose[1], dtype=np.float64).reshape(3)])
        self._no_limits = no_limits

    def _adopt_solved(self, goal_position, wrist_position) -> None:
        """self.goal_pose / self.wrist_position as the reference leaves them (symbolic_ik.py:143-171, 711-716)."""
        if not np.isnan(goal_position[0]):
            self.goal_pose = np.array([goal_position, self._pose_in[3:]])
            self.wrist_position = np.array(wrist_position)

    def is_reachable(self, goal_pose) -> Tuple[bool, np.ndarray, Optional[Any], str]:
        """Check if the goal pose ``[[x,y,z],[roll,pitch,yaw]]`` is reachable taking the wrist and
        elbow limits into account; returns (is_reachable, theta_interval, theta_to_joints_func, state)."""
        self._store_pose(goal_pose, False)
        r = self._scalar(False)
        self._adopt_solved(r["goal_position_solved"], r["wrist_position_solved"])
        state = STATE_STRINGS[int(r["state"])]
        if r["reachable"]:
            return True, np.array(r["interval"]), self.get_joints, state
        return False, np.array([]), None, state

    def is_reachable_no_limits(self, goal_pose) -> Tuple[bool, np.ndarray, Optional[Any]]:
        """Reachability without the wrist / elbow limits (unreachable goals are projected);
        always (True, [-pi, pi], get_joints) (symbolic_ik.py:85-119)."""
        self._store_pose(goal_pose, True)
        r = self._scalar(True)
        self._adopt_solved(r["goal_position_solved"], r["wrist_position_solved"])
        if r["reachable"]:
            return True, np.array([-np.pi, np.pi]), self.get_joints
        return False, np.array([]), None

    def get_joints(self, theta: float, previous_joints: list = _ZERO7) -> Tuple[np.ndarray, np.ndarray]:
        """Joints for the elbow angle theta on the last solved pose (fresh solve per call).  Like the reference, the
        elbow comes back as get_elbow_position's homogeneous [x, y, z, 1], and as a 3-vector once make_elbow_projection
        fired (symbolic_ik.py:708-714, returned at :863)."""
        if self._pose_in is None:
            raise AttributeError("get_joints called before is_reachable / is_reachable_no_limits")
        r = self._scalar(self._no_limits, theta, previous_joints)
        self._adopt_solved(r["goal_position"], r["wrist_position"])
        e = np.array(r["elbow"])
        self.elbow_position = e if r["projected"] else np.array([e[0], e[1], e[2], 1.0])
        return np.array(r["joints"]), self.elbow_position

    def get_elbow_position(self, theta: float) -> np.ndarray:
        """Elbow position [x, y, z, 1] on the intersection circle of the last solved pose (after ``is_reachable`` or
        ``is_reachable_no_limits``; symbolic_ik.py:684-695)."""
        if self._pose_in is None:
            raise AttributeError("get_elbow_position called before is_reachable")
        e = self._scalar(self._no_limits, theta)["elbow_on_circle"]
        return np.array([e[0], e[1], e[2], 1.0])
