"""``ControlIK`` -- drop-in for ``reachy2_symbolic_ik.control_ik.ControlIK`` on the CUDA library,
plus batched entry points (N poses in discrete mode, T trajectories x W waypoints in continuous
mode).  Reference: constructor ``control_ik.py:28-160``; ``symbolic_inverse_kinematics``
``:162-274``; continuous ``:276-407``; discrete ``:409-462``; ``safety_checks`` ``:464-497``.

All arithmetic (matrix -> euler front end with the identity snap, reachability, elbow-angle
policies, joints, safety chain) runs in the kernels; this module only keeps the controller
state dictionaries the reference keeps, and turns state codes back into its strings.
"""
from __future__ import annotations

import ctypes as C
import os
import time
from typing import Any, Dict, Tuple

import numpy as np

from . import _abi, _native
from .fk import bundled_urdf_path
from .states import STATE_EMERGENCY, STATE_INVALID_ROTATION, STATE_STRINGS, emergency_text
from .symbolic_ik import SymbolicIK, _ptr
from .urdf import get_ik_parameters_from_urdf

DEBUG = False

_DEFAULT_CURRENT_JOINTS = [
    [0.0, 0.2617993877991494, -0.17453292519943295, 0.0, 0.0, 0.0, 0.0],
    [0.0, -0.2617993877991494, 0.17453292519943295, 0.0, 0.0, 0.0, 0.0],
]
_DEFAULT_CURRENT_POSE = [
    np.array([[1, 0, 0, 0], [0, 1, 0, -0.2], [0, 0, 1, -0.66], [0, 0, 0, 1]]),
    np.array([[1, 0, 0, 0], [0, 1, 0, 0.2], [0, 0, 1, -0.66], [0, 0, 0, 1]]),
]


class ControlIK:
    def __init__(
        self,
        current_joints: list = _DEFAULT_CURRENT_JOINTS,
        current_pose: list = _DEFAULT_CURRENT_POSE,
        logger: Any = None,
        urdf: str = "",
        urdf_path: str = "",
        reachy_model: str = "full_kit",
        is_dvt: bool = False,
        device: int | None = None,
    ) -> None:
        self.symbolic_ik_solver: Dict[str, SymbolicIK] = {}
        self.last_call_t: Dict[str, float] = {}
        self.call_timeout = 0.2
        self.nb_search_points = 20
        self.emergency_state = ""
        self.emergency_stop = False
        self.init = True
        self.logger = logger
        if is_dvt:
            self.singularity_offset = 0.03
            if self.logger is not None:
                self.logger.info("DVT mode activated", throttle_duration_sec=0.1)
            else:
                print("DVT mode activated")
        else:
            self.singularity_offset = -1.01
        self.singularity_limit_coeff = 1.0
        self.preferred_theta: Dict[str, float] = {}
        self.previous_theta: Dict[str, float] = {}
        self.previous_sol: Dict[str, np.ndarray] = {}
        self.previous_pose: Dict[str, np.ndarray] = {}
        self.orbita3D_max_angle = np.deg2rad(42.5)

        if urdf_path == "" and urdf == "":
            raise ValueError("No URDF provided")
        if urdf_path != "" and urdf == "":
            full = os.path.join(os.path.dirname(__file__), urdf_path)
            if not os.path.isfile(full) and os.path.basename(urdf_path) == "reachy2.urdf":
                # the reference ships the robot description next to its package
                # ("../config_files/reachy2.urdf"); here the arm chains are bundled instead
                full = bundled_urdf_path()
            if os.path.isfile(full) and os.path.getsize(full) > 0:
                with open(full, "r") as f:
                    urdf = f.read()
            if urdf == "":
                raise ValueError("Empty URDF file")
        if reachy_model == "full_kit" or reachy_model == "headless":
            arms = ["r", "l"]
        elif reachy_model == "starter_kit_right":
            arms = ["r"]
        elif reachy_model == "starter_kit_left":
            arms = ["l"]
        elif reachy_model == "mini":
            arms = []
        else:
            raise ValueError(f"Unknown Reachy model {reachy_model}")
        try:
            ik_parameters = get_ik_parameters_from_urdf(urdf, arms)
        except Exception as e:
            raise ValueError(f"Error while parsing URDF: {e}")

        self._torch = _native.require_cuda() if arms else None
        self._device = None
        for prefix in arms:
            arm = f"{prefix}_arm"
            if ik_parameters != {}:
                self.symbolic_ik_solver[arm] = SymbolicIK(
                    arm=arm, ik_parameters=ik_parameters, singularity_offset=self.singularity_offset,
                    singularity_limit_coeff=self.singularity_limit_coeff, device=device)
            else:
                self.symbolic_ik_solver[arm] = SymbolicIK(
                    arm=arm, wrist_limit=np.rad2deg(self.orbita3D_max_angle), singularity_offset=self.singularity_offset,
                    singularity_limit_coeff=self.singularity_limit_coeff, device=device)
            self._device = self.symbolic_ik_solver[arm]._device
            preferred_theta = -4 * np.pi / 6
            k = 0 if prefix == "r" else 1
            self.preferred_theta[arm] = preferred_theta if prefix == "r" else -np.pi - preferred_theta
            self.previous_sol[arm] = np.array(current_joints[k], dtype=np.float64)
            self.previous_pose[arm] = np.array(current_pose[k], dtype=np.float64)
            self.previous_theta[arm] = self._initial_previous_theta(arm, current_joints)
            self.last_call_t[arm] = 0.0
        self._scalar_bufs: Dict[str, Any] = {}

    def _initial_previous_theta(self, arm: str, current_joints) -> float:
        """``previous_theta`` as the reference's constructor seeds it (control_ik.py:142-159): is_reachable_no_limits on
        the current pose, then the ternary search of ``get_best_theta_to_current_joints`` (utils.py:267-331) -- which
        receives the list of BOTH arms' joints there, so its cost runs over ``len(current_joints)`` rows, each
        broadcast against one joint (SURVEY.md A.6.11).  The value never reaches an output (discrete mode ignores
        it, continuous mode re-initialises on its first call); it is reproduced because it is a visible attribute.
        One launch of a one-thread kernel (``r2ik_ctl_ctor_theta_f64``), result in mapped pinned memory."""
        torch = self._torch
        solver = self.symbolic_ik_solver[arm]
        rows = np.ascontiguousarray([np.asarray(c, dtype=np.float64) for c in current_joints], dtype=np.float64).reshape(-1, 7)
        pose = np.ascontiguousarray(self.previous_pose[arm], dtype=np.float64).reshape(16)
        out = torch.zeros(1, dtype=torch.float64).pin_memory()
        dp = C.POINTER(C.c_double)
        lib = solver._handle.lib
        stream = C.c_void_p(torch.cuda.current_stream(self._device).cuda_stream)
        rc = lib.r2ik_ctl_ctor_theta_f64(solver._handle.h, C.c_double(self.preferred_theta[arm]), rows.ctypes.data_as(dp),
                                         C.c_int32(len(rows)), pose.ctypes.data_as(dp), C.c_void_p(out.data_ptr()), stream)
        _native.check(rc, "r2ik_ctl_ctor_theta_f64")
        _native.check(lib.r2ik_stream_synchronize(stream), "r2ik_stream_synchronize")
        theta = float(out[0])
        if np.isnan(theta):
            raise ValueError("Non-positive determinant (left-handed or null coordinate frame) in rotation matrix")
        return theta

    # ------------------------------------------------------------------ parameters
    def _ctl_params(self, name: str, constrained_mode: str, preferred_theta: float, d_theta_max: float) -> _abi.CtlParams:
        side = 1 if name.startswith("r") else -1
        if constrained_mode == "unconstrained":
            low = False
        elif constrained_mode == "low_elbow":
            low = True
        else:
            # the reference leaves interval_limit unbound here (UnboundLocalError)
            raise ValueError(f"Unknown constrained_mode {constrained_mode}")
        p = _abi.CtlParams()
        p.interval_limit[:] = _native.interval_limit(side, low)
        p.preferred_theta = preferred_theta if side > 0 else -np.pi - preferred_theta
        p.preferred_theta_ctor = self.preferred_theta[name]
        p.d_theta_max = d_theta_max
        p.orbita3d_max_angle = float(self.orbita3D_max_angle)
        p.nb_search_points = int(self.nb_search_points)
        p.nb_search_points_continuous = 10
        return p

    def reach_map(self, name: str, n: int = 256, orientations=None, n_orientations: int = 512, **kw):
        """The controller's workspace map for arm ``name``: int32 CUDA tensor (n,n,n) of per-voxel counts of the
        orientations that discrete mode accepts (``(accepted, reachable)`` with ``with_reachable=True``; see
        ``workspace.ctl_reach_map``; all-reduced over ranks when ``dist=torch.distributed``)."""
        from . import workspace

        return workspace.ctl_reach_map(self, name, n=n, orientations=orientations, n_orientations=n_orientations, **kw)

    def _dev(self, x, shape=None):
        torch = self._torch
        t = torch.as_tensor(np.ascontiguousarray(x, dtype=np.float64) if not hasattr(x, "is_cuda") else x,
                            dtype=torch.float64).to(self._device)
        if shape is not None:
            t = t.reshape(shape)
        return t.contiguous()

    # ------------------------------------------------------------------ batched API
    def symbolic_inverse_kinematics_batch(self, name: str, M, control_type: str = "discrete", current_joints=None,
                                          constrained_mode: str = "unconstrained", current_pose=None,
                                          d_theta_max: float = 0.01, preferred_theta: float = -4 * np.pi / 6,
                                          previous_joints=None, states=None, out=None, phased: bool = True,
                                          exhaustive: bool = False, devices=None, compact=None,
                                          _test_force_serial_mod: int = 0):
        """Batched ``symbolic_inverse_kinematics``.

        discrete:   M (N,4,4) -> joints (N,7), reachable (N,), state (N,) uint8, emergency bits (N,).
                    Every pose is solved against the same previous solution (``previous_joints``,
                    default ``self.previous_sol[name]``), like N independent reference calls.
        continuous: M (T,W,4,4) -> joints (T,W,7), reachable (T,W), state (T,W), states (T,) structured
                    array (``_abi.TRAJ_STATE_DTYPE``) that can be passed back to resume the trajectories.
                    ``states`` may also be a CUDA uint8 tensor (T,80): it is then updated in place and
                    returned as is (no host round trip).
        ``out``: the tuple a previous call returned for CUDA input of the same shape; its tensors are reused.
        ``exhaustive`` (discrete): False = the elbow search finds the arg-min over the nb_search_points samples from
        the crossings of the two elbow tests (cost independent of K); True = every sample is visited by the
        warp-cooperative scan kernel.  Same outputs.
        ``compact`` (discrete): True = the three dense passes over compacted index lists
        (``r2ik_ctl_discrete_compact_f64``; 80 bytes of device scratch per pose, allocated here), False = the single
        kernel, None = by batch size (``COMPACT_MIN_POSES``).  Same outputs.
        ``phased`` (continuous): True = per-waypoint kernels + per-trajectory scans, the finish pass on winding codes
        (``r2ik_ctl_continuous_phased_f64``; needs 10 bytes of device scratch per waypoint, allocated here); False = the single
        one-thread-per-trajectory kernel (the cross-check).  Same flags / states; joints equal to rounding.
        ``devices``: CUDA ordinals of this node to spread a HOST batch over (contiguous slices of the poses / of the
        trajectories, one pipeline per device, no inter-GPU traffic); results are NumPy arrays.
        """
        if devices is not None:
            return self._batch_on_devices(name, M, control_type, devices, current_joints=current_joints,
                                          constrained_mode=constrained_mode, current_pose=current_pose, d_theta_max=d_theta_max,
                                          preferred_theta=preferred_theta, previous_joints=previous_joints, states=states)
        torch = self._torch
        solver = self.symbolic_ik_solver[name]
        par = self._ctl_params(name, constrained_mode, preferred_theta, d_theta_max)
        was_cuda = hasattr(M, "is_cuda") and M.is_cuda
        with torch.cuda.device(self._device):
            stream = C.c_void_p(torch.cuda.current_stream(self._device).cuda_stream)
            Md = self._dev(M)
            if control_type == "discrete":
                n = Md.shape[0]
                Md = Md.reshape(n, 16)
                prev = self._dev(self.previous_sol[name] if previous_joints is None else previous_joints, (7,))
                cur = prev if current_joints is None else self._dev(current_joints, (7,))
                if out is not None and was_cuda:
                    joints, reach, state, emg = out[0], out[1].view(torch.uint8), out[2], out[3]
                else:
                    joints = torch.empty((n, 7), dtype=torch.float64, device=self._device)
                    reach = torch.empty(n, dtype=torch.uint8, device=self._device)
                    state = torch.empty(n, dtype=torch.uint8, device=self._device)
                    emg = torch.empty(n, dtype=torch.uint8, device=self._device)
                lib = solver._handle.lib
                if compact is None:
                    compact = n >= self.COMPACT_MIN_POSES
                if compact and not exhaustive and n > 0:
                    nbytes = lib.r2ik_ctl_discrete_workspace_bytes(C.c_int64(n))
                    ws = self._scratch((nbytes + 7) // 8, stream.value)
                    rc = lib.r2ik_ctl_discrete_compact_f64(solver._handle.h, C.byref(par), _ptr(Md), C.c_int64(n), _ptr(prev),
                                                           _ptr(cur), _ptr(joints), _ptr(reach), _ptr(state), _ptr(emg),
                                                           _ptr(ws), C.c_int64(ws.numel() * 8), stream)
                    _native.check(rc, "r2ik_ctl_discrete_compact_f64")
                else:
                    entry = lib.r2ik_ctl_discrete_scan_f64 if exhaustive else lib.r2ik_ctl_discrete_f64
                    rc = entry(solver._handle.h, C.byref(par), _ptr(Md), C.c_int64(n),
                               _ptr(prev), _ptr(cur), _ptr(joints), _ptr(reach), _ptr(state), _ptr(emg), stream)
                    _native.check(rc, "r2ik_ctl_discrete_f64")
                res = (joints, reach.view(torch.bool), state, emg)
                return res if was_cuda else tuple(x.cpu().numpy() for x in res)
            if control_type == "continuous":
                T, W = Md.shape[0], Md.shape[1]
                Md = Md.reshape(T, W, 16)
                cj = torch.empty((T, 7), dtype=torch.float64, device=self._device)
                cj[:] = self._dev(self.previous_sol[name] if current_joints is None else current_joints)
                cp = torch.empty((T, 16), dtype=torch.float64, device=self._device)
                cp[:] = self._dev(self.previous_pose[name] if current_pose is None else current_pose).reshape(-1, 16)
                states_on_device = hasattr(states, "is_cuda") and states.is_cuda
                if states_on_device:
                    st = states
                else:
                    if states is None:
                        states = np.zeros(T, dtype=_abi.TRAJ_STATE_DTYPE)
                        states["init"] = 1
                    st = torch.from_numpy(np.ascontiguousarray(states).view(np.uint8).reshape(T, -1)).to(self._device)
                if out is not None and was_cuda:
                    joints, reach, state = out[0], out[1].view(torch.uint8), out[2]
                else:
                    joints = torch.empty((T, W, 7), dtype=torch.float64, device=self._device)
                    reach = torch.empty((T, W), dtype=torch.uint8, device=self._device)
                    state = torch.empty((T, W), dtype=torch.uint8, device=self._device)
                if phased:
                    n_wp = T * W
                    ws = self._scratch(n_wp + (n_wp + 3) // 4, stream.value)
                    rc = solver._handle.lib.r2ik_ctl_continuous_phased_f64(
                        solver._handle.h, C.byref(par), _ptr(Md), C.c_int64(T), C.c_int32(W), _ptr(cj), _ptr(cp), _ptr(st),
                        _ptr(joints), _ptr(reach), _ptr(state), _ptr(ws), C.c_int32(int(_test_force_serial_mod)), stream)
                    _native.check(rc, "r2ik_ctl_continuous_phased_f64")
                else:
                    rc = solver._handle.lib.r2ik_ctl_continuous_f64(solver._handle.h, C.byref(par), _ptr(Md), C.c_int64(T),
                                                                    C.c_int32(W), _ptr(cj), _ptr(cp), _ptr(st), _ptr(joints),
                                                                    _ptr(reach), _ptr(state), stream)
                    _native.check(rc, "r2ik_ctl_continuous_f64")
                st_out = st if states_on_device else st.cpu().numpy().reshape(-1).view(_abi.TRAJ_STATE_DTYPE).copy()
                res = (joints, reach.view(torch.bool), state)
                res = res if was_cuda else tuple(x.cpu().numpy() for x in res)
                return (*res, st_out)
            raise ValueError(f"Unknown type {control_type}")

    COMPACT_MIN_POSES = 1 << 18      # measured crossover (scripts/experiments/exp_r2_k2.py): 65 536 poses 39 vs 47 us, 262 144 poses 84 vs 79 us, 1M poses 253 vs 203 us

    def _scratch(self, n: int, stream_key=0):
        """Device scratch of n doubles for the phased continuous / compacted discrete kernels, one buffer per CUDA stream (launches on one
        stream are ordered; two streams, or two threads on two streams, must not share it), grown on demand."""
        torch = self._torch
        cache = self.__dict__.setdefault("_scratch_bufs", {})
        buf = cache.get(stream_key)
        if buf is None or buf.numel() < n or buf.device != self._device:
            buf = cache[stream_key] = torch.empty(n, dtype=torch.float64, device=self._device)
        return buf

    def clear_caches(self) -> None:
        """Drop the cached scratch and host-pipeline device buffers."""
        self.__dict__.pop("_scratch_bufs", None)
        self.__dict__.pop("_pipe_cache", None)

    def _replica(self, device: int) -> "ControlIK":
        """This controller's solvers bound to another CUDA device of the process (same parameters, same controller
        dictionaries): the per-device worker of ``devices=[...]``."""
        device = int(device)
        reps = self.__dict__.setdefault("_replicas", {})
        if self._device is not None and device == self._device.index:
            return self
        if device not in reps:
            import copy

            r = copy.copy(self)
            r.symbolic_ik_solver = {arm: sv.replica(device) for arm, sv in self.symbolic_ik_solver.items()}
            r._device = self._torch.device("cuda", device)
            r.__dict__.pop("_scratch_bufs", None)
            r.__dict__.pop("_pipe_cache", None)
            r._scalar_bufs = {}
            reps[device] = r
        r = reps[device]
        r.nb_search_points = self.nb_search_points
        r.previous_sol, r.previous_pose, r.preferred_theta = self.previous_sol, self.previous_pose, self.preferred_theta
        return r

    def _batch_on_devices(self, name, M, control_type, devices, **kw):
        from .workspace import shard_range

        torch = self._torch
        if hasattr(M, "is_cuda") and M.is_cuda:
            raise ValueError("devices=[...] spreads a host batch; a CUDA tensor already lives on one device")
        Mh = M if hasattr(M, "is_cuda") else torch.from_numpy(np.ascontiguousarray(M, dtype=np.float64))
        Mh = Mh.to(torch.float64).contiguous()
        n = Mh.shape[0]
        if control_type == "discrete":
            out = self.alloc_host_outputs("discrete", n)
        elif control_type == "continuous":
            out = self.alloc_host_outputs("continuous", (n, Mh.shape[1]))
        else:
            raise ValueError(f"Unknown type {control_type}")
        devices = [int(d) for d in devices]
        per_traj = {}
        if control_type == "continuous":          # per-trajectory arguments follow their trajectories
            for key, single_ndim in (("current_joints", 1), ("current_pose", 2), ("states", 0)):
                v = kw.get(key)
                if v is not None and np.ndim(v) == single_ndim + 1 and len(v) == n and np.shape(v) != (4, 4):
                    per_traj[key] = v
        workers = []
        for r, d in enumerate(devices):
            lo, hi = shard_range(n, r, len(devices))
            if hi == lo:
                continue
            kws = dict(kw)
            for key, v in per_traj.items():
                kws[key] = v[lo:hi]
            sub = tuple(o[lo:hi] for o in out)
            rep = self._replica(d)
            rep.symbolic_inverse_kinematics_batch_host(name, Mh[lo:hi], control_type, out=sub, _wait=False, **kws)
            workers.append(rep)
        for rep in workers:
            rep._wait_pipelines()
        res = [o.numpy() for o in out]
        res[1] = res[1].astype(bool)
        if control_type == "continuous":
            res[3] = res[3].reshape(-1).view(_abi.TRAJ_STATE_DTYPE).copy()
        return tuple(res)

    def _wait_pipelines(self):
        for pipe in getattr(self, "_pipe_cache", {}).values():
            for s in pipe["streams"]:
                s.synchronize()
        for pipe in self.__dict__.pop("_native_pipes", []):
            pipe.wait()

    # ------------------------------------------------------------------ host-buffer pipelines
    def alloc_host_outputs(self, control_type: str, shape) -> tuple:
        """Pinned host output buffers for ``symbolic_inverse_kinematics_batch_host`` (reusable across calls).
        discrete: shape = N -> (joints (N,7), reachable (N,) u8, state (N,) u8, emergency (N,) u8);
        continuous: shape = (T, W) -> (joints (T,W,7), reachable (T,W) u8, state (T,W) u8, states (T,80) u8)."""
        torch = self._torch
        pin = lambda *sz, dt=torch.uint8: torch.empty(sz, dtype=dt).pin_memory()
        if control_type == "discrete":
            n = int(shape)
            return (pin(n, 7, dt=torch.float64), pin(n), pin(n), pin(n))
        if control_type == "continuous":
            T, W = shape
            return (pin(T, W, 7, dt=torch.float64), pin(T, W), pin(T, W), pin(T, _abi.TRAJ_STATE_DTYPE.itemsize))
        raise ValueError(f"Unknown type {control_type}")

    def symbolic_inverse_kinematics_batch_host(self, name: str, M_host, control_type: str = "discrete", out=None,
                                               chunk: int | None = None, n_streams: int = 3, current_joints=None,
                                               constrained_mode: str = "unconstrained", current_pose=None,
                                               d_theta_max: float = 0.01, preferred_theta: float = -4 * np.pi / 6,
                                               previous_joints=None, states=None, _wait: bool = True):
        """Host-to-host ``symbolic_inverse_kinematics_batch``: ``M_host`` is a CPU tensor (ideally pinned),
        (N,4,4)/(N,16) for discrete mode or (T,W,4,4)/(T,W,16) for continuous mode; the results land in
        ``out`` (pinned CPU tensors from ``alloc_host_outputs``).  The batch is cut into chunks -- ``chunk``
        poses in discrete mode, ``chunk`` waypoints of every trajectory in continuous mode -- that flow
        H2D -> kernel -> D2H on CUDA streams, so both PCIe directions overlap the kernels.  Synchronous on
        return."""
        torch = self._torch
        solver = self.symbolic_ik_solver[name]
        par = self._ctl_params(name, constrained_mode, preferred_theta, d_theta_max)
        lib, h = solver._handle.lib, solver._handle.h
        if not hasattr(M_host, "is_cuda"):
            M_host = torch.from_numpy(np.ascontiguousarray(M_host, dtype=np.float64))
        if M_host.is_cuda:
            raise ValueError("symbolic_inverse_kinematics_batch_host takes host matrices; use symbolic_inverse_kinematics_batch "
                             "for CUDA tensors")
        # the copies below address raw rows of the host buffers: dense float64 only (a float32 tensor or a strided view
        # such as big[:, :W] would be read with the wrong pitch)
        M_host = M_host.to(torch.float64).contiguous()
        dev = self._device
        f64, u8 = torch.float64, torch.uint8
        with torch.cuda.device(dev):
            cur_stream = torch.cuda.current_stream(dev)
            if control_type == "discrete":
                n = M_host.shape[0]
                P = M_host.reshape(n, 16)
                chunk = chunk or (1 << 16)
                if out is None:
                    out = self.alloc_host_outputs("discrete", n)
                for i, (cols, dtype) in enumerate(((7, f64), (1, u8), (1, u8), (1, u8))):
                    o = out[i]
                    if not hasattr(o, "is_cuda") or o.is_cuda or o.dtype != dtype or o.numel() != n * cols or not o.is_contiguous():
                        raise ValueError(f"out[{i}] must be a contiguous CPU tensor of {n} x {cols} {dtype} (see alloc_host_outputs)")
                prev = np.ascontiguousarray(self.previous_sol[name] if previous_joints is None else previous_joints, dtype=np.float64).reshape(7)
                cur = prev if current_joints is None else np.ascontiguousarray(current_joints, dtype=np.float64).reshape(7)
                pipe = solver._pipeline(chunk, n_streams)      # the native chunk loop of libr2ik.so (r2ik_pipeline_*)
                dp = C.POINTER(C.c_double)
                rc = lib.r2ik_pipeline_ctl_discrete_f64(pipe.p, C.byref(par), C.c_void_p(P.data_ptr()), C.c_int64(n),
                                                        prev.ctypes.data_as(dp), cur.ctypes.data_as(dp),
                                                        C.c_void_p(out[0].data_ptr()), C.c_void_p(out[1].data_ptr()),
                                                        C.c_void_p(out[2].data_ptr()), C.c_void_p(out[3].data_ptr()))
                _native.check_pipeline(rc, "r2ik_pipeline_ctl_discrete_f64")
                if _wait:
                    pipe.wait()
                else:
                    self.__dict__.setdefault("_native_pipes", []).append(pipe)
                return out
            elif control_type == "continuous":
                # A trajectory is a recursion over its waypoints, so K3's run time is set by W, not by T: the
                # pipeline therefore cuts the WAYPOINT axis.  Chunk c = waypoints [w0, w1) of every trajectory
                # (a strided block of the (T, W, 16) host array, moved by 2-D copies); the controller states
                # stay on the device between chunks (R2ikTrajState is the resume point).  Copies in, kernels
                # and copies out run on three streams chained by events.
                T, W = M_host.shape[0], M_host.shape[1]
                P = M_host.reshape(T, W, 16)
                wc = chunk or max(1, min(W, (1 << 18) // max(T, 1)))          # waypoints per chunk
                if out is None:
                    out = self.alloc_host_outputs("continuous", (T, W))
                want = (((T, W, 7), f64), ((T, W), u8), ((T, W), u8), ((T, _abi.TRAJ_STATE_DTYPE.itemsize), u8))
                for i, (shape, dtype) in enumerate(want):
                    o = out[i]
                    if (not hasattr(o, "is_cuda") or o.is_cuda or o.dtype != dtype or tuple(o.shape) != shape
                            or not o.is_contiguous()):
                        raise ValueError(f"out[{i}] must be a contiguous CPU tensor of shape {shape} and dtype {dtype} "
                                         "(see alloc_host_outputs)")
                cj = torch.empty((T, 7), dtype=f64, device=dev)
                cj[:] = self._dev(self.previous_sol[name] if current_joints is None else current_joints)
                cp = torch.empty((T, 16), dtype=f64, device=dev)
                cp[:] = self._dev(self.previous_pose[name] if current_pose is None else current_pose).reshape(-1, 16)
                if states is None:
                    states = np.zeros(T, dtype=_abi.TRAJ_STATE_DTYPE)
                    states["init"] = 1
                st = torch.from_numpy(np.ascontiguousarray(states).view(np.uint8).reshape(T, -1)).to(dev)
                n_slots = max(2, n_streams)
                pipe = self._pipeline(("continuous", T, wc, n_slots), lambda: dict(
                    M=torch.empty((T, wc, 16), dtype=f64, device=dev), joints=torch.empty((T, wc, 7), dtype=f64, device=dev),
                    reach=torch.empty((T, wc), dtype=u8, device=dev), state=torch.empty((T, wc), dtype=u8, device=dev),
                    ws=torch.empty(T * wc + (T * wc + 3) // 4, dtype=f64, device=dev)),
                    max(3, n_slots))
                s_in, s_k, s_out = pipe["streams"][:3]
                for s in (s_in, s_k, s_out):
                    s.wait_stream(cur_stream)
                ev = [dict(h2d=torch.cuda.Event(), k=None, d2h=None) for _ in range(n_slots)]

                def copy2d(dst_ptr, dpitch, src_ptr, spitch, width, stream):
                    rc = lib.r2ik_copy2d_async(C.c_void_p(dst_ptr), dpitch, C.c_void_p(src_ptr), spitch, width, T,
                                               C.c_void_p(stream.cuda_stream))
                    _native.check(rc, "r2ik_copy2d_async")

                for ci, w0 in enumerate(range(0, W, wc)):
                    w1 = min(W, w0 + wc)
                    m = w1 - w0
                    e, b = ev[ci % n_slots], pipe["bufs"][ci % n_slots]
                    if e["k"] is not None:
                        s_in.wait_event(e["k"])                   # the kernel that read this slot's poses is done
                    copy2d(b["M"].data_ptr(), m * 128, P.data_ptr() + w0 * 128, W * 128, m * 128, s_in)
                    e["h2d"].record(s_in)
                    s_k.wait_event(e["h2d"])
                    if e["d2h"] is not None:
                        s_k.wait_event(e["d2h"])                  # this slot's previous results have left
                    rc = lib.r2ik_ctl_continuous_phased_f64(h, C.byref(par), _ptr(b["M"]), C.c_int64(T), C.c_int32(m), _ptr(cj),
                                                           _ptr(cp), _ptr(st), _ptr(b["joints"]), _ptr(b["reach"]),
                                                           _ptr(b["state"]), _ptr(b["ws"]), C.c_int32(0),
                                                           C.c_void_p(s_k.cuda_stream))
                    _native.check(rc, "r2ik_ctl_continuous_phased_f64")
                    e["k"] = torch.cuda.Event()
                    e["k"].record(s_k)
                    s_out.wait_event(e["k"])
                    copy2d(out[0].data_ptr() + w0 * 56, W * 56, b["joints"].data_ptr(), m * 56, m * 56, s_out)
                    copy2d(out[1].data_ptr() + w0, W, b["reach"].data_ptr(), m, m, s_out)
                    copy2d(out[2].data_ptr() + w0, W, b["state"].data_ptr(), m, m, s_out)
                    e["d2h"] = torch.cuda.Event()
                    e["d2h"].record(s_out)
                s_out.wait_stream(s_k)
                with torch.cuda.stream(s_out):
                    out[3].copy_(st, non_blocking=True)
            else:
                raise ValueError(f"Unknown type {control_type}")
            if _wait:
                for s in pipe["streams"]:
                    s.synchronize()
        return out

    _PIPE_CACHE_MAX = 4   # distinct pipeline shapes kept per controller (device buffers)

    def _pipeline(self, key, make_bufs, n_streams: int):
        cache = getattr(self, "_pipe_cache", None)
        if cache is None:
            cache = self._pipe_cache = {}
        if key not in cache:
            torch = self._torch
            while len(cache) >= self._PIPE_CACHE_MAX:      # bounded: the oldest pipeline's buffers go back to the allocator
                cache.pop(next(iter(cache)))
            cache[key] = {"streams": [torch.cuda.Stream(device=self._device) for _ in range(n_streams)],
                          "bufs": [make_bufs() for _ in range(n_streams)]}
        return cache[key]

    # ------------------------------------------------------------------ scalar API (reference signature)
    def symbolic_inverse_kinematics(  # noqa: C901
        self,
        name: str,
        M: np.ndarray,
        control_type: str,
        current_joints: list = [],
        constrained_mode: str = "unconstrained",
        current_pose: np.ndarray = np.array([]),
        d_theta_max: float = 0.01,
        preferred_theta: float = -4 * np.pi / 6,
    ) -> Tuple[np.ndarray, bool, str]:
        if control_type == "unfreeze":
            self.emergency_stop = False
            self.emergency_state = ""
            self.init = True
            if self.logger is not None:
                self.logger.info(f"{name} Unfreeze", throttle_duration_sec=1.0)
            else:
                print(f"{name} Unfreeze")
        if self.emergency_stop:
            if self.logger is not None:
                self.logger.info(f"{name} Emergency state: {self.emergency_state}", throttle_duration_sec=1.0)
            else:
                print(f"{name} Emergency state: {self.emergency_state}")
            return self.previous_sol[name], False, self.emergency_state
        M = np.asarray(M, dtype=np.float64)
        if len(current_pose) == 0:
            current_pose = self.previous_pose[name]
        if current_joints == []:
            current_joints = self.previous_sol[name].tolist()

        if control_type == "continuous" or control_type == "unfreeze":
            ik_joints, is_reachable, state = self._continuous_one(name, M, current_joints, current_pose, constrained_mode,
                                                                  preferred_theta, d_theta_max)
        elif control_type == "discrete":
            ik_joints, is_reachable, state = self._discrete_one(name, M, current_joints, constrained_mode, preferred_theta)
        else:
            raise ValueError(f"Unknown type {control_type}")
        self.previous_pose[name] = M
        return ik_joints, is_reachable, state

    # One control tick = ONE kernel launch + one stream synchronisation: the inputs and the results of the N = 1 call live
    # in a page of mapped pinned host memory that the kernel reads and writes directly (no allocation, no cudaMemcpy).
    _SC_M, _SC_PREV, _SC_CUR, _SC_CP, _SC_ST, _SC_J, _SC_FLAGS = 0, 16, 23, 30, 46, 56, 63   # offsets in doubles

    def _scalar_page(self, name: str):
        b = self._scalar_bufs.get(name)
        if b is None:
            torch = self._torch
            page = torch.zeros(64, dtype=torch.float64).pin_memory()
            b = self._scalar_bufs[name] = dict(page=page, f=page.numpy(), u8=page.numpy().view(np.uint8), base=page.data_ptr())
        return b

    def _discrete_one(self, name, M, current_joints, constrained_mode, preferred_theta):
        torch = self._torch
        solver = self.symbolic_ik_solver[name]
        par = self._ctl_params(name, constrained_mode, preferred_theta, 0.01)
        b = self._scalar_page(name)
        f, u8, base = b["f"], b["u8"], b["base"]
        f[self._SC_M:self._SC_M + 16] = M.reshape(16)
        f[self._SC_PREV:self._SC_PREV + 7] = self.previous_sol[name]
        f[self._SC_CUR:self._SC_CUR + 7] = current_joints
        at = lambda off: C.c_void_p(base + 8 * off)   # noqa: E731
        fl = 8 * self._SC_FLAGS
        lib = solver._handle.lib
        stream = C.c_void_p(torch.cuda.current_stream(self._device).cuda_stream)
        rc = lib.r2ik_ctl_discrete_f64(solver._handle.h, C.byref(par), at(self._SC_M), C.c_int64(1), at(self._SC_PREV),
                                       at(self._SC_CUR), at(self._SC_J), C.c_void_p(base + fl), C.c_void_p(base + fl + 1),
                                       C.c_void_p(base + fl + 2), stream)
        _native.check(rc, "r2ik_ctl_discrete_f64")
        _native.check(lib.r2ik_stream_synchronize(stream), "r2ik_stream_synchronize")
        reach, code, bits = int(u8[fl]), int(u8[fl + 1]), int(u8[fl + 2])
        if code == STATE_INVALID_ROTATION:
            raise ValueError("Non-positive determinant (left-handed or null coordinate frame) in rotation matrix")
        if bits:
            self.emergency_state += emergency_text(bits)
            self.emergency_stop = True
        return f[self._SC_J:self._SC_J + 7].copy(), bool(reach), STATE_STRINGS[code]

    def _continuous_one(self, name, M, current_joints, current_pose, constrained_mode, preferred_theta, d_theta_max):
        torch = self._torch
        solver = self.symbolic_ik_solver[name]
        par = self._ctl_params(name, constrained_mode, preferred_theta, d_theta_max)
        t = time.time()
        timed_out = abs(t - self.last_call_t[name]) > self.call_timeout            # control_ik.py:296-304
        st = np.zeros(1, dtype=_abi.TRAJ_STATE_DTYPE)
        st["init"] = 1 if timed_out else int(self.init)
        st["previous_theta"] = self.previous_theta[name]
        if not timed_out and len(self.previous_sol[name]) != 0:
            st["has_previous_sol"] = 1
            st["previous_sol"][0] = self.previous_sol[name]
        b = self._scalar_page(name)
        f, u8, base = b["f"], b["u8"], b["base"]
        f[self._SC_M:self._SC_M + 16] = M.reshape(16)
        f[self._SC_CUR:self._SC_CUR + 7] = np.asarray(current_joints, dtype=np.float64)
        f[self._SC_CP:self._SC_CP + 16] = np.asarray(current_pose, dtype=np.float64).reshape(16)
        u8[8 * self._SC_ST:8 * self._SC_ST + 80] = st.view(np.uint8)
        at = lambda off: C.c_void_p(base + 8 * off)   # noqa: E731
        fl = 8 * self._SC_FLAGS
        lib = solver._handle.lib
        stream = C.c_void_p(torch.cuda.current_stream(self._device).cuda_stream)
        rc = lib.r2ik_ctl_continuous_f64(solver._handle.h, C.byref(par), at(self._SC_M), C.c_int64(1), C.c_int32(1),
                                         at(self._SC_CUR), at(self._SC_CP), at(self._SC_ST), at(self._SC_J),
                                         C.c_void_p(base + fl), C.c_void_p(base + fl + 1), stream)
        _native.check(rc, "r2ik_ctl_continuous_f64")
        _native.check(lib.r2ik_stream_synchronize(stream), "r2ik_stream_synchronize")
        reach, code = int(u8[fl]), int(u8[fl + 1])
        if code == STATE_INVALID_ROTATION:
            # scipy raises inside get_euler_from_homogeneous_matrix (control_ik.py:216), before the reference touches
            # any controller state: nothing of this call is kept
            raise ValueError("Non-positive determinant (left-handed or null coordinate frame) in rotation matrix")
        if timed_out:
            self.init = True
        self.last_call_t[name] = t
        st = u8[8 * self._SC_ST:8 * self._SC_ST + 80].copy().view(_abi.TRAJ_STATE_DTYPE)
        self.previous_theta[name] = float(st["previous_theta"][0])
        self.previous_sol[name] = np.array(st["previous_sol"][0])
        self.init = bool(st["init"][0])
        bits = int(st["emergency_bits"][0])
        if st["emergency_stop"][0]:
            self.emergency_stop = True
            self.emergency_state += emergency_text(bits)
            if bits & _abi.EMG_DISCONTINUITY:
                self.emergency_state += (f"\n EMERGENCY STOP: joints are not continuous \n previous_joints: "
                                         f"{self.previous_sol[name]} \n joints: (see device log)")
        state = self.emergency_state if code == STATE_EMERGENCY else STATE_STRINGS[code]
        return f[self._SC_J:self._SC_J + 7].copy(), bool(reach), state
