"""ctypes binding of ``lib/libr2ik.so`` (C ABI in ``include/r2ik.h``).

There is no CPU implementation behind these calls: a missing library or a machine without a
CUDA device raises immediately."""
from __future__ import annotations

import ctypes as C
import os

from . import _abi

_LIB_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "lib", "libr2ik.so")
_lib = None


def use_library(path: str) -> None:
    """Bind another build of the same C ABI (the tuning variants of scripts/build_variants.py) instead of the in-tree
    ``lib/libr2ik.so``.  An explicit call of the experiment scripts, before the first ``load()``; nothing in the
    package reads the environment for it."""
    global _LIB_PATH
    if _lib is not None:
        raise R2ikError("use_library() must be called before the library is loaded")
    _LIB_PATH = os.path.abspath(path)


EXPORTS = (
    "r2ik_abi_version", "r2ik_last_error", "r2ik_create", "r2ik_destroy", "r2ik_get_constants",
    "r2ik_interval_limit", "r2ik_symik_solve_f64", "r2ik_symik_solve_f32", "r2ik_symik_no_limits_f64", "r2ik_elbow_positions_f64",
    "r2ik_symik_sweep_f64", "r2ik_symik_scalar_f64", "r2ik_stream_synchronize", "r2ik_ctl_ctor_theta_f64",
    "r2ik_ctl_discrete_f64", "r2ik_ctl_discrete_scan_f64", "r2ik_ctl_discrete_compact_f64", "r2ik_ctl_discrete_workspace_bytes", "r2ik_ctl_continuous_f64", "r2ik_ctl_continuous_phased_f64", "r2ik_reach_map_u32", "r2ik_reach_map_f64_u32", "r2ik_reach_map_range_u16", "r2ik_fk_f64", "r2ik_copy2d_async",
    "r2ik_dfma_probe", "r2ik_ffma_probe",
    "r2ik_pipeline_create", "r2ik_pipeline_destroy", "r2ik_pipeline_wait", "r2ik_pipeline_last_error", "r2ik_pipeline_symik_f64",
    "r2ik_pipeline_symik_f32", "r2ik_pipeline_ctl_discrete_f64",
)


class R2ikError(RuntimeError):
    pass


def lib_path() -> str:
    return _LIB_PATH


def load() -> C.CDLL:
    """Load libr2ik.so (loading itself needs no device; every compute entry does)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(_LIB_PATH):
        raise R2ikError(
            f"{_LIB_PATH} is missing: build it with `python -m reachy2_symbolic_ik_b200.build` "
            "(nvcc, sm_100a).  This package has no CPU fallback.")
    L = C.CDLL(_LIB_PATH)
    vp, i32, i64 = C.c_void_p, C.c_int32, C.c_int64
    L.r2ik_abi_version.restype = C.c_int
    L.r2ik_last_error.restype = C.c_char_p
    L.r2ik_create.argtypes = [C.POINTER(_abi.ArmConfig), C.c_int, C.POINTER(vp)]
    L.r2ik_destroy.argtypes = [vp]
    L.r2ik_get_constants.argtypes = [vp, C.POINTER(_abi.ArmConstants)]
    L.r2ik_interval_limit.argtypes = [C.c_int, C.c_int, C.POINTER(C.c_double)]
    L.r2ik_symik_solve_f64.argtypes = [vp, C.c_int, vp, vp, vp, i64, vp, vp, vp, vp, vp, vp]
    L.r2ik_symik_solve_f32.argtypes = [vp, C.c_int, vp, vp, vp, i64, vp, vp, vp, vp, vp, vp, vp, vp]
    L.r2ik_symik_no_limits_f64.argtypes = [vp, C.c_int, vp, vp, vp, i32, i64, vp, vp, vp, vp]
    L.r2ik_elbow_positions_f64.argtypes = [vp, C.c_int, vp, vp, i32, i64, i32, vp, vp, vp]
    L.r2ik_symik_sweep_f64.argtypes = [vp, C.c_int, vp, i64, vp, i32, i32, i32, vp, vp, vp, vp, vp, vp, vp, vp]
    L.r2ik_symik_scalar_f64.argtypes = [vp, C.POINTER(_abi.ScalarQuery), vp, vp]
    L.r2ik_stream_synchronize.argtypes = [vp]
    L.r2ik_ctl_ctor_theta_f64.argtypes = [vp, C.c_double, C.POINTER(C.c_double), i32, C.POINTER(C.c_double), vp, vp]
    L.r2ik_ctl_discrete_f64.argtypes = [vp, C.POINTER(_abi.CtlParams), vp, i64, vp, vp, vp, vp, vp, vp, vp]
    L.r2ik_ctl_discrete_scan_f64.argtypes = [vp, C.POINTER(_abi.CtlParams), vp, i64, vp, vp, vp, vp, vp, vp, vp]
    L.r2ik_ctl_discrete_compact_f64.argtypes = [vp, C.POINTER(_abi.CtlParams), vp, i64, vp, vp, vp, vp, vp, vp, vp, i64, vp]
    L.r2ik_ctl_discrete_workspace_bytes.argtypes = [i64]
    L.r2ik_ctl_discrete_workspace_bytes.restype = i64
    L.r2ik_ctl_continuous_f64.argtypes = [vp, C.POINTER(_abi.CtlParams), vp, i64, i32, vp, vp, vp, vp, vp, vp, vp]
    L.r2ik_ctl_continuous_phased_f64.argtypes = [vp, C.POINTER(_abi.CtlParams), vp, i64, i32, vp, vp, vp, vp, vp, vp, vp, i32, vp]
    L.r2ik_reach_map_u32.argtypes = [vp, C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(i32), vp, i32, i32, vp, vp]
    L.r2ik_reach_map_f64_u32.argtypes = [vp, C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(i32), vp, i32, i32, vp, vp]
    L.r2ik_reach_map_range_u16.argtypes = [vp, C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(i32), vp, i32, i32, i64, i64, i32, i32, vp, vp]
    L.r2ik_fk_f64.argtypes = [C.POINTER(_abi.FkChain), C.c_int, vp, i64, vp, vp]
    L.r2ik_copy2d_async.argtypes = [vp, C.c_size_t, vp, C.c_size_t, C.c_size_t, C.c_size_t, vp]
    L.r2ik_dfma_probe.argtypes = [C.c_int, i32, C.POINTER(C.c_double), C.POINTER(C.c_double), vp]
    L.r2ik_ffma_probe.argtypes = [C.c_int, i32, C.POINTER(C.c_double), C.POINTER(C.c_double), vp]
    L.r2ik_pipeline_create.argtypes = [vp, C.c_int, i64, i32, C.POINTER(vp)]
    L.r2ik_pipeline_destroy.argtypes = [vp]
    L.r2ik_pipeline_wait.argtypes = [vp]
    L.r2ik_pipeline_last_error.restype = C.c_char_p
    L.r2ik_pipeline_symik_f64.argtypes = [vp, C.c_int, vp, i64, vp, vp, vp, vp, vp]
    L.r2ik_pipeline_symik_f32.argtypes = [vp, C.c_int, vp, i64, vp, vp, vp, vp, vp]
    L.r2ik_pipeline_ctl_discrete_f64.argtypes = [vp, C.POINTER(_abi.CtlParams), vp, i64, C.POINTER(C.c_double),
                                                 C.POINTER(C.c_double), vp, vp, vp, vp]
    for name in EXPORTS:
        fn = getattr(L, name)  # AttributeError here = the library does not export what r2ik.h declares
        if name not in ("r2ik_abi_version", "r2ik_last_error", "r2ik_pipeline_last_error"):
            fn.restype = C.c_int
    if L.r2ik_abi_version() != _abi.ABI_VERSION:
        raise R2ikError(f"libr2ik.so ABI {L.r2ik_abi_version()} != expected {_abi.ABI_VERSION}; rebuild")
    _lib = L
    return L


def check(rc: int, what: str) -> None:
    if rc != 0:
        msg = load().r2ik_last_error().decode(errors="replace")
        kind = "argument error" if rc > 0 else "CUDA error"
        raise R2ikError(f"{what}: {kind} {rc}: {msg}")


def check_pipeline(rc: int, what: str) -> None:
    if rc != 0:
        msg = load().r2ik_pipeline_last_error().decode(errors="replace")
        kind = "argument error" if rc > 0 else "CUDA error"
        raise R2ikError(f"{what}: {kind} {rc}: {msg}")


class Pipeline:
    """Owns one r2ik_pipeline (device staging buffers + three streams + events) of a handle."""

    def __init__(self, handle: "Handle", chunk: int, n_slots: int):
        self.lib = handle.lib
        self.handle = handle          # keeps the r2ik_handle alive
        self._p = C.c_void_p()
        check_pipeline(self.lib.r2ik_pipeline_create(handle.h, handle.device, C.c_int64(int(chunk)), C.c_int32(int(n_slots)),
                                                     C.byref(self._p)), "r2ik_pipeline_create")

    @property
    def p(self):
        return self._p

    def wait(self) -> None:
        check_pipeline(self.lib.r2ik_pipeline_wait(self._p), "r2ik_pipeline_wait")

    def __del__(self):
        try:
            if getattr(self, "_p", None) and self._p.value:
                self.lib.r2ik_pipeline_destroy(self._p)
                self._p = C.c_void_p()
        except Exception:
            pass


def require_cuda():
    """torch is the device-memory / stream plumbing; the compute is libr2ik.so."""
    import torch

    if not torch.cuda.is_available():
        raise R2ikError("no CUDA device: reachy2_symbolic_ik_b200 runs on the GPU only (no CPU fallback)")
    return torch


class Handle:
    """Owns one r2ik_handle (per-arm constants bound to one CUDA device)."""

    def __init__(self, cfg: _abi.ArmConfig, device: int | None = None):
        torch = require_cuda()
        self.lib = load()
        self.device = torch.cuda.current_device() if device is None else int(device)
        self.cfg = cfg
        self._h = C.c_void_p()
        check(self.lib.r2ik_create(C.byref(cfg), self.device, C.byref(self._h)), "r2ik_create")
        self.constants = _abi.ArmConstants()
        check(self.lib.r2ik_get_constants(self._h, C.byref(self.constants)), "r2ik_get_constants")

    @property
    def h(self):
        return self._h

    def __del__(self):
        try:
            if getattr(self, "_h", None) and self._h.value:
                self.lib.r2ik_destroy(self._h)
                self._h = C.c_void_p()
        except Exception:
            pass


def interval_limit(side: int, low_elbow: bool):
    out = (C.c_double * 2)()
    check(load().r2ik_interval_limit(int(side), int(bool(low_elbow)), out), "r2ik_interval_limit")
    return [out[0], out[1]]
