"""Argument checks of the controller's workspace map entry (r2ik_ctl_reach_map_u32) on libr2ik.so without a device:
every invalid argument is refused with an R2IK_ERR_* code and the entry's name in r2ik_last_error() before any CUDA
call (the handle is never dereferenced on these paths)."""
import ctypes as C

import numpy as np
import pytest

from reachy2_symbolic_ik_b200 import _abi

ERR_NULL, ERR_ARG = 1, 2


@pytest.fixture(scope="module")
def lib():
    from reachy2_symbolic_ik_b200 import _native, build

    build.build()
    return _native.load()


def test_argument_errors_do_not_need_a_device(lib):
    buf = (C.c_double * 64)()
    fake_handle = C.c_void_p(C.addressof(buf))
    ori, acc, rea = C.c_void_p(C.addressof(buf) + 8), C.c_void_p(C.addressof(buf) + 16), C.c_void_p(C.addressof(buf) + 24)
    origin = np.zeros(3); step = np.full(3, 0.01)
    dp, ip = C.POINTER(C.c_double), C.POINTER(C.c_int32)
    par = _abi.CtlParams()
    par.nb_search_points = 20
    i32 = C.c_int32

    def call(h=fake_handle, p=None, o=origin, s=step, d=(4, 4, 4), orientations=ori, b=0, e=8, a=acc, r=rea, K=20):
        par.nb_search_points = K
        dims = None if d is None else np.array(d, dtype=np.int32)
        return lib.r2ik_ctl_reach_map_u32(
            h, C.byref(par) if p is None else p, None if o is None else o.ctypes.data_as(dp),
            None if s is None else s.ctypes.data_as(dp), None if dims is None else dims.ctypes.data_as(ip), orientations,
            i32(b), i32(e), a, r, None)

    def refused(code, **kw):
        lib.r2ik_last_error.restype = C.c_char_p
        assert call(**kw) == code, kw
        assert b"r2ik_ctl_reach_map_u32" in lib.r2ik_last_error(), kw

    refused(ERR_NULL, h=None)
    refused(ERR_NULL, p=C.POINTER(_abi.CtlParams)())
    refused(ERR_NULL, o=None)
    refused(ERR_NULL, s=None)
    refused(ERR_NULL, d=None)
    refused(ERR_NULL, orientations=None)
    refused(ERR_NULL, a=None)
    refused(ERR_ARG, d=(0, 4, 4))
    refused(ERR_ARG, d=(4, -1, 4))
    refused(ERR_ARG, d=(4, 4, 0))
    refused(ERR_ARG, b=5, e=4)
    refused(ERR_ARG, b=-1, e=4)
    refused(ERR_ARG, K=1)
    refused(ERR_ARG, K=-5)
    refused(ERR_ARG, d=(1 << 30, 1 << 30, 1 << 30))     # more voxels than one launch covers
    refused(ERR_ARG, K=1, h=fake_handle, a=None)          # nb_search_points is checked with the handle, before the pointers


def test_discrete_workspace_bytes_beyond_2gb(lib):
    """The controller map's yardstick (the compacted discrete entry on every materialised pose of a 64^3 x 128 map, 33.5 M
    poses) needs more than 2 GB of workspace: the size query returns it as a 64-bit count."""
    n = 64 ** 3 * 128
    assert lib.r2ik_ctl_discrete_workspace_bytes(C.c_int64(n)) >= 80 * n > 2 ** 31
