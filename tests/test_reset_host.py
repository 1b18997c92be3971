"""Environment reset (rkFDBatchResetEnvs / rkFDBatchResetEnvsDevice) without a device engine: both calls refuse with a
message that names rkFDUpdateInit, and the Python binding declares their signatures."""
import ctypes as C

import numpy as np

import rokifd_b200  # noqa: F401
from rokifd_b200 import capi
from rokifd_b200 import chains as ch


def test_reset_signatures_declared():
    L = capi.lib()
    assert L.rkFDBatchResetEnvs.restype is C.c_int and len(L.rkFDBatchResetEnvs.argtypes) == 6
    assert L.rkFDBatchResetEnvsDevice.restype is C.c_int and len(L.rkFDBatchResetEnvsDevice.argtypes) == 7
    assert L.rkFDBatchResetKernelCount.restype is C.c_longlong


def test_reset_needs_an_engine():
    fd, _ = capi.create_world(ch.world_c3(base_z=0.1), B=4)
    L = capi.lib()
    envs = np.array([0, 2], np.int32)
    q = np.zeros((2, fd.size))
    assert L.rkFDBatchResetEnvs(fd.h, 2, envs.ctypes.data, q.ctypes.data, None, None) != 0
    assert "rkFDUpdateInit" in fd.last_error()
    assert L.rkFDBatchResetEnvs(fd.h, 0, None, None, None, None) != 0
    assert "rkFDUpdateInit" in fd.last_error()
    assert L.rkFDBatchResetEnvsDevice(fd.h, 0, 2, envs.ctypes.data, q.ctypes.data, None, None) != 0
    assert "rkFDUpdateInit" in fd.last_error()
    assert fd.reset_kernel_count == 0
    fd.destroy()
