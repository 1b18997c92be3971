"""TEST-ONLY reference for external wrenches (rkFDBatchSetExtWrench): the oracle with a wrench per link
(tests/ext_wrench/ork_ext_wrench.c), which compiles the unchanged oracle source into a library of its own, in a temporary
directory, and works on worlds made by the usual one.  The host harness of the kernel core takes the wrenches itself
(hostsim_py.HostSim(..., ext_links=...))."""
import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

from oracle.oracle import OracleWorld

_HERE = os.path.dirname(os.path.abspath(__file__))
_vp, _dp, _ip = C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_int)
_LIBS = {}
NDOF = {"fixed": 0, "revolute": 1, "prismatic": 1, "spherical": 3, "float": 6, "cylindrical": 2, "hooke": 2, "breakablefloat": 6}


def _build(name, cmd):
    if name not in _LIBS:
        tmp = tempfile.mkdtemp(prefix="rkfd_ext_wrench_")
        atexit.register(shutil.rmtree, tmp, True)
        so = os.path.join(tmp, name)
        subprocess.check_call(cmd + ["-o", so])
        _LIBS[name] = C.CDLL(so)
    return _LIBS[name]


def oracle_lib():
    L = _build("libork_ext_wrench.so", ["/usr/bin/gcc", "-O3", "-march=x86-64-v3", "-fno-fast-math", "-fopenmp", "-fPIC", "-shared",
                                        os.path.join(_HERE, "ext_wrench", "ork_ext_wrench.c"), "-lm"])
    L.ork_env_new.restype = _vp
    L.ork_env_new.argtypes = [_vp]
    L.ork_env_free.argtypes = [_vp]
    L.ork_env_set_state.argtypes = [_vp, _dp, _dp]
    L.ork_env_set_motor_input.argtypes = [_vp, _dp]
    L.ork_env_get_state.argtypes = [_vp, _dp, _dp, _dp]
    L.ork_env_get_pivot.argtypes = [_vp, _ip, _dp]
    L.ork_env_get_broken.argtypes = [_vp, _ip]
    L.ork_ext_update_init.argtypes = [_vp, _dp]
    L.ork_ext_update.argtypes = [_vp, _dp]
    L.ork_ext_eval.argtypes = [_vp, _dp, C.c_int]
    return L


def _d(a):
    a = np.ascontiguousarray(a, dtype=np.float64)
    return a, a.ctypes.data_as(_dp)


class OracleEnvWrench:
    """one oracle environment of world `ow` (an OracleWorld) with the wrench table W[nl][6] (force at the centre of mass, torque
    about it, world axes; zero until set)"""

    def __init__(self, ow):
        self.ow, self.L = ow, oracle_lib()
        self.h = self.L.ork_env_new(ow.h)
        self.W = np.zeros((max(ow.nl, 1), 6))

    def __del__(self):
        if getattr(self, "h", None):
            self.L.ork_env_free(self.h)
            self.h = None

    def set_state(self, q, qd):
        self.L.ork_env_set_state(self.h, _d(q)[1], _d(qd)[1])

    def set_motor_input(self, u):
        self.L.ork_env_set_motor_input(self.h, _d(u)[1])

    def set_ext_wrench(self, link, w):
        self.W[link] = np.asarray(w, float).reshape(6)

    def _w(self):
        self._keep = np.ascontiguousarray(self.W)
        return self._keep.ctypes.data_as(_dp)

    def update_init(self):
        self.L.ork_ext_update_init(self.h, self._w())

    def update(self):
        self.L.ork_ext_update(self.h, self._w())

    def eval(self, ref=False):
        self.L.ork_ext_eval(self.h, self._w(), int(ref))
        return self.get_state()[2]

    def get_state(self):
        n = max(self.ow.nq, 1)
        q, qd, qdd = np.zeros(n), np.zeros(n), np.zeros(n)
        self.L.ork_env_get_state(self.h, q.ctypes.data_as(_dp), qd.ctypes.data_as(_dp), qdd.ctypes.data_as(_dp))
        return q[:self.ow.nq], qd[:self.ow.nq], qdd[:self.ow.nq]

    def pivot_bits(self, world):
        """the engine's pivot convention: the friction pivot types, and the first dof of a broken breakable-float joint set"""
        n = max(self.ow.nq, 1)
        t, p = np.zeros(n, np.int32), np.zeros(n)
        self.L.ork_env_get_pivot(self.h, t.ctypes.data_as(_ip), p.ctypes.data_as(_dp))
        brk = np.zeros(max(self.ow.nl, 1), np.int32)
        self.L.ork_env_get_broken(self.h, brk.ctypes.data_as(_ip))
        qofs = np.cumsum([0] + [NDOF[l.jtype] for l in world.flat_links()])[:-1]
        t = t[:self.ow.nq]
        t[qofs[brk[:self.ow.nl] != 0]] = 1
        return t


def oracle_run(w, q, qd, u, links, W, nsteps):
    """every environment through the oracle with its wrench W[e] on `links`: (q, q', q'', pivot bits) after rkFDUpdateInit and
    nsteps steps"""
    ow = OracleWorld(w)
    out = [np.zeros_like(q), np.zeros_like(q), np.zeros_like(q), np.zeros(q.shape, np.int32)]
    for e in range(q.shape[0]):
        env = OracleEnvWrench(ow)
        env.set_state(q[e], qd[e]); env.set_motor_input(u[e])
        for k, l in enumerate(links):
            env.set_ext_wrench(l, W[e, k])
        env.update_init()
        for _ in range(nsteps):
            env.update()
        out[0][e], out[1][e], out[2][e] = env.get_state()
        out[3][e] = env.pivot_bits(w)
    return out

