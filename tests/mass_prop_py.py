"""TEST-ONLY helpers for per-environment mass properties (rkFDBatchSetMassProp): the host harness of the kernel core with
StateDev::mp (tests/mass_prop/hostsim_mass_prop.cpp, compiled from the unchanged harness source into a library of its own, in a
temporary directory) and the reference for an environment: the unchanged oracle on a copy of the world whose declared links
carry that environment's mass, centre of mass and inertia."""
import atexit
import copy
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

from hostsim_py import HostSim
from oracle.oracle import OracleWorld

_HERE = os.path.dirname(os.path.abspath(__file__))
_CSRC = os.path.join(os.path.dirname(_HERE), "roki-fd_b200", "csrc")
_vp, _dp, _ip = C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_int)
_LIB = []


def hostsim_lib():
    if not _LIB:
        tmp = tempfile.mkdtemp(prefix="rkfd_mass_prop_")
        atexit.register(shutil.rmtree, tmp, True)
        so = os.path.join(tmp, "libhostsim_mass_prop.so")
        subprocess.check_call(["/usr/bin/g++", "-O2", "-mfma", "-ffp-contract=off", "-std=c++17", "-fPIC", "-shared", "-I" + _CSRC,
                               os.path.join(_HERE, "mass_prop", "hostsim_mass_prop.cpp"), os.path.join(_CSRC, "rkfd_model.cpp"), "-o", so])
        L = C.CDLL(so)
        L.hostsim_mp_declare.argtypes = [_vp, C.c_int, _ip]
        L.hostsim_mp_set.argtypes = [_vp, _dp]
        L.hostsim_mp_nmp.argtypes = [_vp]
        _LIB.append(L)
    return _LIB[0]


def row(mass, com, inertia):
    """(mass, com, Ic xx xy xz yy yz zz): the row of one link"""
    I = np.asarray(inertia, float)
    return np.array([mass, *np.asarray(com, float), I[0, 0], I[0, 1], I[0, 2], I[1, 1], I[1, 2], I[2, 2]])


def own_rows(w, links):
    """(n, 10): the model's own mass properties of `links`"""
    fl = w.flat_links()
    return np.array([row(fl[l].mass, fl[l].com, 0.5 * (np.asarray(fl[l].inertia) + np.asarray(fl[l].inertia).T)) for l in links])


def hostsim(world, B, links=None, spec=None, ext_links=None):
    """a HostSim of the kernel core; links: the links that take mass properties (set_mass_prop(hs, MP)), ext_links: the links that
    take an external wrench (ext_wrench_py.set_ext_wrench after this)"""
    hs = HostSim(world, B, spec=spec)
    if ext_links is not None:
        from ext_wrench_py import hostsim_lib as ext_lib
        li = np.ascontiguousarray(ext_links, np.int32).reshape(-1)
        if ext_lib().hostsim_ext_declare(hs.h, li.shape[0], li.ctypes.data_as(_ip)) != 0:
            raise RuntimeError("external wrench declaration refused")
    if links is not None:
        li = np.ascontiguousarray(links, np.int32).reshape(-1)
        if hostsim_lib().hostsim_mp_declare(hs.h, li.shape[0], li.ctypes.data_as(_ip)) != 0:
            raise RuntimeError("mass property declaration refused")
    return hs


def set_mass_prop(hs, MP):
    """MP (B, nmp, 10)"""
    L = hostsim_lib()
    MP = np.ascontiguousarray(MP, np.float64)
    assert MP.size == hs.B * 10 * L.hostsim_mp_nmp(hs.h)
    L.hostsim_mp_set(hs.h, MP.ctypes.data_as(_dp))


def world_with(w, links, rows):
    """a copy of world w whose links `links` (flat_links() indices) carry the mass properties rows[k]"""
    we = copy.deepcopy(w)
    objs = [l for c in we.moving_chains() for l in c.links]       # the links flat_links() copies, in its order
    for l, r in zip(links, rows):
        o = objs[l]
        o.mass, o.com = float(r[0]), np.array(r[1:4], float)
        o.inertia = np.array([[r[4], r[5], r[6]], [r[5], r[7], r[8]], [r[6], r[8], r[9]]], float)
    return we


def oracle_run_mp(w, q, qd, u, links, MP, nsteps, W=None, wlinks=None):
    """every environment e through the unchanged oracle on world_with(w, links, MP[e]): (q, q', q'') after rkFDUpdateInit and
    nsteps steps.  W (B, len(wlinks), 6): external wrenches on wlinks as well (ext_wrench_py.oracle_run)"""
    out = [np.zeros_like(q), np.zeros_like(q), np.zeros_like(q)]
    for e in range(q.shape[0]):
        we = world_with(w, links, MP[e])
        if W is None:
            r = OracleWorld(we).batch_run(q[e:e + 1], qd[e:e + 1], u[e:e + 1], nsteps=nsteps)
        else:
            from ext_wrench_py import oracle_run
            r = oracle_run(we, q[e:e + 1], qd[e:e + 1], u[e:e + 1], wlinks, W[e:e + 1], nsteps)
        for k in range(3):
            out[k][e] = r[k][0]
    return out


def randomise(w, links, B, seed, mass=0.5, com=0.02, scale=(0.5, 1.5)):
    """(B, n, 10): the model's own values with masses randomised by +-mass, centres of mass shifted by up to `com` and inertias
    scaled by a factor in `scale` (positive definite by construction)"""
    rng = np.random.default_rng(seed)
    base = own_rows(w, links)
    MP = np.repeat(base[None], B, axis=0)
    MP[:, :, 0] *= rng.uniform(1 - mass, 1 + mass, (B, len(links)))
    MP[:, :, 1:4] += rng.uniform(-com, com, (B, len(links), 3))
    MP[:, :, 4:] *= rng.uniform(*scale, (B, len(links), 1))
    return MP
