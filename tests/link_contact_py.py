"""TEST-ONLY references for the link contact wrench (rkFDBatchGetLinkContactWrench): the oracle's per-link contact wrench
(tests/link_contact/ork_link_wrench.c, which compiles the unchanged oracle source into a library of its own, in a temporary
directory, and works on worlds made by the usual one), one oracle step from a loaded state, the readout compiled with g++ on
the host harness's states (tests/link_contact/hostsim_link_contact.cpp, likewise beside the unchanged harness), a numpy
restatement, and the worlds the tests run."""
import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

import rokifd_b200  # noqa: F401
from rokifd_b200 import chains as ch
from oracle.oracle import OracleWorld
from workloads import brick_wall_states, brick_wall_world, flat_states, flat_world, mm_states, mm_world

_HERE = os.path.dirname(os.path.abspath(__file__))
_vp, _dp, _ip = C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_int)
_LIB = None
_HLIB = None
_CSRC = os.path.join(os.path.dirname(_HERE), "roki-fd_b200", "csrc")

# relative tolerance of each world's solver, as the parity tests take it (tests/workloads.py::workload)
WORLDS = {"c3": 1e-9, "c4_penalty": 1e-9, "c4_volume": 1e-6, "c5_mlcp": 1e-9, "c5_vert": 1e-7, "box_stack": 1e-9,
          "box_stack_rigid_mlcp": 1e-9, "box_stack_rigid_vert": 1e-7, "arm_box_floor": 1e-9}
# share of environments that must match: the dense Vert path finds its multipliers by a Jacobi pseudo-inverse where the oracle
# refines zLESolveMP to rounding, so one step may split from the oracle's (the parity tests accept 75 % there); elsewhere all
SHARE = {"box_stack_rigid_vert": 0.75}


def assert_matches_oracle(got, ref, name):
    """the readout matches the oracle's link wrench within the world's tolerance in (a share SHARE of) the environments"""
    tol = WORLDS[name]
    assert np.isfinite(got).all(), name
    err = np.abs(got - ref).reshape(len(ref), -1).max(1) / (1.0 + np.abs(ref).reshape(len(ref), -1).max(1))
    assert (err <= tol).mean() >= SHARE.get(name, 1.0), "%s: %d / %d environments within %.1e (max %.3e)" % (
        name, (err <= tol).sum(), len(err), tol, err.max())


def world(name):
    """(world, sampler(B, seed) -> (q, qd, u))"""
    if name == "arm_box_floor":
        w, q0 = flat_world(name, soft=True)
        return w, lambda B, seed: flat_states(name, w, q0, B, seed=seed)
    if name == "brick_wall":
        w = brick_wall_world([200.0, 4.0, 10.0], [200.0, 0.3, 10.0])
        return w, lambda B, seed: brick_wall_states(w, B, seed)
    if name.startswith("box_stack"):
        kind = "box_stack_rigid" if "rigid" in name else "box_stack"
        w = mm_world(kind, solver="MLCP" if name.endswith("mlcp") else "Vert")
        return w, lambda B, seed: mm_states(kind, w, B, seed=seed)
    if name.startswith("c4"):
        w = ch.world_c4_volume() if name == "c4_volume" else ch.world_c4_penalty()
        return w, lambda B, seed: ch.sample_c4_standing(w, B, seed=seed)
    w = {"c3": lambda: ch.world_c3(base_z=0.3), "c5_mlcp": lambda: ch.world_c5(base_z=0.3, solver="MLCP"),
         "c5_vert": lambda: ch.world_c5(base_z=0.3, solver="Vert")}[name]()
    return w, lambda B, seed: ch.sample_state(w, B, seed=seed)


def oracle_lib():
    global _LIB
    if _LIB is None:
        tmp = tempfile.mkdtemp(prefix="rkfd_link_contact_")
        atexit.register(shutil.rmtree, tmp, True)
        so = os.path.join(tmp, "libork_link_wrench.so")
        subprocess.check_call(["/usr/bin/gcc", "-O3", "-march=x86-64-v3", "-fno-fast-math", "-fopenmp", "-fPIC", "-shared",
                               os.path.join(_HERE, "link_contact", "ork_link_wrench.c"), "-lm", "-o", so])
        L = C.CDLL(so)
        L.ork_env_new.restype = _vp
        L.ork_env_new.argtypes = [_vp]
        L.ork_env_free.argtypes = [_vp]
        L.ork_env_set_state.argtypes = [_vp, _dp, _dp]
        L.ork_env_set_motor_input.argtypes = [_vp, _dp]
        L.ork_env_set_contact.argtypes = [_vp, _ip, _ip, _dp]
        L.ork_env_set_pivot.argtypes = [_vp, _ip, _dp]
        L.ork_env_update.argtypes = [_vp]
        L.ork_env_get_link_wrench.argtypes = [_vp, _dp]
        L.ork_env_get_contact.argtypes = [_vp, _ip, _ip, _dp, _dp]
        _LIB = L
    return _LIB


def harness_lib():
    """the readout beside the host harness, built with the flags of libhostsim.so (tests/hostsim_py.py)"""
    global _HLIB
    if _HLIB is None:
        tmp = tempfile.mkdtemp(prefix="rkfd_link_contact_")
        atexit.register(shutil.rmtree, tmp, True)
        so = os.path.join(tmp, "libhostsim_link_contact.so")
        subprocess.check_call(["/usr/bin/g++", "-O2", "-mfma", "-ffp-contract=off", "-std=c++17", "-fPIC", "-shared", "-I" + _CSRC,
                               os.path.join(_HERE, "link_contact", "hostsim_link_contact.cpp"), os.path.join(_CSRC, "rkfd_model.cpp"),
                               "-o", so])
        L = C.CDLL(so)
        L.hostsim_link_contact.argtypes = [_vp, C.c_int] + [_vp] * 3 + [C.c_int] + [_vp] * 3 + [C.c_int]
        _HLIB = L
    return _HLIB


def harness_link_contact(hs, links=None):
    """the readout of rkFDBatchGetLinkContactWrench on the committed state and contact forces of a host harness `hs`
    (hostsim_py.HostSim): (B, n, 6) of `links` (None: all) - force, torque about the link origin, world axes"""
    q, _, _ = hs.get_state()
    pt, _ = hs.get_pivot()
    f = np.ascontiguousarray(hs.get_contact()[3])
    piv = (pt.astype(np.uint64) << np.arange(pt.shape[1], dtype=np.uint64)).sum(1).astype(np.uint32)
    q = np.ascontiguousarray(q)
    n = hs.nl if links is None else len(links)
    li = None if links is None else np.ascontiguousarray(links, np.int32)
    w = np.full((hs.B, n, 6), np.nan)
    err = C.create_string_buffer(256)
    if harness_lib().hostsim_link_contact(hs.h, hs.B, q.ctypes.data, piv.ctypes.data, f.ctypes.data, n,
                                          None if li is None else li.ctypes.data, w.ctypes.data, err, 256) != 0:
        raise RuntimeError(err.value.decode())
    return w


def _d(a):
    a = np.ascontiguousarray(a, dtype=np.float64)
    return a, a.ctypes.data_as(_dp)


def _i(a):
    a = np.ascontiguousarray(a, dtype=np.int32)
    return a, a.ctypes.data_as(_ip)


def oracle_step_wrench(w, q, qd, u, active, kinetic, ref, piv_type, piv_prev):
    """per environment: load (state, contact state, pivots, input) into an oracle environment, take ONE step, and return the
    contact wrench of every link from that step's committing evaluation, (B, nl, 6): force and torque about the link origin in
    world axes, and that evaluation's contact forces (B, nslot, 3).  ork_env_update steps from what was loaded (the t = 0
    committing evaluation of update_init is not run)"""
    L, ow = oracle_lib(), OracleWorld(w)
    B, nl, ns = q.shape[0], w.nl, max(ow.nslot, 1)
    out, cf = np.zeros((B, nl, 6)), np.zeros((B, ns, 3))
    for b in range(B):
        h = L.ork_env_new(ow.h)
        keep = [_d(q[b]), _d(qd[b]), _d(u[b]), _i(active[b]), _i(kinetic[b]), _d(ref[b]), _i(piv_type[b]), _d(piv_prev[b])]
        L.ork_env_set_state(h, keep[0][1], keep[1][1])
        L.ork_env_set_motor_input(h, keep[2][1])
        L.ork_env_set_contact(h, keep[3][1], keep[4][1], keep[5][1])
        L.ork_env_set_pivot(h, keep[6][1], keep[7][1])
        L.ork_env_update(h)
        r = np.zeros((nl, 6))
        L.ork_env_get_link_wrench(h, r.ctypes.data_as(_dp))
        out[b] = r
        a, t = np.zeros(ns, np.int32), np.zeros(ns, np.int32)
        L.ork_env_get_contact(h, a.ctypes.data_as(_ip), t.ctypes.data_as(_ip), np.zeros((ns, 3)).ctypes.data_as(_dp), cf[b].ctypes.data_as(_dp))
        L.ork_env_free(h)
    return out, cf


def assert_wrench_close(got, ref, tol, what):
    """|got - ref| <= tol (1 + max |ref|) per environment"""
    scale = 1.0 + np.abs(ref).reshape(len(ref), -1).max(1)
    err = np.abs(got - ref).reshape(len(ref), -1).max(1) / scale
    assert np.isfinite(got).all(), what
    assert err.max() <= tol, "%s: max scaled error %.3e (env %d) > %.1e" % (what, err.max(), int(err.argmax()), tol)


def restate(w, cf, frames):
    """numpy restatement of the readout for worlds whose boxes are all static floors (contact normal +z), from the contact forces
    cf (B, nslot, 3) and the link frames (B, nl, 12) of the same committed state: per (cell, box) pair, in the slot order of the
    model, +f at each vertex (an elastic force with f_z < 0 left out), or, for a Volume box pair, (force, torque about the
    centre, centre) in its first three slots.  (B, nl, 6): force, torque about the link origin, world axes"""
    boxes = [l.stuff for c in w.chains if c.is_static for l in c.links for _ in l.boxes]
    B = cf.shape[0]
    out = np.zeros((B, w.nl, 6))
    s = 0
    for i, l in enumerate(w.flat_links()):
        R, p = frames[:, i, :9].reshape(B, 3, 3), frames[:, i, 9:]
        for v in l.cells():
            v = np.asarray(v, float).reshape(-1, 3)
            for stuff in boxes:
                typ, n = w._ci_type(l.stuff, stuff), v.shape[0]
                f = cf[:, s:s + n]
                if w.solver == "Volume" and typ == "rigid":
                    if n == 8:
                        out[:, i, :3] += f[:, 0]
                        out[:, i, 3:] += f[:, 1] + np.cross(f[:, 2] - p, f[:, 0])
                else:
                    vw = p[:, None, :] + np.einsum("bij,kj->bki", R, v)
                    keep = (f[:, :, 2] >= 0)[:, :, None] if typ == "elastic" else np.ones_like(f[:, :, :1])
                    out[:, i, :3] += (f * keep).sum(1)
                    out[:, i, 3:] += (np.cross(vw - p[:, None, :], f) * keep).sum(1)
                s += n
    return out
