"""ctypes wrapper of the TEST-ONLY host harness of the kernel core and the link kinematics walk (tests/hostsim/hostsim.cpp)."""
import ctypes as C
import os
import subprocess

import numpy as np

from oracle.oracle import pack_links, CONTACT, SOLVER

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "hostsim")
_CSRC = os.path.join(os.path.dirname(_HERE), "roki-fd_b200", "csrc")
_dp = C.POINTER(C.c_double)
_ip = C.POINTER(C.c_int)
_LIB = None


def lib():
    global _LIB
    if _LIB is None:
        so = os.path.join(_SRC, "libhostsim.so")
        deps = [os.path.join(_SRC, "hostsim.cpp")] + [os.path.join(_CSRC, f) for f in
                                                     ("rkfd_core.cuh", "rkfd_volume.cuh", "rkfd_kin.cuh", "rkfd_math.cuh", "rkfd_types.h",
                                                      "rkfd_model.cpp", "rkfd_model.h")]
        if not os.path.exists(so) or any(os.path.getmtime(d) > os.path.getmtime(so) for d in deps):
            subprocess.check_call(["/usr/bin/g++", "-O2", "-mfma", "-ffp-contract=off", "-std=c++17", "-fPIC", "-shared", "-I" + _CSRC,
                                   os.path.join(_SRC, "hostsim.cpp"), os.path.join(_CSRC, "rkfd_model.cpp"), "-o", so])
        L = C.CDLL(so)
        L.hostsim_new.restype = C.c_void_p
        L.hostsim_new.argtypes = [C.c_int, _ip, _ip, _dp]
        L.hostsim_add_cell.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, _dp]
        L.hostsim_add_box.argtypes = [C.c_void_p, C.c_int, C.c_int, _dp, C.c_double, C.c_double, C.c_double]
        L.hostsim_add_contact_info.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int] + [C.c_double] * 6
        L.hostsim_set_prp.argtypes = [C.c_void_p, C.c_double, C.c_int, C.c_double, C.c_int, C.c_int]
        L.hostsim_declare.argtypes = [C.c_void_p, C.c_int, C.c_int, _ip]
        L.hostsim_finalize.argtypes = [C.c_void_p, C.c_int]
        L.hostsim_error.restype = C.c_char_p
        L.hostsim_error.argtypes = [C.c_void_p]
        L.hostsim_use_spec.argtypes = [C.c_void_p, C.c_int]
        L.hostsim_spec_match.argtypes = [C.c_void_p, C.c_int]
        L.hostsim_spec_mask.restype = C.c_uint
        L.hostsim_spec_mask.argtypes = [C.c_void_p]
        for f in ("hostsim_nq", "hostsim_nl", "hostsim_nslot", "hostsim_nscratch", "hostsim_ext_nfext", "hostsim_mp_nmp", "hostsim_free"):
            getattr(L, f).argtypes = [C.c_void_p]
        L.hostsim_set_state.argtypes = [C.c_void_p, _dp, _dp, _dp]
        L.hostsim_ext_set.argtypes = [C.c_void_p, _dp]
        L.hostsim_mp_set.argtypes = [C.c_void_p, _dp]
        L.hostsim_link_frames.argtypes = [C.c_void_p, C.c_int] + [C.c_void_p] * 3 + [C.c_int] + [C.c_void_p] * 3
        L.hostsim_get_state.argtypes = [C.c_void_p, _dp, _dp, _dp]
        L.hostsim_get_contact.argtypes = [C.c_void_p, _ip, _ip, _dp, _dp]
        L.hostsim_get_pivot.argtypes = [C.c_void_p, _ip, _dp]
        L.hostsim_get_status.argtypes = [C.c_void_p, _ip]
        L.hostsim_run.argtypes = [C.c_void_p, C.c_int, C.c_int]
        _LIB = L
    return _LIB


def _d(a):
    a = np.ascontiguousarray(a, dtype=np.float64)
    return a, a.ctypes.data_as(_dp)


class HostSim:
    """B environments of `world` on the kernel core.  ext_links / mp_links: the links that take an external wrench
    (set_ext_wrench, zero until set) / per-environment mass properties (set_mass_prop, the model's own values until set)"""

    def __init__(self, world, B, spec=None, ext_links=None, mp_links=None):
        L = lib()
        links, nls = [], []
        for ch in world.chains:          # all chains (static ones included), chain-local parents
            nls.append(len(ch.links))
            links += ch.links
        li, ld = pack_links(world, links)
        nls = np.asarray(nls, np.int32)
        self.h = L.hostsim_new(len(nls), nls.ctypes.data_as(_ip), li.ctypes.data_as(_ip), ld.ctypes.data_as(_dp))
        for c, chn in enumerate(world.chains):
            for k, l in enumerate(chn.links):
                for v in (l.cells() if not chn.is_static else l.shapes):
                    v, pv = _d(v)
                    L.hostsim_add_cell(self.h, c, k, v.shape[0], pv)
                for (ctr, d, w, ht) in l.boxes:
                    _, pc = _d(ctr)
                    L.hostsim_add_box(self.h, c, k, pc, d, w, ht)
                for cell, (vel, axis) in l.slides.items():
                    L.hostsim_set_slide.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_double, _dp]
                    L.hostsim_set_slide(self.h, c, k, cell, float(vel), _d(np.asarray(axis, float))[1])
        L.hostsim_unreg_self_collision.argtypes = [C.c_void_p, C.c_int]
        for c, chn in enumerate(world.chains):
            if not chn.self_collide:
                L.hostsim_unreg_self_collision(self.h, c)
        for ci in world.contact_info:
            L.hostsim_add_contact_info(self.h, world.stuff_id(ci.stuff_a), world.stuff_id(ci.stuff_b),
                                       CONTACT[ci.type], ci.K, ci.L, ci.E, ci.V, ci.SF, ci.KF)
        L.hostsim_set_prp(self.h, world.dt, world.pyramid, world.friction_weight, world.max_iter, SOLVER[world.solver])
        L.hostsim_set_integrator.argtypes = [C.c_void_p, C.c_int]
        L.hostsim_set_integrator(self.h, {"RKG": 0, "RK4": 1, "Euler": 2, "Heun": 3}[getattr(world, "integrator", "RKG")])
        for kind, links in ((0, ext_links), (1, mp_links)):
            if links is not None:
                li = np.ascontiguousarray(links, np.int32).reshape(-1)
                L.hostsim_declare(self.h, kind, li.shape[0], li.ctypes.data_as(_ip))
        if L.hostsim_finalize(self.h, B) != 0:       # also refuses a declared link list
            raise RuntimeError(L.hostsim_error(self.h).decode())
        self.B, self.nq, self.nl, self.nslot = B, L.hostsim_nq(self.h), L.hostsim_nl(self.h), L.hostsim_nslot(self.h)
        self.nscratch = L.hostsim_nscratch(self.h)
        # model specialisations the kernel could pick (0: generic): scratch in shared memory / in tensor memory
        self.spec, self.spec_tm, self.spec_rolled = (L.hostsim_spec_match(self.h, k) for k in (0, 1, 2))
        self.spec_mask = L.hostsim_spec_mask(self.h)    # bit id: every specialisation the model is eligible for
        if spec:      # "smem" | "tmem" | "rolled" | "generic_tm", or a specialisation id: run that specialisation's code path
            sid = spec if isinstance(spec, int) else {"smem": self.spec, "tmem": self.spec_tm, "rolled": self.spec_rolled, "generic_tm": 11}[spec]
            assert sid > 0, "model matches no compiled specialisation"
            used = L.hostsim_use_spec(self.h, sid)
            assert used == sid, "model does not match specialisation %d" % sid

    def __del__(self):
        if getattr(self, "h", None):
            lib().hostsim_free(self.h)
            self.h = None

    def set_state(self, q, qd, u=None):
        _, pq = _d(q)
        _, pqd = _d(qd)
        pu = None
        if u is not None:
            _, pu = _d(u)
        lib().hostsim_set_state(self.h, pq, pqd, pu)

    def set_ext_wrench(self, W):
        """W (B, nfext, 6): force at the centre of mass, torque about it, world axes"""
        W, pw = _d(W)
        assert W.size == self.B * 6 * lib().hostsim_ext_nfext(self.h)
        lib().hostsim_ext_set(self.h, pw)

    def set_mass_prop(self, MP):
        """MP (B, nmp, 10)"""
        MP, pm = _d(MP)
        assert MP.size == self.B * 10 * lib().hostsim_mp_nmp(self.h)
        lib().hostsim_mp_set(self.h, pm)

    def link_frames(self, q, qd, piv_type=None, links=None, frames=True, vel=True):
        """the kinematics walk of rkFDBatchGetLinkFrames: frames (B, n, 12) and velocities (B, n, 6) of `links` (None: all) at
        env-major states of any B; piv_type: per-dof pivot bits (B, nq)"""
        q, qd = np.ascontiguousarray(q, np.float64), np.ascontiguousarray(qd, np.float64)
        B = q.shape[0]
        pv = None
        if piv_type is not None:
            pv = (piv_type.astype(np.uint64) << np.arange(piv_type.shape[1], dtype=np.uint64)).sum(1).astype(np.uint32)
        n = self.nl if links is None else len(links)
        li = None if links is None else np.ascontiguousarray(links, np.int32)
        fr = np.full((B, n, 12), np.nan) if frames else None
        v = np.full((B, n, 6), np.nan) if vel else None
        addr = lambda a: None if a is None else a.ctypes.data
        if lib().hostsim_link_frames(self.h, B, q.ctypes.data, qd.ctypes.data, addr(pv), n, addr(li), addr(fr), addr(v)) != 0:
            raise RuntimeError(lib().hostsim_error(self.h).decode())
        return fr, v

    def get_state(self):
        n = max(self.nq, 1)
        q, qd, qdd = (np.zeros((self.B, n)) for _ in range(3))
        lib().hostsim_get_state(self.h, q.ctypes.data_as(_dp), qd.ctypes.data_as(_dp), qdd.ctypes.data_as(_dp))
        return q, qd, qdd

    def get_contact(self):
        n = max(self.nslot, 1)
        a, t = np.zeros((self.B, n), np.int32), np.zeros((self.B, n), np.int32)
        r, f = np.zeros((self.B, n, 3)), np.zeros((self.B, n, 3))
        lib().hostsim_get_contact(self.h, a.ctypes.data_as(_ip), t.ctypes.data_as(_ip), r.ctypes.data_as(_dp), f.ctypes.data_as(_dp))
        return a, t, r, f

    def get_status(self):
        st = np.zeros(self.B, np.int32)
        lib().hostsim_get_status(self.h, st.ctypes.data_as(_ip))
        return st

    def get_pivot(self):
        n = max(self.nq, 1)
        t, p = np.zeros((self.B, n), np.int32), np.zeros((self.B, n))
        lib().hostsim_get_pivot(self.h, t.ctypes.data_as(_ip), p.ctypes.data_as(_dp))
        return t, p

    def eval(self, ref=False):
        lib().hostsim_run(self.h, 2 if ref else 1, 0)

    def step(self, n=1):
        lib().hostsim_run(self.h, 0, n)
