"""Link kinematics (rkFDBatchGetLinkFrames / rkFDBatchGetLinkFramesDevice) without a device: the C-ABI declarations, the calls
refused without rkFDUpdateInit, and the arithmetic of the kinematics walk (roki-fd_b200/csrc/rkfd_kin.cuh, compiled into the
host harness tests/hostsim/kin_harness.cpp) against the oracle's link frames and velocities."""
import atexit
import copy
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np
import pytest

import rokifd_b200  # noqa: F401
from rokifd_b200 import capi
from rokifd_b200 import chains as ch
from hostsim_py import HostSim
from oracle.oracle import OracleWorld, pack_links

NDOF = {"fixed": 0, "revolute": 1, "prismatic": 1, "cylindrical": 2, "hooke": 2, "spherical": 3, "float": 6, "breakablefloat": 6}
ALL_JOINTS = ("revolute", "prismatic", "spherical", "float", "cylindrical", "hooke", "breakablefloat")


# ---- reference: the oracle's frames at a state ----------------------------------------------------------------------------
def as_broken(world, broken):
    """a copy of `world` in which the breakable-float joints of the flat link indices `broken` are float joints - what a
    broken joint is - so that the oracle holds them broken"""
    w = copy.deepcopy(world)
    k = 0
    for chn in w.moving_chains():
        for l in chn.links:
            if k in broken:
                assert l.jtype == "breakablefloat"
                l.jtype = "float"
            k += 1
    return w


def broken_links(world, piv_type):
    """per environment: the flat link indices whose breakable-float joint is broken (pivot bit of the joint's first dof)"""
    out, o = [[] for _ in range(piv_type.shape[0])], 0
    for k, l in enumerate(world.flat_links()):
        if l.jtype == "breakablefloat":
            for e in np.nonzero(piv_type[:, o])[0]:
                out[e].append(k)
        o += NDOF[l.jtype]
    return [tuple(b) for b in out]


def oracle_frames(world, q, qd, broken=None):
    """frames (B, nl, 12) and world-axis velocities (B, nl, 6) of the oracle at states (q, qd)"""
    B, nl = q.shape[0], world.nl
    fr, vel, worlds = np.zeros((B, nl, 12)), np.zeros((B, nl, 6)), {}
    for e in range(B):
        key = broken[e] if broken is not None else ()
        if key not in worlds:
            worlds[key] = OracleWorld(as_broken(world, key))
        env = worlds[key].env()
        env.set_state(q[e], qd[e])
        env.eval(False)
        R, p = env.link_frames()
        v = env.link_vel()                          # link axes
        fr[e, :, :9], fr[e, :, 9:] = R.reshape(nl, 9), p
        vel[e, :, :3] = np.einsum("kij,kj->ki", R, v[:, :3])
        vel[e, :, 3:] = np.einsum("kij,kj->ki", R, v[:, 3:])
    return fr, vel


def assert_frames_close(fr, vel, ofr, ovel, what):
    """R within 1e-12, p within 1e-12 (1 + |p|), velocities within 1e-11 (1 + |v|)"""
    dR = np.abs(fr[..., :9] - ofr[..., :9]).max()
    assert dR <= 1e-12, "%s: R differs by %.3g" % (what, dR)
    dp = (np.abs(fr[..., 9:] - ofr[..., 9:]) / (1 + np.abs(ofr[..., 9:]))).max()
    assert dp <= 1e-12, "%s: p differs by %.3g" % (what, dp)
    if vel is not None:
        dv = (np.abs(vel - ovel) / (1 + np.abs(ovel))).max()
        assert dv <= 1e-11, "%s: velocity differs by %.3g" % (what, dv)


# ---- the host harness of the kinematics walk (tests/hostsim/kin_harness.cpp) ----------------------------------------------
_HERE = os.path.dirname(os.path.abspath(__file__))
_CSRC = os.path.join(os.path.dirname(_HERE), "roki-fd_b200", "csrc")
_KLIB = None


def klib():
    """the harness, compiled with g++ into a temporary directory once per session"""
    global _KLIB
    if _KLIB is None:
        tmp = tempfile.mkdtemp(prefix="rkfd_kin_")
        atexit.register(shutil.rmtree, tmp, True)
        so = os.path.join(tmp, "libkin_harness.so")
        subprocess.check_call(["/usr/bin/g++", "-O2", "-mfma", "-ffp-contract=off", "-std=c++17", "-fPIC", "-shared", "-I" + _CSRC,
                               os.path.join(_HERE, "hostsim", "kin_harness.cpp"), os.path.join(_CSRC, "rkfd_model.cpp"), "-o", so])
        L = C.CDLL(so)
        L.kin_new.restype = C.c_void_p
        L.kin_new.argtypes = [C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
        L.kin_error.restype = C.c_char_p
        L.kin_error.argtypes = [C.c_void_p]
        for f in ("kin_nl", "kin_nq", "kin_free"):
            getattr(L, f).argtypes = [C.c_void_p]
        L.kin_frames.argtypes = [C.c_void_p, C.c_int] + [C.c_void_p] * 3 + [C.c_int] + [C.c_void_p] * 3
        _KLIB = L
    return _KLIB


class KinHarness:
    """the kinematics walk of rkFDBatchGetLinkFrames on the CPU, for the links of `world`"""

    def __init__(self, world):
        L = klib()
        links, nls = [], []
        for chn in world.chains:         # all chains (static ones give no links), chain-local parents
            nls.append(len(chn.links))
            links += chn.links
        li, ld = pack_links(world, links)
        li, ld, nls = np.ascontiguousarray(li), np.ascontiguousarray(ld), np.asarray(nls, np.int32)
        self.h = L.kin_new(len(nls), nls.ctypes.data, li.ctypes.data, ld.ctypes.data)
        self.nl, self.nq = L.kin_nl(self.h), L.kin_nq(self.h)
        if self.nl < 0:
            raise RuntimeError(L.kin_error(self.h).decode())
        assert (self.nl, self.nq) == (world.nl, world.nq)

    def __del__(self):
        if getattr(self, "h", None):
            klib().kin_free(self.h)
            self.h = None

    def frames(self, q, qd, piv_type=None, links=None, frames=True, vel=True):
        """frames (B, n, 12) and velocities (B, n, 6) at env-major states; piv_type: per-dof pivot bits (B, nq)"""
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
        if klib().kin_frames(self.h, B, q.ctypes.data, qd.ctypes.data, addr(pv), n, addr(li), addr(fr), addr(v)) != 0:
            raise RuntimeError(klib().kin_error(self.h).decode())
        return fr, v


def structured(rng, chain):
    """quarter-turn and identity org rotations (the structured transforms of the revolute joint) and org positions on the
    parent's z axis on some links"""
    for l in chain.links[1:]:
        r = rng.integers(5)
        if r == 0:
            l.org_R = np.eye(3)
        elif r == 1:
            l.org_R = ch.rot_x(np.pi / 2)
        elif r == 2:
            l.org_R = ch.rot_x(-np.pi / 2)
        if rng.integers(3) == 0:
            l.org_p = np.array([0.0, 0.0, rng.uniform(-0.3, 0.3)])
    return chain


def random_world(seed):
    """three chains (a floating-root tree, a fixed-root tree, a breakable-float root with a revolute arm), within the 32 dofs
    of the pivot word"""
    rng = np.random.default_rng(seed)
    while True:
        chains = [structured(rng, ch.random_chain(rng, n_links=6, jtypes=ALL_JOINTS, root="float", branching=True, name="a")),
                  structured(rng, ch.random_chain(rng, n_links=6, jtypes=ALL_JOINTS, root="fixed", branching=True, name="b")),
                  structured(rng, ch.random_chain(rng, n_links=3, jtypes=("revolute",), root="breakablefloat", name="c"))]
        w = ch.World(chains=chains)
        jts = {l.jtype for l in w.flat_links()}
        if w.nq <= 32 and len(jts) >= 5:
            return w


def random_states(w, B, seed):
    rng = np.random.default_rng(seed)
    q = rng.uniform(-1.5, 1.5, (B, w.nq))
    qd = rng.uniform(-1.0, 1.0, (B, w.nq))
    piv = np.zeros((B, w.nq), np.int32)
    o = 0
    for l in w.flat_links():
        if l.jtype == "breakablefloat":
            piv[:, o] = rng.integers(0, 2, B)
        o += NDOF[l.jtype]
    return q, qd, piv


# ---- tests ----------------------------------------------------------------------------------------------------------------
def test_link_frame_signatures_declared():
    L = capi.lib()
    assert L.rkFDBatchGetLinkFrames.restype is C.c_int and len(L.rkFDBatchGetLinkFrames.argtypes) == 5
    assert L.rkFDBatchGetLinkFramesDevice.restype is C.c_int and len(L.rkFDBatchGetLinkFramesDevice.argtypes) == 6
    assert L.rkFDBatchLinkFrameKernelCount.restype is C.c_longlong and len(L.rkFDBatchLinkFrameKernelCount.argtypes) == 1


def test_link_frames_need_an_engine():
    fd, _ = capi.create_world(ch.world_c3(base_z=0.1), B=4)
    L = capi.lib()
    links = np.array([0, 7], np.int32)
    fr, v = np.zeros((4, 2, 12)), np.zeros((4, 2, 6))
    assert L.rkFDBatchGetLinkFrames(fd.h, 2, links.ctypes.data, fr.ctypes.data, v.ctypes.data) != 0
    assert "rkFDUpdateInit" in fd.last_error()
    assert L.rkFDBatchGetLinkFrames(fd.h, 0, None, None, None) != 0
    assert "rkFDUpdateInit" in fd.last_error()
    assert L.rkFDBatchGetLinkFramesDevice(fd.h, 0, 2, links.ctypes.data, None, None) != 0
    assert "rkFDUpdateInit" in fd.last_error()
    with pytest.raises(RuntimeError, match="rkFDUpdateInit"):
        fd.batch_get_link_frames()
    assert fd.link_frame_kernel_count == 0
    assert not fr.any() and not v.any()
    fd.destroy()


@pytest.mark.parametrize("seed", [1, 2, 3, 4])
def test_walk_matches_oracle(seed):
    """every joint type, branching trees, a floating and a breakable-float root, general and structured org frames; broken
    and unbroken breakable-float joints"""
    w = random_world(seed)
    B = 24
    q, qd, piv = random_states(w, B, seed + 100)
    fr, vel = KinHarness(w).frames(q, qd, piv)
    brk = broken_links(w, piv)
    assert any(brk) and not all(brk)
    ofr, ovel = oracle_frames(w, q, qd, brk)
    assert_frames_close(fr, vel, ofr, ovel, "random world %d" % seed)


@pytest.mark.parametrize("name", ["c3", "c4_penalty"])
def test_walk_matches_oracle_workloads(name):
    w = ch.world_c3(base_z=0.3) if name == "c3" else ch.world_c4_penalty()
    B = 16
    q, qd, _ = ch.sample_state(w, B, seed=3)
    fr, vel = KinHarness(w).frames(q, qd)
    ofr, ovel = oracle_frames(w, q, qd)
    assert_frames_close(fr, vel, ofr, ovel, name)


def test_walk_after_steps_matches_oracle():
    """the brick wall after a committing evaluation and steps: the middle joint has broken, the others hold"""
    from test_kernel_core_host import brick_wall
    w = ch.World(chains=[brick_wall([200.0, 4.0, 10.0], [200.0, 0.3, 10.0]), ch.floor_soft()],
                 contact_info=[ch.ContactInfo("soft", "wall", "elastic", E=1000.0, V=10.0)])
    B = 4
    rng = np.random.default_rng(0)
    q = np.zeros((B, w.nq)); qd = np.zeros((B, w.nq))
    q[:, 9:12] = rng.uniform(-0.05, 0.05, (B, 3))
    hs = HostSim(w, B)
    hs.set_state(q, qd, np.zeros((B, w.nl)))
    hs.eval(ref=True)
    hs.step(40)
    gq, gqd, _ = hs.get_state()
    piv, _ = hs.get_pivot()
    brk = broken_links(w, piv)
    assert all(b == (2,) for b in brk)
    fr, vel = KinHarness(w).frames(gq, gqd, piv)
    ofr, ovel = oracle_frames(w, gq, gqd, brk)
    assert_frames_close(fr, vel, ofr, ovel, "brick wall")
    assert np.abs(vel[:, 2:, :3]).max() > 1e-3          # the falling bricks move


def test_walk_selection():
    """subsets, permutations and duplicates are the matching columns of the all-links walk, bit for bit; one output alone
    is the same as with the other"""
    w = random_world(5)
    B = 8
    q, qd, piv = random_states(w, B, 7)
    kh = KinHarness(w)
    fr, vel = kh.frames(q, qd, piv)
    for links in ([w.nl - 1], [3, 0, 3, w.nl - 2, w.nl - 1], list(range(w.nl))[::-1], [6] * 32):
        f2, v2 = kh.frames(q, qd, piv, links)
        assert np.array_equal(f2, fr[:, links]) and np.array_equal(v2, vel[:, links])
    f3, v3 = kh.frames(q, qd, piv, [2, 5], vel=False)
    assert v3 is None and np.array_equal(f3, fr[:, [2, 5]])
    f4, v4 = kh.frames(q, qd, piv, [2, 5], frames=False)
    assert f4 is None and np.array_equal(v4, vel[:, [2, 5]])
    for bad in ([w.nl], [-1], [0] * 33):
        with pytest.raises(RuntimeError):
            kh.frames(q, qd, piv, bad)
