"""Link kinematics (rkFDBatchGetLinkFrames / rkFDBatchGetLinkFramesDevice) without a device: the C-ABI declarations, the calls
refused without rkFDUpdateInit, and the arithmetic of the kinematics walk (roki-fd_b200/csrc/rkfd_kin.cuh, compiled into the
host harness tests/hostsim/hostsim.cpp) against the oracle's link frames and velocities."""
import ctypes as C

import numpy as np
import pytest

import rokifd_b200  # noqa: F401
from rokifd_b200 import capi
from rokifd_b200 import chains as ch
from hostsim_py import HostSim
from workloads import NDOF, assert_frames_close, brick_wall_world, broken_links, oracle_frames, random_world


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
    fr, vel = HostSim(w, 1).link_frames(q, qd, piv)
    brk = broken_links(w, piv)
    assert any(brk) and not all(brk)
    ofr, ovel = oracle_frames(w, q, qd, brk)
    assert_frames_close(fr, vel, ofr, ovel, "random world %d" % seed)


@pytest.mark.parametrize("name", ["c3", "c4_penalty"])
def test_walk_matches_oracle_workloads(name):
    w = ch.world_c3(base_z=0.3) if name == "c3" else ch.world_c4_penalty()
    B = 16
    q, qd, _ = ch.sample_state(w, B, seed=3)
    fr, vel = HostSim(w, 1).link_frames(q, qd)
    ofr, ovel = oracle_frames(w, q, qd)
    assert_frames_close(fr, vel, ofr, ovel, name)


def test_walk_after_steps_matches_oracle():
    """the brick wall after a committing evaluation and steps: the middle joint has broken, the others hold"""
    w = brick_wall_world([200.0, 4.0, 10.0], [200.0, 0.3, 10.0])
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
    fr, vel = hs.link_frames(gq, gqd, piv)
    ofr, ovel = oracle_frames(w, gq, gqd, brk)
    assert_frames_close(fr, vel, ofr, ovel, "brick wall")
    assert np.abs(vel[:, 2:, :3]).max() > 1e-3          # the falling bricks move


def test_walk_selection():
    """subsets, permutations and duplicates are the matching columns of the all-links walk, bit for bit; one output alone
    is the same as with the other"""
    w = random_world(5)
    B = 8
    q, qd, piv = random_states(w, B, 7)
    kh = HostSim(w, 1)
    fr, vel = kh.link_frames(q, qd, piv)
    for links in ([w.nl - 1], [3, 0, 3, w.nl - 2, w.nl - 1], list(range(w.nl))[::-1], [6] * 32):
        f2, v2 = kh.link_frames(q, qd, piv, links)
        assert np.array_equal(f2, fr[:, links]) and np.array_equal(v2, vel[:, links])
    f3, v3 = kh.link_frames(q, qd, piv, [2, 5], vel=False)
    assert v3 is None and np.array_equal(f3, fr[:, [2, 5]])
    f4, v4 = kh.link_frames(q, qd, piv, [2, 5], frames=False)
    assert f4 is None and np.array_equal(v4, vel[:, [2, 5]])
    for bad in ([w.nl], [-1], [0] * 33):
        with pytest.raises(RuntimeError):
            kh.link_frames(q, qd, piv, bad)
