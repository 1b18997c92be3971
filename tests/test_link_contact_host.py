"""Link contact wrench (rkFDBatchGetLinkContactWrench / -Device) without a device: the C-ABI declarations, the calls refused
without rkFDUpdateInit, and the readout (roki-fd_b200/csrc/rkfd_link_contact.cuh, compiled with g++ beside the host harness:
tests/link_contact/hostsim_link_contact.cpp) against the oracle's per-link contact wrench after one step from the harness's
state."""
import ctypes as C

import numpy as np
import pytest

import rokifd_b200  # noqa: F401
from rokifd_b200 import capi
from rokifd_b200 import chains as ch
from hostsim_py import HostSim
from link_contact_py import WORLDS, assert_matches_oracle, assert_wrench_close, harness_link_contact, oracle_step_wrench, restate, world

B = 24          # environments per world (the oracle runs one at a time)
# harness steps before the compared step (300 elsewhere): broken bricks reach the floor, the rest touch early
SETTLE = {"brick_wall": 700, "box_stack": 60, "box_stack_rigid_mlcp": 60, "box_stack_rigid_vert": 60, "arm_box_floor": 60}


def run(name, seed=3, oracle=True, settle=None):
    """the harness after SETTLE steps, the oracle's wrench after one step from that state, and the harness after the same step"""
    w, sample = world(name)
    q, qd, u = sample(B, seed)
    hs = HostSim(w, B)
    hs.set_state(q, qd, u)
    hs.eval(ref=True)
    hs.step(settle or SETTLE.get(name, 300))
    gq, gqd, _ = hs.get_state()
    a, t, r, _ = hs.get_contact()
    pt, pp = hs.get_pivot()
    ref = oracle_step_wrench(w, gq, gqd, u, a, t, r, pt, pp) if oracle else None
    hs.step(1)
    return w, hs, ref


def test_link_contact_signatures_declared():
    L = capi.lib()
    assert L.rkFDBatchGetLinkContactWrench.restype is C.c_int and len(L.rkFDBatchGetLinkContactWrench.argtypes) == 4
    assert L.rkFDBatchGetLinkContactWrenchDevice.restype is C.c_int and len(L.rkFDBatchGetLinkContactWrenchDevice.argtypes) == 5
    assert L.rkFDBatchLinkContactKernelCount.restype is C.c_longlong and len(L.rkFDBatchLinkContactKernelCount.argtypes) == 1


def test_link_contact_needs_an_engine():
    fd, _ = capi.create_world(ch.world_c3(base_z=0.1), B=4)
    L = capi.lib()
    links = np.array([0, 7], np.int32)
    w = np.zeros((4, 2, 6))
    assert L.rkFDBatchGetLinkContactWrench(fd.h, 2, links.ctypes.data, w.ctypes.data) != 0
    assert "rkFDUpdateInit" in fd.last_error()
    assert L.rkFDBatchGetLinkContactWrench(fd.h, 0, None, None) != 0
    assert "rkFDUpdateInit" in fd.last_error()
    assert L.rkFDBatchGetLinkContactWrenchDevice(fd.h, 0, 2, links.ctypes.data, w.ctypes.data) != 0
    assert "rkFDUpdateInit" in fd.last_error()
    with pytest.raises(RuntimeError, match="rkFDUpdateInit"):
        fd.batch_get_link_contact_wrench()
    assert fd.link_contact_kernel_count == 0
    assert not w.any()
    fd.destroy()


@pytest.mark.parametrize("name", sorted(WORLDS))
def test_readout_matches_oracle(name):
    w, hs, (ref, _) = run(name)
    got = harness_link_contact(hs)
    assert got.shape == (B, w.nl, 6)
    assert np.abs(ref).max() > 0, "no contact in %s" % name
    assert_matches_oracle(got, ref, name)


@pytest.mark.parametrize("name", ["c4_penalty"])
def test_pulling_contacts_left_out(name):
    """elastic slots whose penalty force points into the floor (its normal is +z) are in the contact forces but were never
    applied: there the naive sum of the forces differs from the readout, and the readout is the oracle's.  150 steps in, the
    soles of the biped bounce"""
    w, hs, (ref, _) = run(name, settle=150)
    a, _, _, f = hs.get_contact()
    pull = ((a == 1) & (f[:, :, 2] < 0)).any(1)
    assert pull.any(), "no pulling contact in %s" % name
    got = harness_link_contact(hs)
    naive = f.sum(1)                                # every slot is a vertex of a moving link against the floor
    total = got[:, :, :3].sum(1)
    assert not np.allclose(total[pull], naive[pull], rtol=0, atol=1e-9)
    assert np.allclose(total[~pull], naive[~pull], rtol=1e-12, atol=1e-9)
    assert_wrench_close(got[pull], ref[pull], WORLDS[name], name)


def test_selection_and_refusals():
    w, hs, _ = run("c4_penalty")
    nl = w.nl
    full = harness_link_contact(hs)
    for links in ([nl - 1], [4, 0, 4, nl - 1, 2], list(range(nl))[::-1], [3] * 32, None):
        got = harness_link_contact(hs, links)
        cols = list(range(nl)) if links is None else links
        assert np.array_equal(got, full[:, cols]), links
    assert harness_link_contact(hs, []).shape == (B, 0, 6)
    for links in ([nl], [-1], [0] * 33):
        with pytest.raises(RuntimeError):
            harness_link_contact(hs, links)


@pytest.mark.parametrize("name", ["c3", "c4_penalty", "c4_volume", "c5_mlcp", "brick_wall"])
def test_numpy_restatement(name):
    """the numpy restatement the GPU tests use agrees with the harness's readout (the brick wall, broken and unbroken joints, is
    checked here only: the oracle keeps a broken joint's state apart from its pivot bits, so it cannot be loaded mid-run)"""
    w, hs, _ = run(name, oracle=name != "brick_wall")
    if name == "brick_wall":
        brk = (hs.get_pivot()[0][:, [0, 6, 12]] == 1).sum(1)
        assert (brk > 0).any() and (brk < 3).any()
    q, qd, _ = hs.get_state()
    pt, _ = hs.get_pivot()
    fr, _ = hs.link_frames(q, qd, pt, vel=False)
    _, _, _, f = hs.get_contact()
    assert_wrench_close(harness_link_contact(hs), restate(w, f, fr), 1e-12, name)
