"""Link contact wrench (rkFDBatchGetLinkContactWrench / rkFDBatchGetLinkContactWrenchDevice) on the GPU: one engine step against
one oracle step from the engine's own state, a numpy restatement from the engine's contact forces and link frames on every
environment, a box at rest, invariance under re-sort, shards and the device variant, stream ordering, and no effect on the run."""
import numpy as np
import pytest

import rokifd_b200  # noqa: F401
from rokifd_b200 import chains as ch
from gpu_batch import capi, start, steps, snapshot, assert_same, pick, num_shards  # noqa: F401
from link_contact_py import WORLDS, assert_matches_oracle, assert_wrench_close, oracle_step_wrench, restate, world

pytestmark = pytest.mark.gpu

SETTLE = {"brick_wall": 700, "box_stack": 60, "box_stack_rigid_mlcp": 60, "box_stack_rigid_vert": 60, "arm_box_floor": 60}


@pytest.mark.parametrize("name", sorted(set(WORLDS) - {"box_stack_rigid_vert"}))
def test_one_step_against_oracle(capi, name):
    """after N engine steps: the engine's state, contact state, pivots and input loaded into the oracle, one step of each (the
    dense Vert path of the rigid box stack, which serves the environments of a warp one after the other, is checked on the host
    harness, tests/test_link_contact_host.py)"""
    w, sample = world(name)
    B = 128
    q, qd, u = sample(B, 5)
    fd = start(capi, w, q, qd, u)
    steps(fd, SETTLE.get(name, 300))
    gq, gqd, _ = fd.batch_get_state()
    a, t, r, _ = fd.batch_get_contact()
    pt, pp = fd.batch_get_pivot()
    ref, _ = oracle_step_wrench(w, gq, gqd, u, a, t, r, pt, pp)
    fd.update()
    got = fd.batch_get_link_contact_wrench()
    assert got.shape == (B, w.nl, 6) and np.abs(ref).max() > 0
    assert_matches_oracle(got, ref, name)
    fd.destroy()


@pytest.mark.parametrize("name", ["c3", "c4_penalty", "c4_volume", "c5_mlcp", "c5_vert", "brick_wall"])
def test_numpy_restatement(capi, name):
    """on every environment: the readout from the engine's contact forces (rkFDBatchGetContactForce), link frames and the
    world's vertices, with the dot(f, n) < 0 exclusion and the Volume layout"""
    w, sample = world(name)
    B = 2048
    q, qd, u = sample(B, 7)
    fd = start(capi, w, q, qd, u)
    steps(fd, SETTLE.get(name, 300))
    fr, _ = fd.batch_get_link_frames(vel=False)
    f = fd.batch_get_contact()[3]
    got = fd.batch_get_link_contact_wrench()
    assert np.abs(got).max() > 0
    ok = np.ones(B, bool)
    if name == "c4_volume":             # status bit 2: more colliding pairs than the Volume solver takes (rows unspecified)
        ok = (fd.batch_get_status() & 4) == 0
    assert_wrench_close(got[ok], restate(w, f, fr)[ok], 1e-12, name)
    fd.destroy()


def test_external_wrench_excluded(capi):
    """a declared external wrench on the contact link changes the motion, not what the readout sums"""
    w, sample = world("c3")
    B = 1024
    q, qd, u = sample(B, 9)
    W = np.random.default_rng(9).uniform(-10, 10, (B, 1, 6)); W[:, 0, 2] -= 20.0
    fd = start(capi, w, q, qd, u, ext=([7], W))
    steps(fd, 300)
    fr, _ = fd.batch_get_link_frames(vel=False)
    got = fd.batch_get_link_contact_wrench()
    assert np.abs(got[:, 7]).max() > 0
    assert_wrench_close(got, restate(w, fd.batch_get_contact()[3], fr), 1e-12, "c3 with an external wrench")
    fd.destroy()


@pytest.mark.parametrize("half,solver", [("soft", "Vert"), ("hard", "MLCP"), ("hard", "Vert")])
def test_box_at_rest(capi, half, solver):
    """C1's box after 3,000 steps (3 s) on one half of floor_hardsoft.  On the soft half (elastic pair, penalty path) it rests:
    net contact force (0, 0, m g) and no torque about the centre of mass, within 1 % of m g (force) and of m g times 0.1 m
    (torque).  On the hard half (rigid pair) neither rigid solver brings it to rest - it keeps rocking on its corners, and the
    committing evaluation's force is not m g - so there the readout is checked against the oracle's step from the same state"""
    w = ch.world_c1_box(solver=solver)
    l = w.flat_links()[0]
    B = 32
    rng = np.random.default_rng(3)
    zmin = min(np.asarray(v, float).reshape(-1, 3)[:, 2].min() for v in l.cells())
    q = np.zeros((B, w.nq)); q[:, 0] = rng.uniform(-0.5, 0.5, B); q[:, 1] = (-1.25 if half == "soft" else 1.25) + rng.uniform(-0.3, 0.3, B)
    q[:, 2] = -zmin + 0.002
    u = np.zeros((B, w.nl))
    fd = start(capi, w, q, np.zeros((B, w.nq)), u)
    fd.update_n(3000)
    if half == "hard":
        gq, gqd, _ = fd.batch_get_state()
        a, t, r, _ = fd.batch_get_contact()
        pt, pp = fd.batch_get_pivot()
        ref, _ = oracle_step_wrench(w, gq, gqd, u, a, t, r, pt, pp)
        fd.update()
        got = fd.batch_get_link_contact_wrench()
        assert np.abs(ref[:, 0, 2]).min() > 0
        assert_matches_oracle(got, ref, "c5_" + solver.lower())      # the tolerances of the rigid solvers
        fd.destroy()
        return
    got = fd.batch_get_link_contact_wrench([0])[:, 0]
    fr, _ = fd.batch_get_link_frames([0], vel=False)
    R, o = fr[:, 0, :9].reshape(B, 3, 3), fr[:, 0, 9:]
    c = o + np.einsum("bij,j->bi", R, np.asarray(l.com, float))
    mg = l.mass * 9.80665
    tc = got[:, 3:] + np.cross(o - c, got[:, :3])
    assert np.abs(got[:, :3] - np.array([0, 0, mg])).max() <= 1e-2 * mg
    assert np.abs(tc).max() <= 1e-2 * mg * 0.1
    fd.destroy()


def test_invariance(capi):
    """re-sort on and off, one shard and two, host and device variants: bit-identical"""
    import torch
    w, sample = world("c4_penalty")
    B = 4096
    q, qd, u = sample(B, 5)
    runs = {"sorted": start(capi, w, q, qd, u), "unsorted": start(capi, w, q, qd, u, resort=0),
            "two shards": start(capi, w, q, qd, u, devices=[0, 0])}
    for fd in runs.values():
        steps(fd, 150)
    assert runs["sorted"].resort_count > 0 and runs["unsorted"].resort_count == 0
    assert num_shards(capi, runs["two shards"]) == 2
    ref = runs["sorted"].batch_get_link_contact_wrench()
    assert np.abs(ref).max() > 0
    for k, fd in runs.items():
        assert np.array_equal(fd.batch_get_link_contact_wrench(), ref), k
    links = [6, 3, 6, 0]
    assert np.array_equal(runs["sorted"].batch_get_link_contact_wrench(links), ref[:, links])
    k0 = runs["two shards"].link_contact_kernel_count
    runs["two shards"].batch_get_link_contact_wrench([3])
    assert runs["two shards"].link_contact_kernel_count == k0 + 2        # one launch per shard
    fd = runs["sorted"]
    tw = torch.full((B, 4, 6), 7.25, dtype=torch.float64, device="cuda")
    fd.batch_get_link_contact_wrench_device(0, links, tw.data_ptr())
    fd.batch_sync()
    assert np.array_equal(tw.cpu().numpy(), ref[:, links])
    tw.fill_(7.25)
    k0 = fd.link_contact_kernel_count
    for shard, ls in ((0, [w.nl]), (0, [-1]), (0, [0] * 33), (1, [0]), (-1, [0])):
        with pytest.raises(RuntimeError):
            fd.batch_get_link_contact_wrench_device(shard, ls, tw.data_ptr())
    fd.batch_get_link_contact_wrench([])
    fd.batch_sync()
    assert (tw == 7.25).all() and fd.link_contact_kernel_count == k0
    for fd in runs.values():
        fd.destroy()


def test_device_variant_stream_ordered(capi):
    """the device call on the engine's stream: ordered after the steps queued before it without waiting for them"""
    import torch
    w, sample = world("c4_penalty")
    B = 4096
    q, qd, u = sample(B, 7)
    fd = start(capi, w, q, qd, u)
    steps(fd, 150)
    dev = torch.device("cuda", 0)
    stream = torch.cuda.Stream(device=dev)
    fd.batch_set_stream(stream.cuda_stream)
    links = [3, 6]
    tw = torch.zeros((B, 2, 6), dtype=torch.float64, device=dev)
    torch.cuda.synchronize()
    k0 = fd.link_contact_kernel_count
    with torch.cuda.stream(stream):
        torch.cuda._sleep(100_000_000)            # ~50 ms of work ahead of the steps on the engine's stream
    fd.update_n(3)
    fd.batch_get_link_contact_wrench_device(0, links, tw.data_ptr())
    assert not stream.query()                     # returned while the stream was still busy
    assert fd.link_contact_kernel_count == k0 + 1
    stream.synchronize()
    ref = fd.batch_get_link_contact_wrench(links)  # the post-step state
    assert np.abs(ref).max() > 0 and np.array_equal(tw.cpu().numpy(), ref)
    fd.destroy()


def test_read_only(capi):
    """calls between steps change nothing; after a reset, the reset environments report what a new simulator started from the
    same states reports"""
    w, sample = world("c4_penalty")
    B = 1024
    q, qd, u = sample(B, 9)
    fd, twin = start(capi, w, q, qd, u), start(capi, w, q, qd, u)
    for _ in range(5):
        fd.batch_get_link_contact_wrench()
        fd.batch_get_link_contact_wrench([3])
        steps(fd, 8); steps(twin, 8)
    assert_same(snapshot(fd), np.arange(B), snapshot(twin), np.arange(B), "with link-contact calls vs without")
    envs = pick(B, 0.1, 3)
    nq_, nqd_, nu_ = [a[:len(envs)] for a in sample(B, 13)]
    fd.batch_reset_envs(envs, nq_, nqd_, nu_)
    fresh = start(capi, w, nq_, nqd_, nu_)
    got, ref = fd.batch_get_link_contact_wrench(), fresh.batch_get_link_contact_wrench()
    assert np.abs(ref).max() > 0 and np.array_equal(got[envs], ref)
    for x in (fd, twin, fresh):
        x.destroy()
