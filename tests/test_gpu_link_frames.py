"""Link kinematics (rkFDBatchGetLinkFrames / rkFDBatchGetLinkFramesDevice) on the GPU: world frames and velocities of every
environment match the oracle on the state read back from the engine; re-sorted slots, shards, link selection and the device
variant do not change a bit; the calls write nothing of the engine's state."""
import numpy as np
import pytest

import rokifd_b200  # noqa: F401
from rokifd_b200 import chains as ch
from test_link_frames_host import assert_frames_close, broken_links, oracle_frames, random_world
from test_gpu_reset import brick_wall_world, brick_wall_states, num_shards, snapshot, assert_same, pick

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def capi():
    from rokifd_b200 import capi as c
    assert c.device_count() > 0, "no CUDA device: the product path has no CPU fallback"
    return c


def setup(name):
    """(world, B, sampler(B, seed) -> (q, qd, u))"""
    if name == "arm_box_floor":
        from test_kernel_core_host import flat_world, flat_states
        w, q0 = flat_world(name, soft=True)
        return w, 512, lambda B, seed: flat_states(name, w, q0, B, seed=seed)
    if name == "brick_wall":
        w = brick_wall_world()
        return w, 256, lambda B, seed: brick_wall_states(w, B, seed)
    if name == "random_tree":
        w = random_world(11)
        return w, 256, lambda B, seed: ch.sample_state(w, B, seed=seed)
    if name == "c4":
        w = ch.world_c4_penalty()
        return w, 256, lambda B, seed: ch.sample_c4_standing(w, B, seed=seed)
    w = {"c2": ch.world_c2, "c3": lambda: ch.world_c3(base_z=0.3), "c5_mlcp": lambda: ch.world_c5(base_z=0.3, solver="MLCP")}[name]()
    return w, 1024, lambda B, seed: ch.sample_state(w, B, seed=seed)


def start(capi, w, q, qd, u, devices=None, resort=None):
    fd, _ = capi.create_world(w, B=q.shape[0], devices=devices)
    if resort is not None:
        fd.batch_set_resort_interval(resort)
    fd.batch_set_state(q, qd); fd.batch_set_motor_input(u); fd.update_init()
    return fd


def steps(fd, k):
    for _ in range(k):         # one call per step: the engine re-sorts between calls
        fd.update()


@pytest.mark.parametrize("name", ["c2", "c3", "c4", "c5_mlcp", "arm_box_floor", "random_tree", "brick_wall"])
def test_link_frames_match_oracle(capi, name):
    w, B, sample = setup(name)
    q, qd, u = sample(B, 3)
    fd = start(capi, w, q, qd, u)
    steps(fd, 40)
    fr, vel = fd.batch_get_link_frames()
    assert fr.shape == (B, w.nl, 12) and vel.shape == (B, w.nl, 6)
    gq, gqd, _ = fd.batch_get_state()
    piv, _ = fd.batch_get_pivot()
    brk = broken_links(w, piv)
    if name == "brick_wall":
        assert any(brk) and not all(len(b) == 3 for b in brk)      # broken and unbroken joints
        assert all(2 in b and 1 not in b for b in brk)
    ofr, ovel = oracle_frames(w, gq, gqd, brk)
    assert_frames_close(fr, vel, ofr, ovel, name)
    fd.destroy()


def test_resort_and_shards_invisible(capi):
    """re-sorted slots (default interval) vs slot = environment, and two shards vs one: bit-identical"""
    w, B, sample = setup("c3")
    B = 4096
    q, qd, u = sample(B, 5)
    runs = {"sorted": start(capi, w, q, qd, u), "unsorted": start(capi, w, q, qd, u, resort=0),
            "two shards": start(capi, w, q, qd, u, devices=[0, 0])}
    if capi.device_count() >= 2:
        runs["two devices"] = start(capi, w, q, qd, u, devices=[0, 1])
    for fd in runs.values():
        steps(fd, 40)
    assert runs["sorted"].resort_count > 0 and runs["unsorted"].resort_count == 0
    assert num_shards(capi, runs["two shards"]) == 2
    ref = runs["sorted"].batch_get_link_frames()
    for k, fd in runs.items():
        fr, vel = fd.batch_get_link_frames()
        assert np.array_equal(fr, ref[0]) and np.array_equal(vel, ref[1]), k
    k0 = runs["two shards"].link_frame_kernel_count
    runs["two shards"].batch_get_link_frames([7])
    assert runs["two shards"].link_frame_kernel_count == k0 + 2        # one launch per shard
    for fd in runs.values():
        fd.destroy()


def test_selection_and_refusals(capi):
    import torch
    w, B, sample = setup("random_tree")
    q, qd, u = sample(B, 5)
    fd = start(capi, w, q, qd, u)
    steps(fd, 10)
    fr, vel = fd.batch_get_link_frames()
    nl = w.nl
    for links in ([nl - 1], [4, 0, 4, nl - 1, 2], list(range(nl))[::-1], [3] * 32, None):
        f2, v2 = fd.batch_get_link_frames(links)
        cols = list(range(nl)) if links is None else links
        assert np.array_equal(f2, fr[:, cols]) and np.array_equal(v2, vel[:, cols]), links
    f3, v3 = fd.batch_get_link_frames([1, 5], vel=False)
    assert v3 is None and np.array_equal(f3, fr[:, [1, 5]])
    f4, v4 = fd.batch_get_link_frames([1, 5], frames=False)
    assert f4 is None and np.array_equal(v4, vel[:, [1, 5]])
    # device variant: a NULL output leaves that buffer untouched; refused calls leave both untouched
    dev = torch.device("cuda", 0)
    tf = torch.full((B, 2, 12), 7.25, dtype=torch.float64, device=dev)
    tv = torch.full((B, 2, 6), 7.25, dtype=torch.float64, device=dev)
    fd.batch_get_link_frames_device(0, [1, 5], tf.data_ptr(), None)
    fd.batch_sync()
    assert np.array_equal(tf.cpu().numpy(), fr[:, [1, 5]]) and (tv == 7.25).all()
    tf.fill_(7.25)
    fd.batch_get_link_frames_device(0, [1, 5], None, tv.data_ptr())
    fd.batch_sync()
    assert np.array_equal(tv.cpu().numpy(), vel[:, [1, 5]]) and (tf == 7.25).all()
    tv.fill_(7.25)
    k0 = fd.link_frame_kernel_count
    for shard, links in ((0, [nl]), (0, [-1]), (0, [0] * 33), (1, [0]), (-1, [0])):
        with pytest.raises(RuntimeError):
            fd.batch_get_link_frames_device(shard, links, tf.data_ptr(), tv.data_ptr())
    with pytest.raises(RuntimeError):
        fd.batch_get_link_frames([nl])
    fd.batch_get_link_frames([])                                    # nlink = 0: nothing
    fd.batch_sync()
    assert (tf == 7.25).all() and (tv == 7.25).all()
    assert fd.link_frame_kernel_count == k0
    fd.destroy()


def test_device_variant_stream_ordered(capi):
    """the device call on the engine's stream: bit-identical to the host call, ordered after the steps queued before it
    without waiting for them"""
    import torch
    w, B, sample = setup("c3")
    B = 4096
    q, qd, u = sample(B, 7)
    fd = start(capi, w, q, qd, u)
    steps(fd, 20)
    dev = torch.device("cuda", 0)
    stream = torch.cuda.Stream(device=dev)
    fd.batch_set_stream(stream.cuda_stream)
    links = [7, 0, 3]
    tf = torch.zeros((B, 3, 12), dtype=torch.float64, device=dev)
    tv = torch.zeros((B, 3, 6), dtype=torch.float64, device=dev)
    fd.batch_get_link_frames_device(0, links, tf.data_ptr(), tv.data_ptr())
    fd.batch_sync()
    fr, vel = fd.batch_get_link_frames(links)
    assert np.array_equal(tf.cpu().numpy(), fr) and np.array_equal(tv.cpu().numpy(), vel)
    torch.cuda.synchronize()
    k0 = fd.link_frame_kernel_count
    with torch.cuda.stream(stream):
        torch.cuda._sleep(100_000_000)            # ~50 ms of work ahead of the steps on the engine's stream
    fd.update_n(3)
    fd.batch_get_link_frames_device(0, links, tf.data_ptr(), tv.data_ptr())
    assert not stream.query()                     # returned while the stream was still busy
    assert fd.link_frame_kernel_count == k0 + 1
    stream.synchronize()
    fr, vel = fd.batch_get_link_frames(links)     # the post-step state
    assert np.array_equal(tf.cpu().numpy(), fr) and np.array_equal(tv.cpu().numpy(), vel)
    fd.destroy()


def test_read_only(capi):
    """calls between steps change nothing (state, contact state, status); after a reset, the frames of the reset environments
    are those of a new simulator started from the same states"""
    w, B, sample = setup("c3")
    q, qd, u = sample(B, 9)
    fd, twin = start(capi, w, q, qd, u), start(capi, w, q, qd, u)
    for _ in range(5):
        fd.batch_get_link_frames()
        fd.batch_get_link_frames([7], vel=False)
        steps(fd, 8); steps(twin, 8)
    assert_same(snapshot(fd), np.arange(B), snapshot(twin), np.arange(B), "with link-frame calls vs without")
    envs = pick(B, 0.1, 3)
    nq_, nqd_, nu_ = [a[:len(envs)] for a in sample(B, 13)]
    fd.batch_reset_envs(envs, nq_, nqd_, nu_)
    fresh = start(capi, w, nq_, nqd_, nu_)
    fr, vel = fd.batch_get_link_frames()
    ffr, fvel = fresh.batch_get_link_frames()
    assert np.array_equal(fr[envs], ffr) and np.array_equal(vel[envs], fvel)
    for x in (fd, twin, fresh):
        x.destroy()
