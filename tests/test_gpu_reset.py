"""Environment reset (rkFDBatchResetEnvs / rkFDBatchResetEnvsDevice) on the GPU: a reset environment is bit for bit the
environment of a new simulator started from the same state (right after the call and in every later step), and the
environments not listed are bit for bit those of a run without the call."""
import numpy as np
import pytest

import rokifd_b200  # noqa: F401
from rokifd_b200 import chains as ch
from gpu_batch import capi, start, steps, snapshot, assert_same, pick, num_shards  # noqa: F401
from workloads import world

pytestmark = pytest.mark.gpu

BATCH = {"c2": 4096, "c3": 4096, "c4_penalty": 2048, "c4_volume": 2048, "c5_mlcp": 4096, "c5_vert": 4096, "arm_box_floor": 2048,
         "brick_wall": 256}


def setup(name):
    """(world, B, sampler(B, seed) -> (q, qd, u), the world re-sorts its slots)"""
    w, sample = world(name)
    return w, BATCH[name], sample, name != "c2"


def check_reset(capi, name, with_u, frac=0.1, devices=None, B=None):
    w, B0, sample, sorts = setup(name)
    B = B or B0
    q, qd, u = sample(B, 11)
    fd, twin = start(capi, w, q, qd, u, devices), start(capi, w, q, qd, u, devices)
    steps(fd, 40); steps(twin, 40)
    if sorts:
        assert fd.resort_count > 0
    envs = pick(B, frac, 5) if frac < 1 else np.random.default_rng(5).permutation(B).astype(np.int32)
    others = np.setdiff1d(np.arange(B), envs)
    nq_, nqd_, nu_ = sample(B, 23)
    nq_, nqd_, nu_ = nq_[:len(envs)], nqd_[:len(envs)], nu_[:len(envs)]
    launches = fd.launch_count
    fd.batch_reset_envs(envs, nq_, nqd_, nu_ if with_u else None)
    assert fd.launch_count == launches + num_shards(capi, fd)     # one step-kernel launch per shard
    fresh = start(capi, w, nq_, nqd_, nu_ if with_u else u[envs])
    for seg in range(2):
        s, t, f = snapshot(fd), snapshot(twin), snapshot(fresh)
        assert_same(s, envs, f, np.arange(len(envs)), "%s: reset vs new simulator after %d steps" % (name, 30 * seg))
        assert_same(s, others, t, others, "%s: other environments after %d steps" % (name, 30 * seg))
        if seg == 0:
            steps(fd, 30); steps(twin, 30); steps(fresh, 30)
    return fd, twin, fresh, envs, s


@pytest.mark.parametrize("name,with_u", [("c3", True), ("c3", False), ("c2", True), ("c4_penalty", False), ("c5_mlcp", True),
                                         ("c5_vert", False), ("c4_volume", True), ("arm_box_floor", False), ("brick_wall", True)])
def test_reset_equals_new_simulator(capi, name, with_u):
    fd, twin, fresh, envs, s = check_reset(capi, name, with_u)
    if name == "brick_wall":
        # the middle joint breaks in the committing evaluation at t=0: broken again after the reset, not merely cleared
        assert (s["piv_type"][envs][:, [0, 6, 12]] == [0, 1, 0]).all()
    if name in ("c3", "c4_volume", "arm_box_floor"):
        assert s["active"][envs].sum() > 0            # the reset environments are in contact again
    for x in (fd, twin, fresh):
        x.destroy()


def test_reset_from_device_arrays(capi):
    """rkFDBatchResetEnvsDevice with ids and states in torch CUDA tensors: bit-identical to the host variant, and the call is
    ordered on the engine's stream without waiting for it."""
    import torch
    w, B, sample, _ = setup("c3")
    q, qd, u = sample(B, 11)
    fd_h, fd_d = start(capi, w, q, qd, u), start(capi, w, q, qd, u)
    steps(fd_h, 40); steps(fd_d, 40)
    envs = pick(B, 0.1, 7)
    nq_, nqd_, nu_ = [a[:len(envs)] for a in sample(B, 29)]
    fd_h.batch_reset_envs(envs, nq_, nqd_, nu_)
    dev = torch.device("cuda", 0)
    te = torch.from_numpy(envs).to(dev)
    tq, tqd, tu = [torch.from_numpy(np.ascontiguousarray(a)).to(dev) for a in (nq_, nqd_, nu_)]
    stream = torch.cuda.Stream(device=dev)
    fd_d.batch_set_stream(stream.cuda_stream)
    torch.cuda.synchronize()
    k0 = fd_d.reset_kernel_count
    fd_d.batch_reset_envs_device(0, len(envs), te.data_ptr(), tq.data_ptr(), tqd.data_ptr(), tu.data_ptr())     # allocates
    assert fd_d.reset_kernel_count == k0 + 3
    with torch.cuda.stream(stream):
        torch.cuda._sleep(100_000_000)            # ~50 ms of work ahead of the reset on the engine's stream
    fd_d.batch_reset_envs_device(0, len(envs), te.data_ptr(), tq.data_ptr(), tqd.data_ptr(), tu.data_ptr())     # the same reset again
    assert not stream.query()                     # returned while the stream was still busy
    stream.synchronize()
    a, b = snapshot(fd_h), snapshot(fd_d)
    assert_same(a, np.arange(B), b, np.arange(B), "device variant vs host variant")
    steps(fd_h, 20); steps(fd_d, 20)
    a, b = snapshot(fd_h), snapshot(fd_d)
    assert_same(a, np.arange(B), b, np.arange(B), "device variant vs host variant after 20 steps")
    # indices outside [0, B) are skipped on the device
    bad = torch.tensor([-1, B, B + 100], dtype=torch.int32, device=dev)
    torch.cuda.synchronize()
    fd_d.batch_reset_envs_device(0, 3, bad.data_ptr(), tq.data_ptr())
    fd_d.batch_sync()
    assert_same(a, np.arange(B), snapshot(fd_d), np.arange(B), "out-of-range device indices")
    for x in (fd_h, fd_d):
        x.destroy()


def test_reset_edge_cases(capi):
    w, B, sample, _ = setup("c3")
    B = 1024
    q, qd, u = sample(B, 11)
    fd, twin = start(capi, w, q, qd, u), start(capi, w, q, qd, u)
    steps(fd, 40); steps(twin, 40)
    # n = 0: nothing is launched
    l0, k0 = fd.launch_count, fd.reset_kernel_count
    fd.batch_reset_envs(np.zeros(0, np.int32), np.zeros((0, w.nq)))
    fd.batch_reset_envs_device(0, 0, 0, 0)
    assert (fd.launch_count, fd.reset_kernel_count) == (l0, k0)
    # refused calls change nothing
    q1 = np.zeros((2, w.nq))
    for envs in ([0, B], [-1, 3], [5, 5]):
        with pytest.raises(RuntimeError):
            fd.batch_reset_envs(np.array(envs, np.int32), q1)
    with pytest.raises(RuntimeError):
        fd.batch_reset_envs(np.array([1, 2], np.int32), None)
    with pytest.raises(RuntimeError):
        fd.batch_reset_envs_device(1, 0, 0, 0)
    assert (fd.launch_count, fd.reset_kernel_count) == (l0, k0)
    assert_same(snapshot(fd), np.arange(B), snapshot(twin), np.arange(B), "after refused calls")
    steps(fd, 10); steps(twin, 10)
    assert_same(snapshot(fd), np.arange(B), snapshot(twin), np.arange(B), "10 steps after refused calls")
    fd.destroy(); twin.destroy()
    # n = B: every environment as in a new simulator
    for x in check_reset(capi, "c3", True, frac=1.0, B=1024)[:3]:
        x.destroy()


def test_reset_longer_than_one_chunk(capi):
    """70,000 environments of C2 (the sub-state holds 65,536): two chunks, each one step-kernel launch"""
    w = ch.world_c2()
    B = 72000
    q, qd, u = ch.sample_state(w, B, seed=3)
    fd, twin = start(capi, w, q, qd, u), start(capi, w, q, qd, u)
    steps(fd, 5); steps(twin, 5)
    envs = np.random.default_rng(1).permutation(B)[:70000].astype(np.int32)
    others = np.setdiff1d(np.arange(B), envs)
    nq_, nqd_, _ = [a[:len(envs)] for a in ch.sample_state(w, B, seed=4)]
    l0, k0 = fd.launch_count, fd.reset_kernel_count
    fd.batch_reset_envs(envs, nq_, nqd_)
    assert fd.launch_count == l0 + 2 and fd.reset_kernel_count == k0 + 6
    fresh = start(capi, w, nq_, nqd_, u[envs])
    for seg in range(2):
        s, t, f = snapshot(fd), snapshot(twin), snapshot(fresh)
        assert_same(s, envs, f, np.arange(len(envs)), "C2 70,000: reset vs new simulator")
        assert_same(s, others, t, others, "C2 70,000: other environments")
        steps(fd, 5); steps(twin, 5); steps(fresh, 5)
    for x in (fd, twin, fresh):
        x.destroy()


def test_reset_across_shards(capi):
    """a list that spans two shards: two GPUs when present, else two shards on device 0"""
    devices = [0, 1] if capi.device_count() >= 2 else [0, 0]
    fd, twin, fresh, envs, _ = check_reset(capi, "c3", True, devices=devices)
    assert num_shards(capi, fd) == 2
    half = fd.env_num // 2
    assert (envs < half).any() and (envs >= half).any()
    for x in (fd, twin, fresh):
        x.destroy()
