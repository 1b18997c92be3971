"""External wrenches (rkFDBatchSetExtWrenchLinks / rkFDBatchSetExtWrench / rkFDBatchSetExtWrenchDevice) on the GPU: every
contact solver against the oracle, the kernel choice, zero wrenches against the undeclared world, re-sorted slots and shards,
the device setter, the t = 0 evaluation, resets and a hovering body."""
import numpy as np
import pytest

import rokifd_b200  # noqa: F401
from ext_wrench_py import oracle_run
from gpu_batch import capi, start, steps, state  # noqa: F401
from workloads import free_body, world

pytestmark = pytest.mark.gpu

LINKS = {"c2": [7], "c3": [7, 3], "c4": [0, 3], "c4_volume": [0], "c5_mlcp": [7, 4], "c5_vert": [7], "arm_box_floor": [3, 2],
         "random_tree": [0, 5, 12], "brick_wall": [3]}
TOL = {"c5_vert": 1e-7, "c4_volume": 1e-6}
BATCH = {"c2": 1024, "c3": 1024, "c4": 256, "c4_volume": 512, "c5_mlcp": 1024, "c5_vert": 512, "arm_box_floor": 512,
         "random_tree": 256, "brick_wall": 256}


def setup(name):
    """(world, B, sampler(B, seed) -> (q, qd, u, W)); W: per-environment wrenches on LINKS[name]"""
    w, sample = world(name)
    n = len(LINKS[name])

    def sample_w(B, seed):
        q, qd, u = sample(B, seed)
        rng = np.random.default_rng(seed + 1000)
        W = np.concatenate([rng.uniform(-15, 15, (B, n, 3)), rng.uniform(-1, 1, (B, n, 3))], axis=2)
        return q, qd, u, W
    return w, BATCH[name], sample_w


@pytest.mark.parametrize("name", list(LINKS))
def test_matches_oracle(capi, name):
    w, B, sample = setup(name)
    q, qd, u, W = sample(B, 3)
    links = LINKS[name]
    fd = start(capi, w, q, qd, u, ext=(links, W))
    n = 40
    steps(fd, n)
    gq, gqd, _ = fd.batch_get_state()
    sel = np.r_[0:32, B - 16:B]
    oq, oqd, _, _ = oracle_run(w, q[sel], qd[sel], u[sel], links, W[sel], n)
    for a, b, what in ((gq[sel], oq, "q"), (gqd[sel], oqd, "q'")):
        err = np.abs(a - b).max() / max(np.abs(b).max(), 1.0)
        assert err < TOL.get(name, 1e-9), (name, what, err)
    ref = start(capi, w, q, qd, u)
    steps(ref, n)
    assert np.abs(ref.batch_get_state()[0] - gq).max() > 1e-6          # the wrench moved the worlds
    fd.destroy(); ref.destroy()


def test_declared_world_runs_the_generic_kernel(capi):
    w, B, sample = setup("c3")
    q, qd, u, W = sample(256, 1)
    plain, decl = start(capi, w, q, qd, u), start(capi, w, q, qd, u, ext=([7], W[:, :1]))
    assert plain.kernel_variant()[3] == 5
    assert decl.kernel_variant()[3] in (0, 11)
    plain.destroy(); decl.destroy()


@pytest.mark.parametrize("name", ["c3", "c4_volume"])
def test_zero_wrench_is_bit_identical(capi, name, monkeypatch):
    """declared links with zero wrenches step like the undeclared world forced onto the same kernel variant"""
    w, B, sample = setup(name)
    q, qd, u, W = sample(B, 4)
    decl = start(capi, w, q, qd, u, ext=(LINKS[name], np.zeros_like(W)))
    variant = decl.kernel_variant()
    steps(decl, 40)
    s_decl = state(decl)
    decl.destroy()            # one engine per variant at a time: the two worlds' scratch columns differ in size
    monkeypatch.setenv("RKFD_SPEC", str(variant[3]))
    plain = start(capi, w, q, qd, u)
    assert plain.kernel_variant() == variant
    steps(plain, 40)
    for a, b in zip(s_decl, state(plain)):
        assert np.array_equal(a, b)
    plain.destroy()


def test_rows_follow_the_slots(capi):
    """re-sort every step against never, and two shards against one: bit-identical per environment"""
    w, B, sample = setup("c3")
    B = 4096
    q, qd, u, W = sample(B, 5)
    runs = [start(capi, w, q, qd, u, resort=r, ext=([7, 3], W)) for r in (1, 0)] + [start(capi, w, q, qd, u, devices=[0, 0], ext=([7, 3], W))]
    if capi.device_count() >= 2:
        runs.append(start(capi, w, q, qd, u, devices=[0, 1], ext=([7, 3], W)))
    for fd in runs:
        steps(fd, 30)
    assert runs[0].resort_count > 0
    s0 = state(runs[0])
    for fd in runs[1:]:
        for a, b in zip(s0, state(fd)):
            assert np.array_equal(a, b)
    for fd in runs:
        fd.destroy()


def test_device_setter_equals_host_setter(capi):
    import torch
    w, B, sample = setup("c3")
    B = 2048
    q, qd, u, W = sample(B, 6)
    W2 = np.random.default_rng(9).uniform(-10, 10, W.shape)
    a, b = start(capi, w, q, qd, u, ext=([7, 3], W)), start(capi, w, q, qd, u, ext=([7, 3], W))
    steps(a, 20); steps(b, 20)                                  # re-sorted slots by now
    assert a.resort_count > 0
    a.batch_set_ext_wrench(W2)
    t = torch.from_numpy(W2).cuda()
    torch.cuda.synchronize()
    b.batch_set_ext_wrench_device(0, t.data_ptr())
    steps(a, 20); steps(b, 20)
    for x, y in zip(state(a), state(b)):
        assert np.array_equal(x, y)
    a.destroy(); b.destroy()


def test_pending_wrench_enters_the_first_evaluation(capi):
    w, B, sample = setup("c3")
    q, qd, u, W = sample(64, 7)
    fd, plain = start(capi, w, q, qd, u, ext=([7, 3], W)), start(capi, w, q, qd, u)
    gqdd, pqdd = fd.batch_get_state()[2], plain.batch_get_state()[2]
    _, _, oqdd, _ = oracle_run(w, q, qd, u, [7, 3], W, 0)
    assert np.abs(gqdd - oqdd).max() < 1e-9 * max(np.abs(oqdd).max(), 1.0)
    assert np.abs(gqdd - pqdd).max() > 1e-3
    fd.destroy(); plain.destroy()


@pytest.mark.parametrize("name", ["c3", "brick_wall"])
def test_reset_keeps_the_wrench(capi, name):
    """a reset environment equals a new simulator started from its state with its wrench; the others are untouched"""
    w, B, sample = setup(name)
    q, qd, u, W = sample(B, 8)
    links = LINKS[name]
    fd, twin = start(capi, w, q, qd, u, ext=(links, W)), start(capi, w, q, qd, u, ext=(links, W))
    steps(fd, 20); steps(twin, 20)
    envs = np.arange(3, B, 7)
    q2, qd2, u2, _ = sample(B, 9)
    fd.batch_reset_envs(envs, q2[envs], qd2[envs], u2[envs])
    fresh = start(capi, w, q2[envs], qd2[envs], u2[envs], ext=(links, W[envs]))
    steps(fd, 20); steps(twin, 20); steps(fresh, 20)
    others = np.setdiff1d(np.arange(B), envs)
    sf, st_, sn = state(fd), state(twin), state(fresh)
    for x, y, z in zip(sf, st_, sn):
        assert np.array_equal(x[envs], z)
        assert np.array_equal(x[others], y[others])
    for x in (fd, twin, fresh):
        x.destroy()


def test_hovering_body_stays_put(capi):
    w = free_body()
    B = 64
    q = np.tile([0.1, -0.2, 0.5, 0.3, -0.4, 0.2], (B, 1)); qd = np.zeros((B, 6))
    W = np.zeros((B, 1, 6)); W[:, 0, 2] = 1.7 * 9.80665
    fd = start(capi, w, q, qd, np.zeros((B, 1)), ext=([0], W))
    fd.update_n(1000)
    gq, gqd, gqdd = fd.batch_get_state()
    assert np.abs(gq - q).max() < 1e-12 and np.abs(gqd).max() < 1e-12 and np.abs(gqdd).max() < 1e-12
    fd.destroy()
