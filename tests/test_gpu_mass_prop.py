"""Per-environment mass properties (rkFDBatchSetMassPropLinks / rkFDBatchSetMassProp / rkFDBatchSetMassPropDevice) on the GPU:
every contact solver against the oracle run on per-environment worlds, the kernel choice, the model's own values against the
undeclared world, re-sorted slots and shards, the device setter, the t = 0 evaluation, resets and boxes of different masses
resting on a soft floor."""
import numpy as np
import pytest

import rokifd_b200  # noqa: F401
from rokifd_b200 import chains as ch
import ref_numpy as rn
from gpu_batch import capi, start, steps, state  # noqa: F401
from mass_prop_py import oracle_run_mp, own_rows, randomise
from workloads import world

pytestmark = pytest.mark.gpu

LINKS = {"c2": [7], "c3": [7, 3], "c4": [0, 3], "c4_volume": [0], "c5_mlcp": [7, 4], "c5_vert": [7], "arm_box_floor": [3, 2],
         "random_tree": [0, 5, 12], "brick_wall": [3]}
TOL = {"c5_vert": 1e-7, "c4_volume": 1e-6}
BATCH = {"c2": 1024, "c3": 1024, "c4": 256, "c4_volume": 512, "c5_mlcp": 1024, "c5_vert": 512, "arm_box_floor": 512,
         "random_tree": 256, "brick_wall": 256}


def setup(name):
    """(world, B, sampler(B, seed) -> (q, qd, u, MP)); MP: per-environment mass properties of LINKS[name]"""
    w, states = world(name)

    def sample(B, seed):
        q, qd, u = states(B, seed)
        return q, qd, u, randomise(w, LINKS[name], B, seed + 2000)
    return w, BATCH[name], sample


@pytest.mark.parametrize("name", list(LINKS))
def test_matches_oracle(capi, name):
    w, B, sample = setup(name)
    B += 37                   # a ragged batch: the last block is partly padding
    q, qd, u, MP = sample(B, 3)
    links = LINKS[name]
    fd = start(capi, w, q, qd, u, mp=(links, MP))
    n = 40
    steps(fd, n)
    gq, gqd, _ = fd.batch_get_state()
    assert (fd.batch_get_status() == 0).all()
    sel = np.r_[0:32, B - 16:B]
    oq, oqd, _ = oracle_run_mp(w, q[sel], qd[sel], u[sel], links, MP[sel], n)
    for a, b, what in ((gq[sel], oq, "q"), (gqd[sel], oqd, "q'")):
        err = np.abs(a - b).max() / max(np.abs(b).max(), 1.0)
        assert err < TOL.get(name, 1e-9), (name, what, err)
    ref = start(capi, w, q, qd, u)
    steps(ref, n)
    assert np.abs(ref.batch_get_state()[0] - gq).max() > 1e-6          # the mass properties moved the worlds
    fd.destroy(); ref.destroy()


def test_declared_world_runs_the_generic_kernel(capi):
    w, B, sample = setup("c3")
    q, qd, u, MP = sample(256, 1)
    plain, decl = start(capi, w, q, qd, u), start(capi, w, q, qd, u, mp=([7], MP[:, :1]))
    assert plain.kernel_variant()[3] == 5
    assert decl.kernel_variant()[3] in (0, 11)
    plain.destroy(); decl.destroy()


@pytest.mark.parametrize("explicit", [False, True])
@pytest.mark.parametrize("name", ["c3", "c4_volume"])
def test_own_values_are_bit_identical(capi, name, explicit, monkeypatch):
    """declared links holding the model's own values (the default rows, or set explicitly) step like the undeclared world forced
    onto the same kernel variant: pass 2 forms the constant table's values bit for bit"""
    w, B, sample = setup(name)
    q, qd, u, _ = sample(B, 4)
    links = LINKS[name]
    decl = start(capi, w, q, qd, u, mp=(links, np.repeat(own_rows(w, links)[None], B, axis=0) if explicit else None))
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
    w, _, sample = setup("c3")
    B = 4096
    q, qd, u, MP = sample(B, 5)
    runs = [start(capi, w, q, qd, u, resort=r, mp=([7, 3], MP)) for r in (1, 0)] + [start(capi, w, q, qd, u, devices=[0, 0], mp=([7, 3], MP))]
    if capi.device_count() >= 2:
        runs.append(start(capi, w, q, qd, u, devices=[0, 1], mp=([7, 3], MP)))
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
    w, _, sample = setup("c3")
    B = 2048
    q, qd, u, MP = sample(B, 6)
    MP2 = randomise(w, [7, 3], B, 99)
    a, b = start(capi, w, q, qd, u, mp=([7, 3], MP)), start(capi, w, q, qd, u, mp=([7, 3], MP))
    steps(a, 20); steps(b, 20)                                  # re-sorted slots by now
    assert a.resort_count > 0
    a.batch_set_mass_prop(MP2)
    t = torch.from_numpy(MP2).cuda()
    torch.cuda.synchronize()
    b.batch_set_mass_prop_device(0, t.data_ptr())
    steps(a, 20); steps(b, 20)
    for x, y in zip(state(a), state(b)):
        assert np.array_equal(x, y)
    a.destroy(); b.destroy()


def test_pending_values_enter_the_first_evaluation(capi):
    """values set before update_init enter the committing evaluation at t = 0; a refused call keeps them, and a declaration
    after update_init is refused"""
    w, _, sample = setup("c3")
    q, qd, u, MP = sample(64, 7)
    fd, _ = capi.create_world(w, B=64)
    fd.batch_set_mass_prop_links([7, 3]); fd.batch_set_mass_prop(MP)
    bad = MP.copy(); bad[5, 1, 0] = -1.0
    with pytest.raises(RuntimeError, match="environment 5, link 3"):
        fd.batch_set_mass_prop(bad)
    fd.batch_set_state(q, qd); fd.batch_set_motor_input(u); fd.update_init()
    with pytest.raises(RuntimeError, match="before rkFDUpdateInit"):
        fd.batch_set_mass_prop_links([7])
    plain = start(capi, w, q, qd, u)
    gqdd, pqdd = fd.batch_get_state()[2], plain.batch_get_state()[2]
    _, _, oqdd = oracle_run_mp(w, q, qd, u, [7, 3], MP, 0)
    assert np.abs(gqdd - oqdd).max() < 1e-9 * max(np.abs(oqdd).max(), 1.0)
    assert np.abs(gqdd - pqdd).max() > 1e-3
    fd.destroy(); plain.destroy()


@pytest.mark.parametrize("name", ["c3", "brick_wall"])
def test_reset_keeps_the_mass_properties(capi, name):
    """a reset environment equals a new simulator started from its state with its mass properties; the others are untouched"""
    w, B, sample = setup(name)
    q, qd, u, MP = sample(B, 8)
    links = LINKS[name]
    fd, twin = start(capi, w, q, qd, u, mp=(links, MP)), start(capi, w, q, qd, u, mp=(links, MP))
    steps(fd, 20); steps(twin, 20)
    envs = np.arange(3, B, 7)
    q2, qd2, u2, _ = sample(B, 9)
    fd.batch_reset_envs(envs, q2[envs], qd2[envs], u2[envs])
    fresh = start(capi, w, q2[envs], qd2[envs], u2[envs], mp=(links, MP[envs]))
    steps(fd, 20); steps(twin, 20); steps(fresh, 20)
    others = np.setdiff1d(np.arange(B), envs)
    sf, st_, sn = state(fd), state(twin), state(fresh)
    for x, y, z in zip(sf, st_, sn):
        assert np.array_equal(x[envs], z)
        assert np.array_equal(x[others], y[others])
    for x in (fd, twin, fresh):
        x.destroy()


def test_boxes_of_different_masses_settle_at_their_own_depth(capi):
    """a box on the soft floor settles at the penetration m g / (4 E) of its own mass (the oracle pin of a resting box, one mass
    per environment)"""
    E = 1000.0
    w = ch.World(chains=[ch.box(), ch.floor_soft()], contact_info=[ch.ContactInfo("soft", "body", "elastic", E=E, V=10.0)])
    B = 64
    m = np.linspace(0.25, 1.5, B)
    MP = np.repeat(own_rows(w, [0])[None], B, axis=0)
    MP[:, 0, 0] = m; MP[:, 0, 4:] *= (m / 0.5)[:, None]
    q = np.tile([0, 0, 0.05 + 1e-4, 0, 0, 0], (B, 1)); qd = np.zeros((B, 6))
    fd = start(capi, w, q, qd, np.zeros((B, 1)), mp=([0], MP))
    fd.update_n(4000)
    gq, gqd, _ = fd.batch_get_state()
    depth = 0.05 - gq[:, 2]
    assert np.abs(depth - m * rn.G / (4 * E)).max() < 1e-6
    assert np.abs(gqd).max() < 1e-6 and (fd.batch_get_status() == 0).all()
    fd.destroy()
