"""Helpers of the GPU batch tests (-m gpu): the C-ABI fixture (test modules import `capi` by name), a batch started from a
state, one call per step, and bit-for-bit comparison of environments."""
import numpy as np
import pytest

import rokifd_b200  # noqa: F401


@pytest.fixture(scope="module")
def capi():
    from rokifd_b200 import capi as c
    assert c.device_count() > 0, "no CUDA device: the product path has no CPU fallback"
    return c


def start(capi, w, q, qd, u, devices=None, resort=None, ext=None, mp=None):
    """a batch of world w after rkFDUpdateInit at (q, qd, u); ext / mp = (links, rows or None): links that take an external
    wrench / mass properties, and their rows (None: the engine's initial rows)"""
    fd, _ = capi.create_world(w, B=q.shape[0], devices=devices)
    if resort is not None:
        fd.batch_set_resort_interval(resort)
    if ext is not None:
        fd.batch_set_ext_wrench_links(ext[0])
        if ext[1] is not None:
            fd.batch_set_ext_wrench(ext[1])
    if mp is not None:
        fd.batch_set_mass_prop_links(mp[0])
        if mp[1] is not None:
            fd.batch_set_mass_prop(mp[1])
    fd.batch_set_state(q, qd); fd.batch_set_motor_input(u); fd.update_init()
    return fd


def steps(fd, k):
    for _ in range(k):         # one call per step: the engine re-sorts between calls
        fd.update()


def state(fd):
    return fd.batch_get_state() + (fd.batch_get_status(),) + tuple(fd.batch_get_contact())


def snapshot(fd):
    q, qd, qdd = fd.batch_get_state()
    a, t, r, f = fd.batch_get_contact()
    pt, pp = fd.batch_get_pivot()
    return dict(q=q, qd=qd, qdd=qdd, active=a, kinetic=t, ref=r, f=f, piv_type=pt, piv_prev=pp, status=fd.batch_get_status())


def assert_same(x, xi, y, yi, what):
    """environments xi of snapshot x are bit-identical to environments yi of snapshot y (anchors and forces on active slots)"""
    act = y["active"][yi] == 1
    for k in x:
        a, b = x[k][xi], y[k][yi]
        if k in ("ref", "f"):
            a, b = a * act[:, :, None], b * act[:, :, None]
        assert np.array_equal(a, b), "%s: %s differs in %d environments" % (what, k, int((a != b).reshape(len(a), -1).any(1).sum()))


def pick(B, frac, seed):
    """an unsorted subset of ~frac * B environments that contains 0 and B-1"""
    rng = np.random.default_rng(seed)
    envs = rng.choice(np.arange(1, B - 1), max(int(frac * B) - 2, 0), replace=False)
    envs = np.concatenate([envs, [0, B - 1]]).astype(np.int32)
    rng.shuffle(envs)
    return envs


def num_shards(capi, fd):
    n = 0
    while capi.lib().rkFDBatchDevicePtr(fd.h, n, 0, None, None):
        n += 1
    return n
