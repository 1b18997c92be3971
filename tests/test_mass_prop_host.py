"""Per-environment mass properties (rkFDBatchSetMassPropLinks / rkFDBatchSetMassProp) without a GPU: an analytic pin of the
parallel-axis term, a hovering body whose external wrench acts at its own centre of mass, the generic kernel core (host
harness) against the oracle run on per-environment worlds under every contact solver, the model's own values against no
declaration bit for bit, and the argument checks of the C-ABI."""
import ctypes as C

import numpy as np
import pytest

import rokifd_b200  # noqa: F401
from rokifd_b200 import capi
from rokifd_b200 import chains as ch
import ref_numpy as rn
from ext_wrench_py import set_ext_wrench, spec_mask
from hostsim_py import HostSim
from mass_prop_py import hostsim, set_mass_prop, oracle_run_mp, own_rows, randomise, row
from test_ext_wrench_host import free_body, workload


def spd(rng, scale):
    A = rng.normal(size=(3, 3))
    return (A @ A.T + 0.5 * np.eye(3)) * scale


# ---- physics pins --------------------------------------------------------------------------------------------------------
def pendulum():
    """a fixed base and one revolute link whose axis (link z) is horizontal: gravity lies in the plane of rotation"""
    base = ch.Link(name="base", jtype="fixed", mass=1.0, inertia=np.eye(3) * 0.01)
    arm = ch.Link(name="arm", jtype="revolute", parent=0, mass=2.0, com=np.array([0.2, 0.0, 0.0]), inertia=np.eye(3) * 0.02,
                  org_R=ch.rot_x(np.pi / 2))
    return ch.World(chains=[ch.ChainModel("pendulum", [base, arm])])


def test_pendulum_matches_parallel_axis_formula():
    """q'' at rest = m (c x g_l)_z / (Ic_zz + m (c_x^2 + c_y^2)) for each environment's mass, centre of mass and full Ic"""
    w = pendulum()
    B = 5
    rng = np.random.default_rng(11)
    q = rng.uniform(-3, 3, (B, 1)); qd = np.zeros((B, 1)); u = np.zeros((B, 2))
    MP = np.array([[row(rng.uniform(0.3, 5.0), rng.uniform(-0.3, 0.3, 3), spd(rng, 0.05))] for _ in range(B)])
    hs = hostsim(w, B, [1])
    hs.set_state(q, qd, u); set_mass_prop(hs, MP); hs.eval(ref=True)
    hqdd = hs.get_state()[2]
    _, _, oqdd = oracle_run_mp(w, q, qd, u, [1], MP, 0)
    Ro = ch.rot_x(np.pi / 2)
    for e in range(B):
        m, c, Ic = MP[e, 0, 0], MP[e, 0, 1:4], MP[e, 0, 4:]
        gl = (Ro @ ch.rot_z(q[e, 0])).T @ np.array([0.0, 0.0, -rn.G])
        ref = m * np.cross(c, gl)[2] / (Ic[5] + m * (c[0] ** 2 + c[1] ** 2))
        assert abs(hqdd[e, 0] - ref) < 1e-12 * max(1.0, abs(ref)), (e, hqdd[e, 0], ref)
        assert abs(oqdd[e, 0] - ref) < 1e-12 * max(1.0, abs(ref)), (e, oqdd[e, 0], ref)


def test_hovering_body_with_its_own_mass_stays_put():
    """each environment's body with its own mass and centre of mass, and f = (0, 0, m_e g) at that centre of mass: at rest it
    stays at rest (the wrench acts at the environment's centre of mass, not the model's)"""
    w = free_body()
    B = 4
    rng = np.random.default_rng(5)
    q = np.tile([0.1, -0.2, 0.5, 0.3, -0.4, 0.2], (B, 1)); qd = np.zeros((B, 6))
    MP = np.array([[row(rng.uniform(0.5, 4.0), rng.uniform(-0.1, 0.1, 3), spd(rng, 0.03))] for _ in range(B)])
    W = np.zeros((B, 1, 6)); W[:, 0, 2] = MP[:, 0, 0] * rn.G
    hs = hostsim(w, B, [0], ext_links=[0])
    hs.set_state(q, qd, np.zeros((B, 1))); set_mass_prop(hs, MP); set_ext_wrench(hs, W)
    hs.eval(ref=True); hs.step(200)
    hq, hqd, hqdd = hs.get_state()
    assert np.abs(hq - q).max() < 1e-12 and np.abs(hqd).max() < 1e-12 and np.abs(hqdd).max() < 1e-12


# ---- the generic kernel core against the oracle --------------------------------------------------------------------------
LINKS = {"c3": [7, 3], "arm_box_floor": [3, 2], "c5_mlcp": [7, 4], "c5_vert": [7, 4], "c4_volume": [0]}


def sample_mp(name, B, seed):
    w, _, sample, tol = workload(name)
    q, qd, u, _ = sample(B, seed)
    return w, q, qd, u, randomise(w, LINKS[name], B, seed + 100), tol


@pytest.mark.parametrize("integrator", ["RKG", "RK4"])
@pytest.mark.parametrize("name", list(LINKS))
def test_core_matches_oracle(name, integrator):
    B, n = 6, 30
    w, q, qd, u, MP, tol = sample_mp(name, B, 5)
    w.integrator = integrator
    links = LINKS[name]
    hs = hostsim(w, B, links)
    hs.set_state(q, qd, u); set_mass_prop(hs, MP); hs.eval(ref=True); hs.step(n)
    hq, hqd, _ = hs.get_state()
    oq, oqd, _ = oracle_run_mp(w, q, qd, u, links, MP, n)
    assert (hs.get_status() == 0).all()
    for a, b, what in ((hq, oq, "q"), (hqd, oqd, "q'")):
        err = np.abs(a - b).max() / max(np.abs(b).max(), 1.0)
        assert err < tol, (name, integrator, what, err)
    # the mass properties moved the worlds: without them the core ends elsewhere
    h0 = HostSim(w, B); h0.set_state(q, qd, u); h0.eval(ref=True); h0.step(n)
    assert np.abs(h0.get_state()[0] - hq).max() > 1e-6


@pytest.mark.parametrize("name", ["c3", "c5_mlcp", "c4_volume"])
def test_own_values_are_bit_identical(name):
    """declared links holding the model's own values (the default rows, or the same values set explicitly) step bit for bit
    like the undeclared world on the generic core"""
    B = 4
    w, q, qd, u, _, _ = sample_mp(name, B, 9)
    links = LINKS[name]
    runs = []
    for decl, explicit in ((None, False), (links, False), (links, True)):
        hs = hostsim(w, B, decl)
        hs.set_state(q, qd, u)
        if explicit:
            set_mass_prop(hs, np.repeat(own_rows(w, links)[None], B, axis=0))
        hs.eval(ref=True); hs.step(20)
        runs.append(hs.get_state() + hs.get_contact()[3:] + (hs.get_pivot()[0],))
    for r in runs[1:]:
        for a, b in zip(runs[0], r):
            assert np.array_equal(a, b)


def test_declared_world_takes_no_arm_specialisation():
    w = ch.world_c3(base_z=0.3)
    assert HostSim(w, 1).spec_mask != 0
    assert spec_mask(hostsim(w, 1, [7])) == 0


# ---- C-ABI argument checks (no device needed) --------------------------------------------------------------------------
def flattened_mp_links(fd):
    capi.lib().rkFDUpdateInit(fd.h)        # flattens the world; fails afterwards where no device exists
    return fd.describe_model().get("mp.links[0]")


def test_declaration_checks():
    fd, _ = capi.create_world(ch.world_c3(base_z=0.3), B=3)
    L = capi.lib()
    mp = np.zeros((3, 1, 10))
    assert L.rkFDBatchSetMassProp(fd.h, mp.ctypes.data) != 0 and "no link is declared" in fd.last_error()
    good = np.array([7, 2], np.int32)
    fd.batch_set_mass_prop_links(good)
    for bad in ([8], [-1], [2, 2], list(range(8)) * 5):
        with pytest.raises(RuntimeError, match="rkFDBatchSetMassPropLinks"):
            fd.batch_set_mass_prop_links(bad)
    assert L.rkFDBatchSetMassPropLinks(fd.h, 1, None) != 0
    assert L.rkFDBatchSetMassPropLinks(fd.h, -1, good.ctypes.data) != 0
    assert L.rkFDBatchSetMassPropLinks(fd.h, 33, good.ctypes.data) != 0
    assert L.rkFDBatchSetMassPropDevice(fd.h, 0, mp.ctypes.data) != 0 and "rkFDUpdateInit" in fd.last_error()
    assert flattened_mp_links(fd) == [7.0, 2.0]               # the refused lists changed nothing
    fd.destroy()
    fd, _ = capi.create_world(ch.world_c3(base_z=0.3), B=3)
    fd.batch_set_mass_prop_links([4]); fd.batch_set_mass_prop_links([])
    with pytest.raises(RuntimeError, match="no link is declared"):
        fd.batch_set_mass_prop(mp)
    assert flattened_mp_links(fd) is None                     # n = 0 cleared the declaration
    fd.destroy()


def test_value_checks():
    """the whole array is checked before anything is held: a refused call keeps the earlier pending values, and the message
    names the environment and the link"""
    w = ch.world_c3(base_z=0.3)
    fd, _ = capi.create_world(w, B=3)
    fd.batch_set_mass_prop_links([7, 3])
    good = np.repeat(own_rows(w, [7, 3])[None], 3, axis=0)
    good[:, :, 0] *= 1.5
    fd.batch_set_mass_prop(good)
    impl = fd.h
    for e, k, col, val, msg in ((2, 1, 0, 0.0, "not positive"), (1, 0, 0, -1.0, "not positive"), (0, 1, 5, np.nan, "non-finite"),
                                (1, 1, 2, np.inf, "non-finite"), (2, 0, 5, 10.0, "positive definite"), (0, 0, 4, -1e-3, "positive definite")):
        bad = good.copy(); bad[e, k, col] = val
        with pytest.raises(RuntimeError, match="environment %d, link %d: .*%s" % (e, [7, 3][k], msg)):
            fd.batch_set_mass_prop(bad)
    # an indefinite inertia whose diagonal is positive
    bad = good.copy(); bad[1, 0, 4:] = [1.0, 0.9, 0.9, 1.0, -0.9, 1.0]
    with pytest.raises(RuntimeError, match="environment 1, link 7: the inertia is not positive definite"):
        fd.batch_set_mass_prop(bad)
    assert impl == fd.h
    assert flattened_mp_links(fd) == [7.0, 3.0]
    fd.destroy()


def test_signatures_declared():
    L = capi.lib()
    assert L.rkFDBatchSetMassPropLinks.restype is C.c_int and len(L.rkFDBatchSetMassPropLinks.argtypes) == 3
    assert L.rkFDBatchSetMassProp.restype is C.c_int and len(L.rkFDBatchSetMassProp.argtypes) == 2
    assert L.rkFDBatchSetMassPropDevice.restype is C.c_int and len(L.rkFDBatchSetMassPropDevice.argtypes) == 3
