"""External wrenches on links (rkFDBatchSetExtWrenchLinks / rkFDBatchSetExtWrench) without a GPU: the oracle's convention
against the independent numpy formulation and against physics, the generic kernel core (host harness) against the oracle
under every contact solver, and the argument checks of the C-ABI."""
import ctypes as C

import numpy as np
import pytest

import rokifd_b200  # noqa: F401
from rokifd_b200 import capi
from rokifd_b200 import chains as ch
import ref_numpy as rn
from ext_wrench_py import OracleEnvWrench, oracle_run
from hostsim_py import HostSim
from oracle.oracle import OracleWorld
from workloads import brick_wall_world, free_body, workload

NDOF = rn.NDOF


def aa_to_mat(aa):
    return rn.aa_to_mat(np.asarray(aa, float))


def world_frames(links, q):
    """world rotation and origin of every link (ref_numpy's kinematics)"""
    ofs = np.cumsum([0] + [NDOF[l.jtype] for l in links])
    R, p = [None] * len(links), [None] * len(links)
    for i, l in enumerate(links):
        qi = q[ofs[i]:ofs[i + 1]]
        Rp, pp = (R[l.parent], p[l.parent]) if l.parent >= 0 else (np.eye(3), np.zeros(3))
        Ro = Rp @ np.asarray(l.org_R, float)
        RJ, pJ = np.eye(3), np.zeros(3)
        if l.jtype == "revolute":
            RJ = ch.rot_z(qi[0])
        elif l.jtype == "prismatic":
            pJ = np.array([0, 0, qi[0]])
        elif l.jtype == "spherical":
            RJ = aa_to_mat(qi)
        elif l.jtype == "float":
            pJ, RJ = qi[:3], aa_to_mat(qi[3:])
        elif l.jtype == "cylindrical":
            RJ, pJ = ch.rot_z(qi[1]), np.array([0, 0, qi[0]])
        elif l.jtype == "hooke":
            RJ = ch.rot_z(qi[0]) @ ch.rot_y(qi[1])
        R[i] = Ro @ RJ
        p[i] = pp + Rp @ np.asarray(l.org_p, float) + Ro @ pJ
    return R, p


# ---- the oracle's convention -------------------------------------------------------------------------------------------
@pytest.mark.parametrize("seed", [1, 2, 3, 4])
def test_oracle_matches_newton_euler(seed):
    """random trees with every joint type (floating and fixed roots) and random wrenches on every link: q'' of the oracle's ABA
    equals the dense Newton-Euler solution of ref_numpy with the same wrench moved to the link origin"""
    rng = np.random.default_rng(seed)
    jts = ("revolute", "prismatic", "spherical", "float", "cylindrical", "hooke")
    for root in ("float", "fixed"):
        w = ch.World(chains=[ch.random_chain(rng, 7, jtypes=jts, root=root, branching=True)])
        links = w.flat_links()
        e = OracleEnvWrench(OracleWorld(w))
        q, qd = rng.uniform(-1.5, 1.5, w.nq), rng.uniform(-2, 2, w.nq)
        W = rng.uniform(-5, 5, (w.nl, 6))
        e.set_state(q, qd)
        for i in range(w.nl):
            e.set_ext_wrench(i, W[i])
        qdd = e.eval(False)
        R, _ = world_frames(links, q)
        fext = [(W[i, :3], W[i, 3:] + np.cross(R[i] @ np.asarray(links[i].com, float), W[i, :3])) for i in range(w.nl)]
        ref, _, _ = rn.forward_dynamics(links, q, qd, np.zeros(w.nq), fext=fext)
        ref0, _, _ = rn.forward_dynamics(links, q, qd, np.zeros(w.nq))
        assert np.abs(ref - ref0).max() > 1e-2 * np.abs(ref0).max()          # the wrench matters
        assert np.allclose(qdd, ref, rtol=1e-9, atol=1e-9 * max(1.0, np.abs(ref).max())), (seed, root)


def test_hovering_body_stays_put():
    """f = (0, 0, m g) at the centre of mass cancels gravity: a free body at rest stays at rest, 1,000 steps"""
    w = free_body()
    q = np.array([[0.1, -0.2, 0.5, 0.3, -0.4, 0.2]]); qd = np.zeros((1, 6))
    W = np.array([[[0, 0, 1.7 * rn.G, 0, 0, 0]]])
    oq, oqd, oqdd, _ = oracle_run(w, q, qd, np.zeros((1, 1)), [0], W, 1000)
    assert np.abs(oq - q).max() < 1e-12 and np.abs(oqd).max() < 1e-12 and np.abs(oqdd).max() < 1e-12


def test_pure_torque_on_free_body():
    """a torque n alone: the centre of mass falls with g, and w' = I^-1 (n - w x I w) (world axes)"""
    w = free_body()
    l = w.flat_links()[0]
    rng = np.random.default_rng(3)
    q = np.concatenate([rng.uniform(-0.3, 0.3, 3), rng.uniform(-1, 1, 3)]); qd = rng.uniform(-2, 2, 6)
    n = np.array([0.3, -0.7, 0.5])
    e = OracleEnvWrench(OracleWorld(w))
    e.set_state(q, qd); e.set_ext_wrench(0, np.concatenate([np.zeros(3), n]))
    qdd = e.eval(False)
    R = aa_to_mat(q[3:]); om = qd[3:]; Iw = R @ l.inertia @ R.T; r = R @ l.com
    dom = np.linalg.solve(Iw, n - np.cross(om, Iw @ om))
    acom = qdd[:3] + np.cross(qdd[3:], r) + np.cross(om, np.cross(om, r))
    assert np.allclose(qdd[3:], dom, rtol=1e-12, atol=1e-12)
    assert np.allclose(acom, [0, 0, -rn.G], rtol=0, atol=1e-12)


def test_axis_torque_equals_motor_torque():
    """on the first revolute link of a fixed-base arm, a wrench whose moment about the joint axis is tau gives the q'' of a
    torque motor input tau (the reaction of the motor lands on the fixed base)"""
    rng = np.random.default_rng(7)
    c = ch.random_chain(rng, 5, jtypes=("revolute",))
    c.links[1].motor = ch.Motor(type="trq")
    w = ch.World(chains=[c])
    ow = OracleWorld(w)
    q, qd = rng.uniform(-1.5, 1.5, w.nq), rng.uniform(-1, 1, w.nq)
    tau = 1.3
    R, _ = world_frames(w.flat_links(), q)
    e1 = OracleEnvWrench(ow); e1.set_state(q, qd); u = np.zeros(w.nl); u[1] = tau; e1.set_motor_input(u)
    e2 = OracleEnvWrench(ow); e2.set_state(q, qd); e2.set_ext_wrench(1, np.concatenate([np.zeros(3), tau * R[1][:, 2]]))
    e0 = OracleEnvWrench(ow); e0.set_state(q, qd)
    a0, a1, a2 = e0.eval(False), e1.eval(False), e2.eval(False)
    assert np.abs(a1 - a0).max() > 1e-3
    assert np.allclose(a1, a2, rtol=0, atol=1e-12 * max(1.0, np.abs(a1).max())), np.abs(a1 - a2).max()


@pytest.mark.parametrize("push,breaks", [(30.0, True), (10.0, False)])
def test_push_breaks_a_joint(push, breaks):
    """brick wall whose outer joint gives way at 20 N: a sideways push on the outer brick above the threshold breaks it in the
    committing evaluation; below, it holds (so does everything under gravity alone).  Host harness and oracle agree."""
    w = brick_wall_world([200.0, 200.0, 20.0], [200.0, 200.0, 200.0])
    B = 2
    q = np.zeros((B, w.nq)); qd = np.zeros((B, w.nq)); u = np.zeros((B, w.nl))
    W = np.zeros((B, 1, 6)); W[0, 0, 1] = push
    oq, oqd, oqdd, opiv = oracle_run(w, q, qd, u, [3], W, 0)
    assert opiv[0, 12] == int(breaks) and opiv[1, 12] == 0 and (opiv[:, [0, 6]] == 0).all()
    hs = HostSim(w, B, ext_links=[3])
    hs.set_state(q, qd, u); hs.set_ext_wrench(W); hs.eval(ref=True)
    assert (hs.get_pivot()[0] == opiv).all()


# ---- the generic kernel core against the oracle --------------------------------------------------------------------------
@pytest.mark.parametrize("integrator", ["RKG", "RK4"])
@pytest.mark.parametrize("name", ["c3", "arm_box_floor", "c5_mlcp", "c5_vert", "c4_volume"])
def test_core_matches_oracle(name, integrator):
    w, links, sample, tol = workload(name)
    w.integrator = integrator
    B, n = 6, 30
    q, qd, u, W = sample(B, 5)
    hs = HostSim(w, B, ext_links=links)
    hs.set_state(q, qd, u); hs.set_ext_wrench(W); hs.eval(ref=True); hs.step(n)
    hq, hqd, _ = hs.get_state()
    oq, oqd, _, _ = oracle_run(w, q, qd, u, links, W, n)
    assert (hs.get_status() == 0).all()
    for a, b, what in ((hq, oq, "q"), (hqd, oqd, "q'")):
        err = np.abs(a - b).max() / max(np.abs(b).max(), 1.0)
        assert err < tol, (name, integrator, what, err)
    # the wrench moved the worlds: without it the core ends elsewhere
    h0 = HostSim(w, B); h0.set_state(q, qd, u); h0.eval(ref=True); h0.step(n)
    assert np.abs(h0.get_state()[0] - hq).max() > 1e-6


@pytest.mark.parametrize("name", ["c3", "c5_mlcp", "c4_volume"])
def test_zero_wrench_is_bit_identical(name):
    """a declared world with zero wrenches steps bit for bit like the undeclared world on the generic core"""
    w, links, sample, _ = workload(name)
    B = 4
    q, qd, u, _ = sample(B, 9)
    runs = []
    for decl in (None, links):
        hs = HostSim(w, B, ext_links=decl)
        hs.set_state(q, qd, u)
        if decl:
            hs.set_ext_wrench(np.zeros((B, len(links), 6)))
        hs.eval(ref=True); hs.step(20)
        runs.append(hs.get_state() + hs.get_contact()[3:])
    for a, b in zip(*runs):
        assert np.array_equal(a, b)


def test_declared_world_takes_no_arm_specialisation():
    w = ch.world_c3(base_z=0.3)
    assert HostSim(w, 1).spec_mask != 0
    assert HostSim(w, 1, ext_links=[7]).spec_mask == 0


# ---- C-ABI argument checks (no device needed) --------------------------------------------------------------------------
def flattened_ext_links(fd):
    capi.lib().rkFDUpdateInit(fd.h)        # flattens the world; fails afterwards where no device exists
    return fd.describe_model().get("ext.links[0]")


def test_declaration_checks():
    fd, _ = capi.create_world(ch.world_c3(base_z=0.3), B=3)
    L = capi.lib()
    w = np.zeros((3, 1, 6))
    assert L.rkFDBatchSetExtWrench(fd.h, w.ctypes.data) != 0 and "no link is declared" in fd.last_error()
    good = np.array([7, 2], np.int32)
    fd.batch_set_ext_wrench_links(good)
    for bad in ([8], [-1], [2, 2], list(range(8)) * 5):
        with pytest.raises(RuntimeError, match="rkFDBatchSetExtWrenchLinks"):
            fd.batch_set_ext_wrench_links(bad)
    assert L.rkFDBatchSetExtWrenchLinks(fd.h, 1, None) != 0
    assert L.rkFDBatchSetExtWrenchLinks(fd.h, -1, good.ctypes.data) != 0
    assert L.rkFDBatchSetExtWrenchDevice(fd.h, 0, w.ctypes.data) != 0 and "rkFDUpdateInit" in fd.last_error()
    fd.batch_set_ext_wrench(np.zeros((3, 2, 6)))            # held as pending
    assert flattened_ext_links(fd) == [7.0, 2.0]             # the refused lists changed nothing
    fd.destroy()
    fd, _ = capi.create_world(ch.world_c3(base_z=0.3), B=3)
    fd.batch_set_ext_wrench_links([4]); fd.batch_set_ext_wrench_links([])
    with pytest.raises(RuntimeError, match="no link is declared"):
        fd.batch_set_ext_wrench(w)
    assert flattened_ext_links(fd) is None                   # n = 0 cleared the declaration
    fd.destroy()


def test_signatures_declared():
    L = capi.lib()
    assert L.rkFDBatchSetExtWrenchLinks.restype is C.c_int and len(L.rkFDBatchSetExtWrenchLinks.argtypes) == 3
    assert L.rkFDBatchSetExtWrench.restype is C.c_int and len(L.rkFDBatchSetExtWrench.argtypes) == 2
    assert L.rkFDBatchSetExtWrenchDevice.restype is C.c_int and len(L.rkFDBatchSetExtWrenchDevice.argtypes) == 3
