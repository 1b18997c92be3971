"""Oracle self-tests (SURVEY.md section 4, pyramid level 1): the CPU restatement is checked against an
independent numpy formulation and against physics invariants.  The reference ships no golden
vectors (parity unpinned), so these are what pins the oracle."""
import numpy as np
import pytest

import rokifd_b200  # noqa: F401
from rokifd_b200 import chains as ch
import ref_numpy as rn
from workloads import slide_worlds


def _world(chain, **kw):
    return ch.World(chains=[chain], **kw)


@pytest.mark.parametrize("kind", ["serial_revolute", "mixed_1dof", "branching", "float_root",
                                  "spherical", "float_branching_mixed", "cylindrical_hooke"])
def test_aba_matches_dense_newton_euler(oracle, kind):
    rng = np.random.default_rng(hash(kind) % 2**32)
    for trial in range(5):
        if kind == "serial_revolute":
            c = ch.random_chain(rng, 7)
        elif kind == "mixed_1dof":
            c = ch.random_chain(rng, 6, jtypes=("revolute", "prismatic", "fixed"))
        elif kind == "branching":
            c = ch.random_chain(rng, 9, jtypes=("revolute", "prismatic"), branching=True)
        elif kind == "float_root":
            c = ch.random_chain(rng, 5, root="float")
        elif kind == "spherical":
            c = ch.random_chain(rng, 5, jtypes=("spherical", "revolute"))
        elif kind == "cylindrical_hooke":
            c = ch.random_chain(rng, 7, jtypes=("cylindrical", "hooke", "revolute"), root=("fixed", "float")[trial % 2], branching=trial >= 3)
        else:
            c = ch.random_chain(rng, 10, jtypes=("revolute", "prismatic", "spherical", "fixed"), root="float",
                                branching=True)
        w = _world(c)
        ow = oracle.OracleWorld(w)
        e = ow.env()
        q = rng.uniform(-1.5, 1.5, w.nq)
        qd = rng.uniform(-2, 2, w.nq)
        e.set_state(q, qd)
        qdd = e.eval(False)
        ref, M, h = rn.forward_dynamics(w.flat_links(), q, qd, np.zeros(w.nq))
        assert np.allclose(qdd, ref, rtol=1e-9, atol=1e-9 * max(1.0, np.abs(ref).max())), (kind, trial)


def test_motor_and_joint_friction_enter_aba(oracle):
    rng = np.random.default_rng(5)
    w = ch.world_c2()
    ow = oracle.OracleWorld(w)
    links = w.flat_links()
    for trial in range(5):
        e = ow.env()
        q = rng.uniform(-1.5, 1.5, w.nq); qd = rng.uniform(-1, 1, w.nq); u = rng.uniform(-6, 6, w.nl)
        e.set_state(q, qd); e.set_motor_input(u)
        qdd = e.eval(False)
        td, jm = rn.motor_terms(links, qd, u)
        # joint friction of rkfd_util.c:330-364 with pivot {SF, prev_trq=0}
        tf = np.zeros(w.nq)
        for j in range(w.nq):
            l = links[j + 1]
            t = -jm[j] * qd[j] / w.dt - td[j]
            fmax = abs(l.sfriction)
            tf[j] = np.clip(t, -fmax, fmax)
        ref, _, _ = rn.forward_dynamics(links, q, qd, td + tf, jm=jm)
        assert np.allclose(qdd, ref, rtol=1e-9, atol=1e-9)


def test_free_fall(oracle):
    w = _world(ch.box())
    e = oracle.OracleWorld(w).env()
    q = np.array([0.1, -0.2, 1.0, 0.3, -0.2, 0.1]); qd = np.array([0.3, 0.1, 0.0, 1.0, 2.0, -1.0])
    e.set_state(q, qd)
    qdd = e.eval(False)
    assert np.allclose(qdd[:3], [0, 0, -rn.G], atol=1e-12)
    # isotropic inertia: no gyroscopic torque
    assert np.allclose(qdd[3:], 0, atol=1e-12)
    e.update_init()
    for _ in range(100):
        e.update()
    q1, qd1, _ = e.get_state()
    t = 0.1
    assert np.allclose(q1[:3], q[:3] + qd[:3] * t + 0.5 * np.array([0, 0, -rn.G]) * t * t, atol=1e-12)
    assert np.allclose(qd1[3:], qd[3:], atol=1e-12)
    # constant org-frame angular velocity: R(t) = exp(w t) R(0)
    R1 = rn.aa_to_mat(q1[3:])
    assert np.allclose(R1, rn.aa_to_mat(qd[3:] * t) @ rn.aa_to_mat(q[3:]), atol=1e-9)


def _arm_nomotor():
    return ch.World(chains=[ch.arm7(motors=False)])


def test_energy_conservation_and_rkg_order(oracle):
    q0 = np.array([0.3, -0.5, 0.8, 1.0, -0.7, 0.4, 0.2]); qd0 = np.array([0.5, -0.3, 0.2, 0.1, 0.4, -0.6, 0.3])
    drift = []
    for dt, n in ((2e-3, 100), (1e-3, 200)):
        w = _arm_nomotor(); w.dt = dt
        e = oracle.OracleWorld(w).env()
        e.set_state(q0, qd0)
        E0 = e.energy()
        e.update_init()
        for _ in range(n):
            e.update()
        drift.append(abs(e.energy() - E0))
    assert drift[1] < 1e-7
    # 4th-order integrator: halving dt cuts the drift by ~2^4 (allow slack)
    assert drift[0] / max(drift[1], 1e-300) > 8.0


def test_pendulum_period(oracle):
    L, m = 0.5, 1.0
    base = ch.Link(name="b", jtype="fixed", org_p=np.array([0, 0, 1.0]))
    # joint axis (local z) horizontal: rotate link frame so z -> world y
    pend = ch.Link(name="p", jtype="revolute", parent=0, mass=m, com=np.array([L, 0, 0]), inertia=np.zeros((3, 3)),
                   org_R=ch.rot_x(-np.pi / 2))
    w = ch.World(chains=[ch.ChainModel("pend", [base, pend])], dt=1e-3)
    e = oracle.OracleWorld(w).env()
    # link x axis points along world x at q=0; gravity pulls towards -z == local +y after rot_x(-90)... find equilibrium numerically
    th0 = 0.05
    # equilibrium: COM straight below the pivot
    qeq = None
    for cand in np.linspace(-np.pi, np.pi, 721):
        e.set_state([cand], [0.0])
        if abs(e.eval(False)[0]) < 1e-9:
            R, p = e.link_frames()
            if (R[1] @ pend.com)[2] < 0:
                qeq = cand
    assert qeq is not None
    e.set_state([qeq + th0], [0.0])
    e.update_init()
    t_cross, prev = [], th0
    for k in range(3000):
        e.update()
        cur = e.get_state()[0][0] - qeq
        if prev > 0 >= cur or prev < 0 <= cur:
            t_cross.append(e.t - w.dt * abs(cur) / (abs(cur) + abs(prev)))
        prev = cur
    T = 2 * (t_cross[1] - t_cross[0])
    T_exact = 2 * np.pi * np.sqrt(L / rn.G) * (1 + th0 ** 2 / 16)
    assert abs(T - T_exact) / T_exact < 1e-4


def test_box_rests_on_penalty_ground(oracle):
    """Flat box on the soft floor: steady penetration depth = m g / (4 E) on the 4 bottom vertices."""
    w = ch.World(chains=[ch.box(), ch.floor_soft()],
                 contact_info=[ch.ContactInfo("soft", "body", "elastic", E=1000.0, V=10.0)])
    e = oracle.OracleWorld(w).env()
    e.set_state([0, 0, 0.05 + 1e-4, 0, 0, 0], np.zeros(6))
    e.update_init()
    for _ in range(4000):
        e.update()
    q, qd, qdd = e.get_state()
    depth = 0.05 - q[2]
    assert abs(depth - 0.5 * rn.G / (4 * 1000.0)) < 1e-6
    assert np.abs(qd).max() < 1e-6 and np.abs(qdd).max() < 1e-5
    a, t, r, f = e.get_contact()
    assert a.sum() == 4
    assert abs(f[a == 1][:, 2].sum() - 0.5 * rn.G) < 1e-5


def test_penalty_friction_stick_and_slip(oracle):
    """Box pushed sideways on the soft floor: sticks (SF) for slow speed, slips (KF) when fast, and friction
    decelerates at about mu_k g while slipping."""
    w = ch.World(chains=[ch.box(), ch.floor_soft()],
                 contact_info=[ch.ContactInfo("soft", "body", "elastic", E=1000.0, V=10.0, SF=0.5, KF=0.3)])
    ow = oracle.OracleWorld(w)
    e = ow.env()
    z0 = 0.05 - 0.5 * rn.G / 4000.0
    e.set_state([0, 0, z0, 0, 0, 0], [2.0, 0, 0, 0, 0, 0])
    e.update_init()
    for _ in range(50):
        e.update()
    a, t, r, f = e.get_contact()
    assert (t[a == 1] == 1).all()          # kinetic
    _, qd, qdd = e.get_state()
    assert qd[0] < 2.0
    assert abs(qdd[0] + 0.3 * rn.G) < 0.3 * rn.G * 0.2
    for _ in range(3000):
        e.update()
    a, t, r, f = e.get_contact()
    _, qd, _ = e.get_state()
    assert abs(qd[0]) < 1e-3
    assert (t[a == 1] == 0).all()          # back to static friction


def test_le_solve_mp_matches_pinv(oracle):
    rng = np.random.default_rng(3)
    for n, rank in ((5, 5), (8, 5), (12, 7)):
        B = rng.normal(size=(n, rank))
        A = B @ np.diag(rng.uniform(0.5, 2, rank) * rng.choice([-1, 1], rank)) @ B.T
        b = rng.normal(size=n)
        x = oracle.le_solve_mp_sym(A, b)
        assert np.allclose(x, np.linalg.pinv(A, rcond=1e-10) @ b, atol=1e-9)


def test_qp_asm_matches_scipy(oracle):
    from scipy.optimize import minimize
    rng = np.random.default_rng(11)
    for trial in range(10):
        n, m = 6, 8
        B = rng.normal(size=(n, n)); Q = B @ B.T + np.eye(n)
        c = rng.normal(size=n) * 3
        A = rng.normal(size=(m, n)); x0 = rng.normal(size=n)
        b = A @ x0 - rng.uniform(0.1, 1.0, m)       # x0 strictly feasible
        x, idx, it = oracle.qp_solve_asm(Q, c, A, b, init=x0)
        res = minimize(lambda z: 0.5 * z @ Q @ z + c @ z, x0, jac=lambda z: Q @ z + c, method="SLSQP",
                       constraints=[{"type": "ineq", "fun": lambda z: A @ z - b, "jac": lambda z: A}],
                       options={"ftol": 1e-14, "maxiter": 500})
        assert np.allclose(x, res.x, atol=1e-6), trial
        assert (A @ x - b > -1e-9).all()


def _golden_vert_qps():
    import os
    return np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "vert_qp_c5.npz"))


def test_le_solve_mp_on_ill_conditioned_kkt_matches_50_digit_solution(oracle):
    """[EXT A-14] zLESolveMP = THE minimum-norm solution: on a KKT matrix of BASELINE config C5 (relaxation 1e-4: condition
    ~1e7, redundant active rows: singular) the oracle's solve agrees with the 50-digit pseudo-inverse to a few ulp of the
    primal part, which is what the absolute 1e-12 decisions of rkfd_opt_qp.c:108-110 need."""
    import mpmath as mp
    import ref_qp_mp
    g = _golden_vert_qps()
    e = 2862
    Q, c, nf = g["Q%d" % e], g["c%d" % e], g["nf%d" % e]
    n = len(c)
    for act in ([0, 1, 2, 3, 4, 5, 6, 7, 12], [3, 4, 5, 12], [3, 4, 12]):     # all 8 rows of a vertex (rank 3), 3 of them, 2
        mp.mp.dps = 50
        K = ref_qp_mp.kkt(Q.tolist(), nf.tolist(), act)
        xm = ref_qp_mp.pinv_solve_sym(K, mp.matrix(list(c) + [0] * len(act)))
        Kd = np.array([[float(K[i, j]) for j in range(K.cols)] for i in range(K.rows)])
        xo = oracle.le_solve_mp_sym(Kd, np.concatenate([c, np.zeros(len(act))]))
        xm = np.array([float(v) for v in xm])
        assert np.abs(xo[:n] - xm[:n]).max() <= 4e-16 * np.abs(xm[:n]).max() + 1e-15, (act, np.abs(xo[:n] - xm[:n]).max())
        assert np.abs(xo[n:] - xm[n:]).max() <= 1e-9 * max(1.0, np.abs(xm[n:]).max())


def test_qp_asm_follows_the_exact_arithmetic_path_on_c5_golden_qps(oracle):
    """Golden vectors (tests/golden/vert_qp_c5.npz, made by tests/golden/make_vert_qp_golden.py): rkFDQPSolveASM evaluated in
    50-digit arithmetic on Vert QPs of BASELINE config C5.  In round 1 the oracle left the loop through the anti-cycling
    exit (rkfd_opt_qp.c:152-171) short of the minimiser on every one of them (objective up to 20 % above the minimum),
    because x* of two consecutive iterations differed by the rounding noise of its pseudo-inverse."""
    g = _golden_vert_qps()
    for e in g["envs"]:
        Q, c, nf, xg, ig = g["Q%d" % e], g["c%d" % e], g["nf%d" % e], g["x%d" % e], g["idx%d" % e]
        init = np.zeros(len(c)); init[0::3] = 1.0
        x, idx, it = oracle.qp_solve_asm(Q, c, nf, np.zeros(nf.shape[0]), init)
        assert np.abs(x - xg).max() <= 1e-11 * np.abs(xg).max(), (e, np.abs(x - xg).max())
        assert (idx == ig).all(), e
        assert abs(it - int(g["info%d" % e][0])) <= 1 and int(g["info%d" % e][1]) == 0
        # the answer is the minimiser: KKT residual with non-negative multipliers on the active rows
        from scipy.optimize import nnls
        grad = Q @ x + c
        _, rn = nnls(nf[idx == 1].T, grad)
        assert rn <= 1e-9 * np.abs(grad).max() and (nf @ x).min() > -1e-11


@pytest.mark.parametrize("solver", ["MLCP", "Vert"])
def test_box_rests_on_rigid_ground(oracle, solver):
    w = ch.World(chains=[ch.box(), ch.floor()], contact_info=ch.contact_info_table(), solver=solver)
    e = oracle.OracleWorld(w).env()
    e.set_state([0, 0, 0.05 - 1e-4, 0, 0, 0], np.zeros(6))
    e.update_init()
    for _ in range(500):
        e.update()
    q, qd, qdd = e.get_state()
    assert abs(q[2] - 0.05) < 2e-3
    if solver == "Vert":
        assert np.abs(qd).max() < 2e-2
    else:
        # MLCP: the reference's friction sweep reads rows offset+0/+1 (rkfd_mlcp.c:219-225), which drives
        # a spurious tangential force; only the normal direction settles.  Mirrored, not fixed.
        assert abs(qd[2]) < 2e-2
    a, t, r, f = e.get_contact()
    assert a.sum() == 4
    A, b, fs = e.rigid_system()
    assert A.shape == (12, 12)
    assert np.allclose(A, A.T, atol=1e-8 * np.abs(A).max() + 1e-12) or solver == "MLCP"
    assert abs(f[a == 1][:, 2].sum() - 0.5 * rn.G) < 0.5 * rn.G * 0.2


def test_delassus_matrix_is_J_Minv_JT(oracle):
    """The probe-built A (rkfd_vert.c:153-185) equals J M^-1 J^T from the dense model."""
    w = ch.world_c5(base_z=0.0, solver="Vert")
    ow = oracle.OracleWorld(w)
    rng = np.random.default_rng(7)
    links = w.flat_links()
    for trial in range(20):
        e = ow.env()
        q = rng.uniform(-1.5, 1.5, 7); qd = rng.uniform(-1, 1, 7)
        e.set_state(q, qd)
        e.eval(False)
        a, t, r, f = e.get_contact()
        if a.sum() == 0:
            continue
        A, b, fs = e.rigid_system()
        R, p = e.link_frames()
        verts = links[7].shapes[0]
        _, M, _ = rn.forward_dynamics(links, q, qd, np.zeros(7))
        jm = rn.motor_terms(links, qd, np.zeros(8))[1]
        M = M + np.diag(jm)
        # numeric Jacobian of world vertex positions
        J = []
        for k in np.nonzero(a)[0]:
            Jk = np.zeros((3, 7))
            for j in range(7):
                dq = np.zeros(7); dq[j] = 1e-6
                e2 = ow.env(); e2.set_state(q + dq, qd); e2.eval(False); Rp, pp = e2.link_frames()
                e3 = ow.env(); e3.set_state(q - dq, qd); e3.eval(False); Rm, pm = e3.link_frames()
                Jk[:, j] = ((pp[7] + Rp[7] @ verts[k]) - (pm[7] + Rm[7] @ verts[k])) / 2e-6
            J.append(Jk)
        J = np.vstack(J)          # axes are world x,y,z reordered (n=z, t1=x, t2=y)
        P = np.zeros((3, 3)); P[0, 2] = 1; P[1, 0] = 1; P[2, 1] = 1
        Jc = np.vstack([P @ J[3 * i:3 * i + 3] for i in range(len(J) // 3)])
        Aref = Jc @ np.linalg.solve(M, Jc.T)
        assert np.allclose(A, Aref, rtol=1e-5, atol=1e-6 * np.abs(Aref).max())
        return
    pytest.skip("no contact sampled")


def test_integrator_orders():
    """The four explicit schemes of zODE2AssignRegular converge with their orders on a frictionless double pendulum
    (Euler 1, Heun 2, RK4 and RKG 4): halving dt divides the end-state error by 2 / 4 / 16."""
    import copy
    from oracle import oracle as orc
    w0 = ch.World(chains=[ch.arm_2dof(motors=False)])
    for l in w0.chains[0].links:
        l.viscosity = l.coulomb = l.sfriction = 0.0
    q0, qd0 = np.array([0.4, -0.7]), np.array([0.3, 0.5])

    def end_state(integ, dt, T=0.08):
        w = copy.deepcopy(w0); w.integrator = integ; w.dt = dt
        e = orc.OracleWorld(w).env()
        e.set_state(q0, qd0); e.update_init()
        for _ in range(int(round(T / dt))):
            e.update()
        return np.concatenate(e.get_state()[:2])

    exact = end_state("RK4", 0.08 / 512)
    for integ, order in (("Euler", 1), ("Heun", 2), ("RK4", 4), ("RKG", 4)):
        e1 = np.abs(end_state(integ, 0.08 / 8) - exact).max()
        e2 = np.abs(end_state(integ, 0.08 / 16) - exact).max()
        assert 0.8 * 2 ** order < e1 / e2 < 1.25 * 2 ** order, (integ, e1, e2)


# ---- Volume solver (rkfd_volume.c): pins of the oracle's restatement
def test_lp_matches_scipy(oracle):
    """[EXT A-16] two-phase simplex: optimum value and feasibility verdict against scipy's HiGHS."""
    from scipy.optimize import linprog
    rng = np.random.default_rng(11)
    nfeas = ninf = 0
    for trial in range(60):
        m, n = int(rng.integers(1, 7)), int(rng.integers(3, 30))
        A = rng.normal(size=(m, n))
        if trial % 3:
            b = A @ rng.uniform(0, 1, n)            # feasible by construction
        elif trial % 2:
            b = rng.normal(size=m)
        else:
            A = np.abs(A); b = -np.abs(rng.normal(size=m)) - 0.1     # infeasible: A x >= 0 > b
        c = rng.uniform(0.1, 1.0, n)                # bounded below on x >= 0
        ok, x = oracle.lp_solve(A, b, c)
        ref = linprog(c, A_eq=A, b_eq=b, bounds=[(0, None)] * n, method="highs")
        assert ok == (ref.status == 0), trial
        okf, _ = oracle.lp_solve(A, b)
        assert okf == ok
        if ok:
            nfeas += 1
            assert (x >= -1e-9).all() and np.allclose(A @ x, b, atol=1e-8)
            assert abs(c @ x - ref.fun) < 1e-8 * max(1.0, abs(ref.fun))
        else:
            ninf += 1
    assert nfeas > 10 and ninf > 3


def test_volume_box_rests_in_equilibrium(oracle):
    """A tilted box dropped on the rigid floor with the Volume solver ends flat and at rest; the contact wrench is
    then the weight, applied under the centre of mass, with static friction."""
    w = ch.World(chains=[ch.box(), ch.floor()], solver="Volume")
    e = oracle.OracleWorld(w).env()
    q = np.zeros(6); q[2] = 0.049; q[3] = 0.05; q[4] = 0.02
    qd = np.zeros(6); qd[0] = 0.3
    e.set_state(q, qd); e.set_motor_input(np.zeros(w.nl)); e.update_init()
    for _ in range(1500):
        e.update()
    qq, qqd, qdd = e.get_state()
    npl, ty, wr, ce = e.volume()
    assert np.abs(qqd).max() < 1e-8 and np.abs(qdd).max() < 1e-6
    assert abs(qq[2] - 0.05) < 1e-3                       # flat on the floor (0.1 m cube)
    assert npl[0] == 4 and ty[0] == 0                     # square contact polygon, static friction
    assert np.allclose(wr[0][:3], [0, 0, 0.5 * 9.80665], atol=1e-6)
    # torque about the volume centre balances the offset of the centre of mass: tau = (com - centre) x f
    tau = np.cross(qq[:3] - ce[0], wr[0][:3])
    assert np.allclose(wr[0][3:], -tau, atol=1e-6)


def test_volume_sliding_box_kinetic_friction_ratio(oracle):
    """A box sliding on the rigid floor (it chatters: the friction torque tips it): whenever the pair pushes, it is
    kinetic and the tangential force is KF * (1 - exp(-w v)) * fn against the motion (rkfd_volume.c:715-843,
    rkfd_util.c:193-196: the per-corner friction directions coincide for a translating body)."""
    w = ch.World(chains=[ch.box(), ch.floor()], solver="Volume")
    e = oracle.OracleWorld(w).env()
    q = np.zeros(6); q[2] = 0.0499
    qd = np.zeros(6); qd[0] = 1.0
    e.set_state(q, qd); e.set_motor_input(np.zeros(w.nl)); e.update_init()
    npush = 0
    for _ in range(120):
        e.update()
        qq, qqd, qdd = e.get_state()
        npl, ty, wr, ce = e.volume()
        if npl[0] > 0 and wr[0][2] > 0.1:
            npush += 1
            assert ty[0] == 1
            assert abs(wr[0][0] / wr[0][2] + 0.3 * (1 - np.exp(-100.0 * qqd[0]))) < 5e-3
            assert abs(wr[0][1]) < 1e-6 * wr[0][2]
    assert npush > 20 and 0.5 < qqd[0] < 0.8          # about 0.3 g of deceleration over 0.12 s


def test_volume_surface_integrals_against_the_divergence_theorem(oracle):
    """Independent pins of the contact-volume construction and of the signed surface integrals of rkfd_volume.c:397-491
    for random box poses: with V the volume of (box intersected with the floor half-space) from scipy's convex hull, K the
    compensation and n the contact normal, the centre must be the hull's centroid, Q6 symmetric positive semi-definite with
    linear block (sum of projected face areas) * I, and the depth term c6 = (-K W n, torque) with W the integral of |height|
    over the UNSIGNED projected faces: W = V exactly for a box lying flat (every vertical line crosses the surface once above
    and once below the centre plane: the signed integral of the height over a closed surface is its volume, and its first
    moment about the barycentre vanishes, so the torque part is zero), W >= V for tilted boxes."""
    from scipy.spatial import ConvexHull
    w = ch.World(chains=[ch.box(), ch.floor()], solver="Volume")
    ow = oracle.OracleWorld(w)
    rng = np.random.default_rng(4)
    bv = ch.box_verts(0.1, 0.1, 0.1)
    edges = [(a, b) for a in range(8) for b in range(a + 1, 8) if bin(a ^ b).count("1") == 1]
    nchecked = 0
    for trial in range(40):
        flat = trial % 2 == 0
        q = np.zeros(6); q[:2] = rng.uniform(-0.5, 0.5, 2); q[2] = rng.uniform(0.0, 0.07); q[3:] = rng.uniform(-0.6, 0.6, 3)
        if flat:
            q[2] = rng.uniform(0.0, 0.049); q[3:5] = 0.0
        e = ow.env(); e.set_state(q, np.zeros(6)); e.set_motor_input(np.zeros(w.nl)); e.eval(True)
        npl, ty, wr, ce = e.volume()
        if npl[0] < 3:
            continue
        R, p = e.link_frames()
        vw = bv @ R[0].T + p[0]
        pts = [v for v in vw if v[2] <= 0]
        for a, b in edges:
            if (vw[a][2] < 0) != (vw[b][2] < 0):
                t = vw[a][2] / (vw[a][2] - vw[b][2]); pts.append(vw[a] + t * (vw[b] - vw[a]))
        hull = ConvexHull(np.array(pts))
        if hull.volume < 1e-9:
            continue
        # centroid of the hull from its triangles (signed tetrahedra about an interior point)
        c0 = np.mean(np.array(pts), 0); vol = 0.0; cen = np.zeros(3)
        for tri in hull.simplices:
            a, b, c = (hull.points[i] - c0 for i in tri)
            v6 = abs(np.dot(a, np.cross(b, c))) / 6.0
            vol += v6; cen += v6 * (a + b + c) / 4.0
        cen = c0 + cen / vol
        Q6, c6, nrm = e.volume_constraint()
        K = 1000.0
        assert abs(vol - hull.volume) < 1e-12
        assert np.allclose(ce[0], cen, atol=1e-9)
        assert np.allclose(nrm[0], [0, 0, 1])
        if flat:
            assert np.allclose(c6[0][:3], -K * hull.volume * nrm[0], rtol=1e-9, atol=1e-12)
            assert np.allclose(c6[0][3:], 0.0, atol=1e-9 * K * hull.volume)
            # flat 0.1 m cube: cap and bottom face project to the 0.1 x 0.1 square (the side faces to nothing), centred on the
            # barycentre: Q6 = 2 * [[A I, 0], [0, -int [p x]^2 dA]] with int x^2 dA = int y^2 dA = 0.1^4 / 12
            m2 = 0.1 ** 4 / 12
            assert np.allclose(Q6[0][:3, :3], 0.02 * np.eye(3), atol=1e-12)
            assert np.allclose(Q6[0][:3, 3:], 0.0, atol=1e-12) and np.allclose(Q6[0][3:, :3], 0.0, atol=1e-12)
            assert np.allclose(Q6[0][3:, 3:], 2 * np.diag([m2, m2, 2 * m2]), atol=1e-12)
        else:
            assert np.allclose(c6[0][:2], 0.0, atol=1e-15) and -c6[0][2] >= K * hull.volume * (1 - 1e-9)
        assert np.allclose(Q6[0], Q6[0].T, atol=1e-15)
        assert np.allclose(Q6[0][:3, :3], Q6[0][0, 0] * np.eye(3), atol=1e-15) and Q6[0][0, 0] > 0
        assert np.all(np.linalg.eigvalsh(Q6[0]) > -1e-12)
        nchecked += 1
    assert nchecked >= 15


def test_volume_wrench_respects_unilaterality_and_the_friction_cone(oracle):
    """Random box states on the rigid floor (Volume solver): the pair pushes (fn >= 0); a static pair keeps its tangential force
    inside the Coulomb cone SF * fn; a kinetic one has at most KF * fn (rkfd_volume.c:552-568, 869-916)."""
    w = ch.World(chains=[ch.box(), ch.floor()], solver="Volume")
    ow = oracle.OracleWorld(w)
    rng = np.random.default_rng(8)
    nstat = nkin = 0
    for trial in range(200):
        q = np.zeros(6); q[2] = rng.uniform(0.0, 0.06); q[3:] = rng.uniform(-0.4, 0.4, 3)
        qd = rng.uniform(-1, 1, 6) * (0.0 if trial % 3 == 0 else 1.0)
        e = ow.env(); e.set_state(q, qd); e.set_motor_input(np.zeros(w.nl)); e.eval(True)
        npl, ty, wr, ce = e.volume()
        if npl[0] <= 0:
            continue
        fn, ft = wr[0][2], np.hypot(wr[0][0], wr[0][1])
        assert fn >= 0.0
        if fn == 0.0:
            assert np.allclose(wr[0], 0.0)
            continue
        if ty[0] == 0:
            nstat += 1
            assert ft <= 0.5 * fn * (1 + 1e-9) + 1e-12
        else:
            nkin += 1
            assert ft <= 0.3 * fn * (1 + 1e-9) + 1e-12
    assert nstat > 5 and nkin > 5


def test_moving_vs_moving_contact_conserves_momentum_and_stacks(oracle):
    """Oracle pin of the moving-vs-moving pairs ([EXT A-10] extended; rkfd_util.c:42-60, 268-282): (1) two free boxes colliding in
    free fall exchange momentum - the total linear momentum changes by gravity only, the total angular momentum about the origin by
    the gravity torque only (the contact force acts on one body, its opposite on the other AT THE SAME POINT); (2) a box resting on
    another one on the soft floor: steady penetration m g / (4 E) of the upper box into the lower, 2 m g / (4 E) of the lower into
    the floor (four corner vertices each; the upper box is the smaller one - corners of equal aligned boxes slide along each other's
    faces and a vertex test never sees them)."""
    def mbox(name, side=0.1):
        return ch.ChainModel(name, [ch.Link(name="b", jtype="float", mass=0.5, stuff="body", inertia=np.eye(3) * 8.33e-4,
                                            boxes=[((0.0, 0.0, 0.0), side, side, side)])])
    ci = [ch.ContactInfo("body", "body", "elastic", E=2000.0, V=20.0, SF=0.5, KF=0.3), ch.ContactInfo("soft", "body", "elastic", E=1000.0, V=10.0, SF=0.5, KF=0.3)]
    # (1) collision in free fall
    w = ch.World(chains=[mbox("a"), mbox("b")], contact_info=ci)
    e = oracle.OracleWorld(w).env()
    q = np.zeros(12); q[0:3] = [-0.08, 0.01, 1.0]; q[6:9] = [0.08, -0.02, 1.03]; q[3:6] = [0.1, 0.2, 0.3]; q[9:12] = [-0.2, 0.1, 0.0]
    qd = np.zeros(12); qd[0] = 1.0; qd[6] = -1.5; qd[4] = 2.0; qd[11] = -1.0
    e.set_state(q, qd); e.update_init()
    m, I, g = 0.5, 8.33e-4, 9.80665

    def momenta():
        qq, vv, _ = e.get_state()
        P = m * (vv[0:3] + vv[6:9])
        L = sum(np.cross(qq[o:o + 3], m * vv[o:o + 3]) + I * vv[o + 3:o + 6] for o in (0, 6))       # isotropic inertia: I w in any frame
        return P, L, qq
    P0, L0, q0 = momenta()
    touched, Lg = False, np.zeros(3)
    for k in range(300):
        _, _, qq = momenta()
        Lg += 0.001 * sum(np.cross(qq[o:o + 3], [0, 0, -m * g]) for o in (0, 6))          # gravity torque about the origin (rectangle rule)
        e.update()
        touched |= e.get_contact()[0].sum() > 0
    P1, L1, _ = momenta()
    assert touched
    assert np.allclose(P1 - P0, [0, 0, -2 * m * g * 0.3], atol=1e-9)
    assert np.allclose(L1 - L0, Lg, atol=2e-3 * max(1.0, np.abs(Lg).max()))       # quadrature of the gravity torque limits this check
    # (2) resting stack
    w = ch.World(chains=[mbox("lower"), mbox("upper", 0.08), ch.floor_soft()], contact_info=ci)
    e = oracle.OracleWorld(w).env()
    q = np.zeros(12); q[2] = 0.05; q[8] = 0.14
    e.set_state(q, np.zeros(12)); e.update_init()
    for _ in range(4000):
        e.update()
    qq, vv, _ = e.get_state()
    assert np.abs(vv).max() < 1e-6
    assert abs((0.05 - qq[2]) - 2 * m * g / (4 * 1000.0)) < 1e-6 and abs((0.09 - (qq[8] - qq[2])) - m * g / (4 * 2000.0)) < 1e-6


@pytest.mark.parametrize("solver", ["MLCP", "Vert"])
def test_rigid_moving_vs_moving_contact_conserves_momentum(oracle, solver):
    """Oracle pin of RIGID contact between two moving links (rkfd_vert.c:125-185, rkfd_mlcp.c:76-142: A couples the two chains,
    the test force acts on one link and its opposite on the other): two free boxes colliding in free fall change their total
    linear momentum by gravity only, and they do not pass through each other; under the Vert solver a small box rests ON a larger
    one (rigid: no penetration between them) which sinks 2 m g / (4 E) into the soft floor."""
    def mbox(name, side=0.1):
        return ch.ChainModel(name, [ch.Link(name="b", jtype="float", mass=0.5, stuff="body", inertia=np.eye(3) * 8.33e-4,
                                            boxes=[((0.0, 0.0, 0.0), side, side, side)])])
    ci = [ch.ContactInfo("body", "body", "rigid", K=1000.0, L=0.01, SF=0.5, KF=0.3), ch.ContactInfo("soft", "body", "elastic", E=1000.0, V=10.0, SF=0.5, KF=0.3)]
    w = ch.World(chains=[mbox("a"), mbox("b")], contact_info=ci, solver=solver)
    e = oracle.OracleWorld(w).env()
    q = np.zeros(12); q[0:3] = [-0.08, 0.01, 1.0]; q[6:9] = [0.08, -0.02, 1.03]; q[3:6] = [0.1, 0.2, 0.3]; q[9:12] = [-0.2, 0.1, 0.0]
    qd = np.zeros(12); qd[0] = 1.0; qd[6] = -1.5; qd[4] = 2.0; qd[11] = -1.0
    e.set_state(q, qd); e.update_init()
    m, g = 0.5, 9.80665
    P0 = m * (qd[0:3] + qd[6:9]); touched = 0
    for _ in range(300):
        e.update(); touched += int(e.get_contact()[0].sum() > 0)
    qq, vv, _ = e.get_state()
    assert touched > 3
    assert np.allclose(m * (vv[0:3] + vv[6:9]) - P0, [0, 0, -2 * m * g * 0.3], atol=1e-9)
    assert vv[0] < 0.0 or vv[6] > vv[0] - 1e-9          # they bounced / stuck: box a no longer moves into box b
    if solver == "Vert":
        w = ch.World(chains=[mbox("lower"), mbox("upper", 0.08), ch.floor_soft()], contact_info=ci, solver=solver)
        e = oracle.OracleWorld(w).env()
        q = np.zeros(12); q[2] = 0.05; q[8] = 0.14
        e.set_state(q, np.zeros(12)); e.update_init()
        for _ in range(3000):
            e.update()
        qq, vv, _ = e.get_state()
        assert np.abs(vv).max() < 1e-9
        assert abs((0.05 - qq[2]) - 2 * m * g / (4 * 1000.0)) < 1e-7 and abs(0.09 - (qq[8] - qq[2])) < 1e-7


def test_slide_mode_conveyor_and_crawler(oracle):
    """Oracle pin of the slide mode (rkfd_util.c:26-40, 218-237): (1) a box dropped on a conveyor (static box in slide mode, belt
    speed 0.5 m/s, penalty contact) is dragged until it rides along at the belt speed and then STICKS (static friction: its
    anchors ride on the belt); (2) a box whose own cell is in slide mode propels itself over a plain floor in the opposite
    direction of its belt's surface velocity at the contact (a crawler), approaching the belt speed."""
    W = slide_worlds()
    e = oracle.OracleWorld(W["belt_registered_first_penalty"]()).env()
    q = np.zeros(6); q[2] = 0.05
    e.set_state(q, np.zeros(6)); e.update_init()
    for _ in range(1500):
        e.update()
    qq, vv, _ = e.get_state()
    act, typ = e.get_contact()[0], e.get_contact()[1]
    # (a slow pitch rate remains: the anchors ride at exactly the belt speed, the bottom vertices a little slower)
    assert abs(vv[0] - 0.5) < 2e-3 and np.abs(vv[[1, 2, 3, 5]]).max() < 1e-6 and abs(vv[4]) < 0.05 and act[:4].all() and (typ[:4] == 0).all()
    e = oracle.OracleWorld(W["crawler_box_on_plain_floor_penalty"]()).env()
    e.set_state(q, np.zeros(6)); e.update_init()
    for _ in range(1500):
        e.update()
    qq, vv, _ = e.get_state()
    assert abs(abs(vv[0]) - 0.3) < 5e-3 and qq[0] * vv[0] > 0
