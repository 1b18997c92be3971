"""GPU parity tests proper (-m gpu): the CUDA path, called through the C-ABI (librokifd_b200.so via
rokifd_b200.capi), against the CPU oracle on the same seeded inputs.  Tolerances follow
BASELINE.json's north_star: accelerations and contact forces within 1e-9 relative per evaluation/step;
short-horizon trajectories within the tolerance stated in each test."""
import numpy as np
import pytest

import rokifd_b200  # noqa: F401
from rokifd_b200 import chains as ch
from gpu_batch import capi  # noqa: F401
from workloads import brick_wall_world, flat_world, flat_states, mm_world, mm_states, slide_worlds, slide_states

pytestmark = pytest.mark.gpu


def relerr(a, b):
    a, b = np.asarray(a, float), np.asarray(b, float)
    return np.abs(a - b).max() / max(np.abs(b).max(), 1e-12)


def gpu_world(capi, world, q, qd, u):
    fd, cells = capi.create_world(world, B=q.shape[0])
    fd.batch_set_state(q, qd)
    fd.batch_set_motor_input(u)
    fd.update_init()
    return fd


WORLDS = {
    "c2_arm7": lambda: ch.world_c2(),
    "c3_arm7_penalty": lambda: ch.world_c3(base_z=0.1),
    "c1_box_hardsoft": lambda: ch.World(chains=[ch.box(), ch.floor_hardsoft()],
                                        contact_info=[c for c in ch.contact_info_table() if c.type == "elastic"]
                                        + [ch.ContactInfo("ground", "body", "elastic", E=500.0, V=5.0)]),
    "c1_serial_arm2dof": lambda: ch.world_c1_serial(),
    "c4_biped_penalty": lambda: ch.world_c4_penalty(),
    "arm_and_box": lambda: ch.World(chains=[ch.arm_2dof(), ch.box(), ch.floor_soft()],
                                    contact_info=[ch.ContactInfo("soft", "body", "elastic", E=1000.0, V=10.0)]),
}


@pytest.mark.parametrize("name", list(WORLDS))
def test_init_evaluation_matches_oracle(capi, oracle, name):
    """rkFDUpdateInit's committing evaluation: q'', contact forces/state, friction pivots (1e-9 relative)."""
    w = WORLDS[name]()
    B = 256
    q, qd, u = ch.sample_state(w, B, seed=7)
    if "box" in name:
        o = w.nq - 6
        q[:, o + 2] = np.linspace(-0.02, 0.12, B)
    fd = gpu_world(capi, w, q, qd, u)
    gq, gqd, gqdd = fd.batch_get_state()
    a, t, r, f = fd.batch_get_contact()
    pt, pp = fd.batch_get_pivot()
    assert (fd.batch_get_status() == 0).all()
    ow = oracle.OracleWorld(w)
    worst = 0.0
    for b in range(B):
        e = ow.env(); e.set_state(q[b], qd[b]); e.set_motor_input(u[b])
        ref = e.eval(True)
        worst = max(worst, relerr(gqdd[b], ref))
        oa, ot, orr, of = e.get_contact()
        if w.nslot:
            assert (a[b] == oa).all() and (t[b][oa == 1] == ot[oa == 1]).all(), (name, b)
            assert np.allclose(f[b][oa == 1], of[oa == 1], rtol=1e-9, atol=1e-9)
            assert np.allclose(r[b][oa == 1], orr[oa == 1], rtol=1e-12, atol=1e-12)
        opt, opp = e.get_pivot()
        assert (pt[b] == opt).all() and np.allclose(pp[b], opp, rtol=1e-9, atol=1e-9)
    assert worst < 1e-9, (name, worst)
    fd.destroy()


@pytest.mark.parametrize("name", list(WORLDS))
def test_teacher_forced_steps_match_oracle(capi, oracle, name):
    """Per-step parity with the GPU state reset to the oracle state every step (SURVEY.md section 4, level 3)."""
    w = WORLDS[name]()
    B, nsteps = 64, 5
    q, qd, u = ch.sample_state(w, B, seed=13)
    if "box" in name:
        o = w.nq - 6
        q[:, o + 2] = np.linspace(0.0, 0.12, B)
    fd = gpu_world(capi, w, q, qd, u)
    ow = oracle.OracleWorld(w)
    envs = []
    for b in range(B):
        e = ow.env(); e.set_state(q[b], qd[b]); e.set_motor_input(u[b]); e.update_init(); envs.append(e)
    for s in range(nsteps):
        fd.update()
        gq, gqd, gqdd = fd.batch_get_state()
        oq = np.zeros_like(gq); oqd = np.zeros_like(gq); oqdd = np.zeros_like(gq)
        oa = np.zeros((B, max(w.nslot, 1)), np.int32); ot = oa.copy(); orr = np.zeros((B, max(w.nslot, 1), 3))
        opt = np.zeros((B, w.nq), np.int32); opp = np.zeros((B, w.nq))
        for b, e in enumerate(envs):
            e.update()
            oq[b], oqd[b], oqdd[b] = e.get_state()
            if w.nslot:
                oa[b], ot[b], orr[b], _ = e.get_contact()
            opt[b], opp[b] = e.get_pivot()
        assert relerr(gq, oq) < 1e-9 and relerr(gqd, oqd) < 1e-9, (name, s)
        for b in range(B):
            assert relerr(gqdd[b], oqdd[b]) < 1e-9, (name, s, b, relerr(gqdd[b], oqdd[b]))      # north_star's 1e-9 (measured: 1e-13-class)
        # teacher forcing: put the oracle's full state on the device
        fd.batch_set_state(oq, oqd)
        fd.batch_set_pivot(opt, opp)
        if w.nslot:
            fd.batch_set_contact(oa[:, :w.nslot], ot[:, :w.nslot], orr[:, :w.nslot])
    fd.destroy()


@pytest.mark.parametrize("name,tol", [("c2_arm7", 1e-8), ("c3_arm7_penalty", 1e-6), ("c1_box_hardsoft", 1e-6)])
def test_free_running_trajectory(capi, oracle, name, tol):
    """100 free-running steps: <=1e-8 relative on q without contact, <=1e-6 with contact, for >= 99% of the
    environments (contact/friction mode flips at zTOL-sized margins are counted and reported, not hidden)."""
    w = WORLDS[name]()
    B, nsteps = 128, 100
    q, qd, u = ch.sample_state(w, B, seed=21)
    if "box" in name:
        q[:, 2] = np.linspace(0.03, 0.15, B)
    fd = gpu_world(capi, w, q, qd, u)
    fd.update_n(nsteps)
    gq, gqd, _ = fd.batch_get_state()
    oq, oqd, _, _ = oracle.OracleWorld(w).batch_run(q, qd, u, nsteps=nsteps)
    err = np.array([relerr(gq[b], oq[b]) for b in range(B)])
    frac_ok = (err < tol).mean()
    print("free-running %s: %d/%d envs within %.0e (max err %.2e)" % (name, (err < tol).sum(), B, tol, err.max()))
    assert frac_ok >= 0.99
    fd.destroy()


@pytest.mark.parametrize("kind", ["branching", "float_root_tree", "spherical", "prismatic_mix", "cylindrical_hooke"])
def test_random_topologies(capi, oracle, kind):
    rng = np.random.default_rng({"branching": 1, "float_root_tree": 2, "spherical": 3, "prismatic_mix": 4, "cylindrical_hooke": 5}[kind])
    for trial in range(3):
        if kind == "branching":
            c = ch.random_chain(rng, 9, jtypes=("revolute", "prismatic"), branching=True, motors=True)
        elif kind == "float_root_tree":
            c = ch.random_chain(rng, 8, jtypes=("revolute", "fixed", "spherical"), root="float", branching=True)
        elif kind == "spherical":
            c = ch.random_chain(rng, 5, jtypes=("spherical", "revolute"))
        elif kind == "cylindrical_hooke":     # SURVEY.md section 8(f)2: the remaining RoKi joint types
            c = ch.random_chain(rng, 7, jtypes=("cylindrical", "hooke", "revolute"), root=("fixed", "float")[trial % 2], branching=trial == 2)
        else:
            c = ch.random_chain(rng, 6, jtypes=("revolute", "prismatic", "fixed"), motors=True)
        w = ch.World(chains=[c])
        B = 32
        q = rng.uniform(-1.5, 1.5, (B, w.nq)); qd = rng.uniform(-2, 2, (B, w.nq)); u = rng.uniform(-6, 6, (B, w.nl))
        fd = gpu_world(capi, w, q, qd, u)
        _, _, gqdd = fd.batch_get_state()
        ow = oracle.OracleWorld(w)
        for b in range(B):
            e = ow.env(); e.set_state(q[b], qd[b]); e.set_motor_input(u[b])
            assert relerr(gqdd[b], e.eval(True)) < 1e-9, (kind, trial, b)
        fd.update_n(5)
        gq, gqd, _ = fd.batch_get_state()
        oq, oqd, _, _ = ow.batch_run(q, qd, u, nsteps=5)
        assert relerr(gq, oq) < 1e-9 and relerr(gqd, oqd) < 1e-8, (kind, trial)
        fd.destroy()


def test_scalar_api_drop_in(capi, oracle):
    """B=1 through the scalar reference call sequence of example/chain/boxdrop_hardsoft_test.c:
    Create, ContactInfo, ChainReg, SetDis, SetSolver, UpdateInit, Update..., reading fd->dis/vel/acc."""
    w = ch.World(chains=[ch.box(), ch.floor_soft()], contact_info=[ch.ContactInfo("soft", "body", "elastic", E=100.0, V=1.0)])
    fd = capi.RkFD()
    for ci in w.contact_info:
        fd.contact_info_add(ci)
    cell = fd.chain_reg(w.chains[0])
    fd.chain_reg(w.chains[1])
    dis = np.array([0.0, 0.0, 0.3, 0.3, -0.2, 0.1])
    fd.chain_set_dis(cell, dis)
    fd.prp_set(dt=0.001)
    fd.set_solver("Vert")
    fd.update_init()
    e = oracle.OracleWorld(w).env()
    e.set_state(dis, np.zeros(6)); e.update_init()
    assert relerr(fd.acc, e.get_state()[2]) < 1e-9
    for s in range(300):
        fd.update(); e.update()
    oq, oqd, oqdd = e.get_state()
    assert abs(fd.time - 0.3) < 1e-12
    assert relerr(fd.dis, oq) < 1e-8 and relerr(fd.vel, oqd) < 1e-7
    fd.update_destroy()
    fd.destroy()


def test_shard_count_invariance_and_full_size(capi):
    """C3 at BASELINE.json's full batch (262,144 envs): results do not depend on how the batch is cut
    (two engines with different B see bit-identical per-env results), and every env stays finite."""
    w = ch.world_c3()
    B = 262144
    q, qd, u = ch.sample_state(w, B, seed=20260418)
    fd = gpu_world(capi, w, q, qd, u)
    fd.update_n(10)
    gq, gqd, gqdd = fd.batch_get_state()
    assert (fd.batch_get_status() == 0).all()
    assert np.isfinite(gq).all() and np.isfinite(gqd).all() and np.isfinite(gqdd).all()
    fd.destroy()
    lo, hi = 100000, 100000 + 4096
    fd2 = gpu_world(capi, w, q[lo:hi], qd[lo:hi], u[lo:hi])
    fd2.update_n(10)
    sq, sqd, sqdd = fd2.batch_get_state()
    assert np.array_equal(sq, gq[lo:hi]) and np.array_equal(sqd, gqd[lo:hi]) and np.array_equal(sqdd, gqdd[lo:hi])
    fd2.destroy()


def test_multi_device_sharding(capi, oracle):
    """env e -> device floor(e*G/B); per-env results identical to the single-device run."""
    G = capi.device_count()
    if G < 2:
        pytest.skip("needs >= 2 GPUs")
    w = ch.world_c3()
    B = 8192
    q, qd, u = ch.sample_state(w, B, seed=5)
    fd1 = gpu_world(capi, w, q, qd, u)
    fd1.update_n(10)
    ref = fd1.batch_get_state()
    fd1.destroy()
    fd, _ = capi.create_world(w, B=B, devices=list(range(G)))
    fd.batch_set_state(q, qd); fd.batch_set_motor_input(u); fd.update_init(); fd.update_n(10)
    got = fd.batch_get_state()
    for a, b in zip(ref, got):
        assert np.array_equal(a, b)
    fd.destroy()


def biped_pose(name, q):
    """The random trunk pose made a standing one (both soles near the floor)."""
    if "biped" in name:
        q[:, 2] = 0.44; q[:, 3:6] *= 0.1; q[:, 6:] *= 0.3
    return q


def biped_rigid(solver):
    """Contacts on TWO links of one tree (both soles on the rigid floor): the dense warp-cooperative contact solve."""
    return ch.World(chains=[ch.biped(), ch.floor()],
                    contact_info=[ch.ContactInfo("ground", "body", "rigid", K=1000.0, L=0.001, SF=0.5, KF=0.3)], solver=solver)


RIGID_WORLDS = {
    "c5_arm7_mlcp": lambda: ch.world_c5(base_z=0.1, solver="MLCP"),
    "biped_two_feet_mlcp": lambda: biped_rigid("MLCP"),
    "box_mlcp": lambda: ch.World(chains=[ch.box(), ch.floor()], contact_info=ch.contact_info_table(), solver="MLCP"),
    "box_hardsoft_mlcp": lambda: ch.World(chains=[ch.box(), ch.floor_hardsoft()], contact_info=ch.contact_info_table(), solver="MLCP"),
    "box_vert_default_ci": lambda: ch.World(chains=[ch.box(), ch.floor()], solver="Vert"),
    "arm7_vert_default_ci": lambda: ch.World(chains=[ch.arm7(base_z=0.1, contact_cube=True), ch.floor()], solver="Vert"),
    # two free bodies on the floor: contact links in different chains -> two groups of the wrench-coordinate paths
    "two_box_mlcp": lambda: ch.World(chains=[ch.box("a"), ch.box("b"), ch.floor()], contact_info=ch.contact_info_table(), solver="MLCP"),
    "two_box_vert_default_ci": lambda: ch.World(chains=[ch.box("a"), ch.box("b"), ch.floor()], solver="Vert"),
}

# Vert with relaxation L = 1e-4 (contactinfo.ztk): KKT matrices of condition ~1e7 against the absolute 1e-12 decision
# thresholds of the active-set loop (rkfd_opt_qp.c:33,110,148).  Round 1 agreed on 69 % of the contact environments of C5:
# the ORACLE's pseudo-inverse noise made x* of consecutive iterations differ by more than 1e-12 and the loop left through
# its anti-cycling exit short of the minimiser (the device path was at the minimiser every time: KKT residual 1e-10).
# With the oracle's zLESolveMP refined to rounding (pinned against 50-digit arithmetic, tests/test_oracle_physics.py)
# both sides follow the exact-arithmetic path.  (name, base height, environments, required share of contact environments
# within 1e-9).  "deep" pushes the cube up to 20 cm into the floor: |f dt| ~ 2e3, where 1e-12 is 4 ulp.
STAT_WORLDS = {
    "c5_arm7_vert": (lambda: ch.world_c5(base_z=0.3, solver="Vert"), 4096, 0.999, 1e-9),
    # a free box on the floor: same active sets and friction types everywhere; q'' of the 6-DoF body carries the rounding of
    # both solves amplified by cond(KKT) ~ 1e7 (measured: <= 3.7e-9, continuous - no path difference), hence 1e-8 here
    "box_vert": (lambda: ch.World(chains=[ch.box(), ch.floor()], contact_info=ch.contact_info_table(), solver="Vert"), 512, 0.999, 1e-8),
    "c5_arm7_vert_deep": (lambda: ch.world_c5(base_z=0.1, solver="Vert"), 512, 0.95, 1e-9),
}


@pytest.mark.parametrize("name", list(STAT_WORLDS))
def test_vert_qp_relaxation_1e_4(capi, oracle, name):
    mk, B, frac, tol = STAT_WORLDS[name]
    w = mk()
    q, qd, u = ch.sample_state(w, B, seed=20260418 if B == 4096 else 5)
    if "box" in name:
        q[:, 2] = np.linspace(-0.01, 0.08, B)
        q[:, 1] = np.linspace(-0.3, 0.3, B)
    fd = gpu_world(capi, w, q, qd, u)
    _, _, gqdd = fd.batch_get_state()
    a, t, r, f = fd.batch_get_contact()
    assert np.isfinite(gqdd).all()
    o = oracle.OracleWorld(w).batch_run_state(q, qd, u, nsteps=0)
    oqdd, oa, ot, of = o[2], o[3], o[4], o[5]
    assert (a == oa).all()
    err = np.abs(gqdd - oqdd).max(1) / np.maximum(np.abs(oqdd).max(1), 1e-12)
    m = (oa == 1)[:, :, None]                     # forces of the active slots (the others keep stale values on both sides)
    ferr = np.abs((f - of) * m).reshape(B, -1).max(1) / np.maximum(np.abs(of * m).reshape(B, -1).max(1), 1e-12)
    cont = oa.sum(1) > 0
    assert (err[~cont] < 1e-9).all()
    good = (err[cont] < tol) & (ferr[cont] < tol) & ((t == ot) | (oa == 0)).all(1)[cont]
    print("Vert QP %s: %d/%d contact envs within tolerance of the oracle (q'' and forces), worst q'' %.2e" % (name, good.sum(), cont.sum(), err[cont].max()))
    assert cont.sum() > 20 and good.sum() >= frac * cont.sum()
    fd.destroy()


@pytest.mark.parametrize("name", list(RIGID_WORLDS))
def test_rigid_evaluation_matches_oracle(capi, oracle, name):
    """Rigid contact (A,b by cached-ABA probes + solver) in one committing evaluation.  The Delassus matrix of
    N>DoF/3 contacts is rank deficient up to the 1e-4 relaxation, so rounding differences are amplified by
    cond(A) ~ 1e4..1e6; q'' and contact forces are nevertheless required within north_star's 1e-9 relative (measured
    on the B200 in round 2: at most 6.4e-13 over the eight worlds; the measured maximum is printed)."""
    w = RIGID_WORLDS[name]()
    B = 256
    q, qd, u = ch.sample_state(w, B, seed=5)
    q = biped_pose(name, q)
    if "box" in name:
        q[:, 2] = np.linspace(-0.01, 0.08, B)
        q[:, 1] = np.linspace(-0.3, 0.3, B)
    if "two_box" in name:
        q[:, 8] = np.linspace(0.07, -0.01, B); q[:, 6] += 2.0
    fd = gpu_world(capi, w, q, qd, u)
    _, _, gqdd = fd.batch_get_state()
    a, t, r, f = fd.batch_get_contact()
    ow = oracle.OracleWorld(w)
    worst, nc = 0.0, 0
    for b in range(B):
        e = ow.env(); e.set_state(q[b], qd[b]); e.set_motor_input(u[b])
        ref = e.eval(True)
        oa, ot, orr, of = e.get_contact()
        nc += oa.sum()
        assert (a[b] == oa).all() and (t[b][oa == 1] == ot[oa == 1]).all(), (name, b)
        worst = max(worst, relerr(gqdd[b], ref))
        assert np.allclose(f[b][oa == 1], of[oa == 1], rtol=1e-9, atol=1e-9 * max(1.0, np.abs(of).max()))
    print("rigid %s: %d contacts, max rel err of q'' %.2e" % (name, nc, worst))
    assert nc > 0 and worst < 1e-9
    fd.destroy()


@pytest.mark.parametrize("name", list(RIGID_WORLDS))
def test_rigid_short_trajectory(capi, oracle, name):
    w = RIGID_WORLDS[name]()
    B, nsteps = 128, 20
    q, qd, u = ch.sample_state(w, B, seed=9)
    q = biped_pose(name, q)
    if "box" in name:
        q[:, 2] = np.linspace(0.02, 0.08, B)
    if "two_box" in name:
        q[:, 8] = np.linspace(0.07, 0.03, B); q[:, 6] += 2.0
    fd = gpu_world(capi, w, q, qd, u)
    fd.update_n(nsteps)
    gq, gqd, _ = fd.batch_get_state()
    assert (fd.batch_get_status() == 0).all()
    oq, oqd, _, _ = oracle.OracleWorld(w).batch_run(q, qd, u, nsteps=nsteps)
    err = np.array([relerr(gq[b], oq[b]) for b in range(B)])
    print("rigid trajectory %s: %d/%d envs within 1e-6 (max %.2e)" % (name, (err < 1e-6).sum(), B, err.max()))
    assert (err < 1e-6).mean() >= 0.97
    fd.destroy()


def test_async_transfers_match_synchronous(capi):
    """rkFDBatchSet*Async / GetStateAsync (copy streams + staging ring) give the same result as the blocking calls."""
    import torch
    w = ch.world_c3(base_z=0.1)
    B = 4096
    q, qd, u = ch.sample_state(w, B, seed=3)
    fd = gpu_world(capi, w, q, qd, u)
    fd.update_n(3)
    ref = fd.batch_get_state()
    fd.destroy()
    fd = gpu_world(capi, w, q, qd, u)
    hq, hqd, hu = (torch.from_numpy(np.ascontiguousarray(x)).pin_memory() for x in (q, qd, u))
    oq, oqd, oqdd = (torch.empty((B, w.nq), dtype=torch.float64).pin_memory() for _ in range(3))
    for rep in range(4):          # more transfers than ring buffers in flight
        fd.batch_set_state_async(hq.data_ptr(), hqd.data_ptr())
        fd.batch_set_motor_input_async(hu.data_ptr())
        fd.batch_set_contact(np.zeros((B, w.nslot), np.int32), np.zeros((B, w.nslot), np.int32), np.zeros((B, w.nslot, 3)))
        fd.batch_set_pivot(np.zeros((B, w.nq), np.int32), np.zeros((B, w.nq)))
        fd.batch_eval(True)
        fd.update_n(3)
        fd.batch_get_state_async(oq.data_ptr(), oqd.data_ptr(), oqdd.data_ptr())
    fd.batch_sync()
    for a, b in zip(ref, (oq.numpy(), oqd.numpy(), oqdd.numpy())):
        assert np.array_equal(a, b)
    fd.destroy()


# (RKFD_SPEC, RKFD_FORCE_BLOCK, RKFD_FORCE_MINB): every compiled specialisation that C2/C3 (the 7-DoF arm) can run on
ARM7_VARIANTS = [(5, 128, 4), (5, 256, 2), (5, 512, 1), (3, 256, 2), (3, 512, 1), (3, 128, 4), (3, 128, 3),
                 (1, 128, 1), (1, 256, 1), (0, 128, 1)]


@pytest.mark.parametrize("variant", ARM7_VARIANTS, ids=lambda v: "spec%d_block%d_minb%d" % v)
def test_kernel_variants_agree(capi, oracle, monkeypatch, variant):
    """Every kernel variant of the serial-revolute specialisations (unrolled / rolled link loops, scratch in shared
    or tensor memory, 8-16 resident warps per SM) against the oracle after a committing evaluation + 25 steps of C3
    with contacts, and against the generic table-driven kernel (same arithmetic: agreement to rounding).  The
    batch covers several CTAs per SM so that co-resident CTAs share the SM's tensor memory."""
    spec, block, minb = variant
    w = ch.world_c3(base_z=0.1)
    B = 148 * 4 * 128 + 77
    q, qd, u = ch.sample_state(w, B, seed=21)

    def run(env):
        for k in ("RKFD_SPEC", "RKFD_FORCE_BLOCK", "RKFD_FORCE_MINB"):
            monkeypatch.delenv(k, raising=False)
        for k, v in env.items():
            monkeypatch.setenv(k, str(v))
        fd = gpu_world(capi, w, q, qd, u)
        kv = fd.kernel_variant()
        fd.update_n(25)
        out = fd.batch_get_state(), fd.batch_get_contact(), fd.batch_get_status(), kv
        fd.destroy()
        return out

    (gq, gqd, gqdd), (ga, gt, gr, gf), status, kv = run({"RKFD_SPEC": spec, "RKFD_FORCE_BLOCK": block, "RKFD_FORCE_MINB": minb})
    (rq, rqd, rqdd), (ra, rt, rr, rf), _, rkv = run({"RKFD_SPEC": 0})
    assert kv == (block, 0, 0, spec, minb) and rkv[3] == 0 and (spec == 0 or rkv != kv)       # the engine runs what was forced
    assert (status == 0).all()
    assert relerr(gq, rq) < 1e-11 and relerr(gqd, rqd) < 1e-10 and relerr(gqdd, rqdd) < 1e-8
    assert (ga == ra).mean() > 0.9999 and ga.sum() > 0
    n = 48
    oq, oqd, oqdd, _ = oracle.OracleWorld(w).batch_run(q[:n], qd[:n], u[:n], nsteps=25)
    assert relerr(gq[:n], oq) < 1e-9 and relerr(gqd[:n], oqd) < 1e-8


@pytest.mark.parametrize("variant", [(7, 128, 2, 0), (7, 128, 2, 1), (7, 64, 4, 1), (0, 128, 1, 0)],
                         ids=lambda v: "spec%d_block%d_minb%d_%s" % (v[0], v[1], v[2], "smem" if v[3] else "default"))
def test_rigid_mlcp_kernel_variants_agree(capi, oracle, monkeypatch, variant):
    """C5 with the MLCP solver (single-link wrench-space path): the rolled rigid specialisation (scratch column in HBM -
    the default - and in shared memory) and the generic kernel against each other and against the oracle, over a batch
    that fills several CTAs per SM."""
    spec, block, minb, smem = variant
    w = ch.world_c5(base_z=0.1, solver="MLCP")
    B = 148 * 2 * 128 + 33
    q, qd, u = ch.sample_state(w, B, seed=23)

    def run(env, nsteps):
        for k in ("RKFD_SPEC", "RKFD_FORCE_BLOCK", "RKFD_FORCE_MINB", "RKFD_FORCE_SMEM"):
            monkeypatch.delenv(k, raising=False)
        for k, v in env.items():
            monkeypatch.setenv(k, str(v))
        fd = gpu_world(capi, w, q, qd, u)
        first = fd.batch_get_state()[2].copy(), fd.batch_get_contact()
        kv = fd.kernel_variant()
        fd.update_n(nsteps)
        out = first, fd.batch_get_state(), kv
        fd.destroy()
        return out

    env = {"RKFD_SPEC": spec, "RKFD_FORCE_BLOCK": block, "RKFD_FORCE_MINB": minb}
    if smem:
        env["RKFD_FORCE_SMEM"] = 1
    (a1, c1), (q1, qd1, _), kv = run(env, 8)
    (a0, c0), (q0, qd0, _), rkv = run({"RKFD_SPEC": 0}, 8)
    # the rolled rigid kernel keeps its scratch column in device memory unless RKFD_FORCE_SMEM
    assert kv == (block, int(spec == 7 and not smem), 1, spec, minb) and rkv[2:4] == (1, 0) and (spec == 0 or rkv != kv)
    assert c0[0].sum() > 1000 and (c0[0] == c1[0]).all()
    assert relerr(a1, a0) < 1e-9
    fin = np.isfinite(q0).all(1) & (np.abs(q0).max(1) < 1e3)      # envs that start deep inside the floor blow up
    assert fin.mean() > 0.9
    d = np.abs(q1[fin] - q0[fin]).max(1)
    assert (d < 1e-8).mean() > 0.999
    n = 32
    ow = oracle.OracleWorld(w)
    for b in range(n):
        e = ow.env(); e.set_state(q[b], qd[b]); e.set_motor_input(u[b])
        ref = e.eval(True)
        assert relerr(a1[b], ref) < 1e-8, b


@pytest.mark.parametrize("integ", ["RK4", "Euler", "Heun"])
def test_integrator_menu(capi, oracle, integ):
    """rkFDODE2AssignRegular(fd, RK4 | Euler | Heun) through the C-ABI against the oracle (C3, 20 steps)."""
    w = ch.world_c3(base_z=0.1)
    w.integrator = integ
    B = 96
    q, qd, u = ch.sample_state(w, B, seed=41)
    fd = gpu_world(capi, w, q, qd, u)
    fd.update_n(20)
    gq, gqd, gqdd = fd.batch_get_state()
    fd.destroy()
    oq, oqd, oqdd, _ = oracle.OracleWorld(w).batch_run(q, qd, u, nsteps=20)
    assert relerr(gq, oq) < 1e-9 and relerr(gqd, oqd) < 1e-8


def test_divergent_slow_paths_keep_tensor_memory_accesses_converged(capi, monkeypatch):
    """Lanes of one warp take different branches around the warp-collective tensor-memory accesses of the
    specialised kernels: huge joint angles (the slow argument reduction of sincos) and joint velocities so large
    that the stage-to-stage angle addition falls back to sincos.  The kernels must neither hang nor disagree with
    the generic kernel."""
    w = ch.world_c3(base_z=0.45)
    B = 512
    q, qd, u = ch.sample_state(w, B, seed=77)
    rng = np.random.default_rng(5)
    big = rng.random(B) < 0.3
    q[big] += rng.uniform(-3e6, 3e6, (big.sum(), w.nq))
    fast = rng.random(B) < 0.3
    qd[fast] = rng.uniform(-400, 400, (fast.sum(), w.nq))
    out = []
    for spec in (0, 5, 3):
        monkeypatch.setenv("RKFD_SPEC", str(spec))
        fd = gpu_world(capi, w, q, qd, u)
        assert fd.kernel_variant()[3] == spec
        fd.update_n(3)
        out.append(fd.batch_get_state())
        fd.destroy()
    fin = np.isfinite(out[0][0]).all(1)
    assert fin.mean() > 0.95
    for o in out[1:]:
        assert (np.isfinite(o[0]).all(1) == fin).all()
        assert relerr(o[1][fin], out[0][1][fin]) < 1e-9


@pytest.mark.parametrize("name", ["c4_biped_penalty", "c1_box_hardsoft", "arm_and_box"])
def test_generic_kernel_with_tensor_memory_scratch(capi, monkeypatch, name):
    """The generic table-driven kernel with its T space in tensor memory (RKFD_SPEC=11: trees, floating bases, any joint
    mix without rigid pairs) against the shared-memory generic kernel: same arithmetic, agreement to rounding."""
    w = WORLDS[name]()
    B = 148 * 2 * 128 + 5
    q, qd, u = ch.sample_state(w, B, seed=29)
    out = []
    for spec in (0, 11):
        monkeypatch.setenv("RKFD_SPEC", str(spec))
        fd = gpu_world(capi, w, q, qd, u)
        assert fd.kernel_variant()[3] == spec
        fd.update_n(12)
        out.append(fd.batch_get_state())
        fd.destroy()
    fin = np.isfinite(out[0][0]).all(1)
    assert fin.mean() > 0.95
    for x, y in zip(out[0][:2], out[1][:2]):      # two instantiations: the compiler contracts a few products differently
        assert relerr(y[fin], x[fin]) < 1e-11


@pytest.mark.parametrize("nlinks,spec", [(3, 8), (7, 9), (8, 10)])
def test_general_frame_arm_specialisations(capi, oracle, monkeypatch, nlinks, spec):
    """Random fixed-base serial revolute arms with arbitrary constant frames (2 / 6 / 7 joints, DC motors + joint
    friction): the rolled general-frame specialisation against the generic kernel and the oracle."""
    rng = np.random.default_rng(100 + nlinks)
    w = ch.World(chains=[ch.random_chain(rng, nlinks, jtypes=("revolute",), motors=True)])
    B = 4096 + 17
    q = rng.uniform(-1.5, 1.5, (B, w.nq)); qd = rng.uniform(-2, 2, (B, w.nq)); u = rng.uniform(-6, 6, (B, w.nl))
    out = []
    for sid in (0, spec):
        monkeypatch.setenv("RKFD_SPEC", str(sid))
        fd = gpu_world(capi, w, q, qd, u)
        assert fd.kernel_variant()[3] == sid
        fd.update_n(15)
        out.append(fd.batch_get_state())
        fd.destroy()
    assert relerr(out[1][0], out[0][0]) < 1e-11 and relerr(out[1][1], out[0][1]) < 1e-10
    n = 24
    oq, oqd, _, _ = oracle.OracleWorld(w).batch_run(q[:n], qd[:n], u[:n], nsteps=15)
    assert relerr(out[1][0][:n], oq) < 1e-9 and relerr(out[1][1][:n], oqd) < 1e-8


# ---- Volume solver (rkfd_volume.c, BASELINE config C4): contact volume of a box cell against one face of the static box
VOLUME_WORLDS = {
    "box_volume": lambda: ch.World(chains=[ch.box(), ch.floor()], solver="Volume"),
    "box_volume_ci": lambda: ch.World(chains=[ch.box(), ch.floor()], contact_info=ch.contact_info_table(), solver="Volume"),
    "c4_biped_volume": lambda: ch.world_c4_volume(),                      # two pairs on one tree: coupled 12 x 12 QP
    "arm7_volume": lambda: ch.World(chains=[ch.arm7(base_z=0.1, contact_cube=True), ch.floor()], solver="Volume"),
    "two_box_volume": lambda: ch.World(chains=[ch.box("a"), ch.box("b"), ch.floor()], solver="Volume"),
}


def volume_pose(name, q):
    B = q.shape[0]
    if "biped" in name:
        q[:, 2] = 0.44; q[:, 3:6] *= 0.1; q[:, 6:] *= 0.3
    if "box" in name:
        q[:, 2] = np.linspace(0.0, 0.08, B); q[:, 3:6] *= 0.3
    if "two_box" in name:
        q[:, 8] = np.linspace(0.07, 0.01, B); q[:, 6] += 2.0
    return q


@pytest.mark.parametrize("name", list(VOLUME_WORLDS))
def test_volume_evaluation_matches_oracle(capi, oracle, name):
    """One committing evaluation with the Volume solver on the device: q'' within 1e-9, pair wrenches and volume
    centres (read back through the contact-force slots of the pair) against the oracle."""
    w = VOLUME_WORLDS[name]()
    B = 256
    q, qd, u = ch.sample_state(w, B, seed=5)
    q = volume_pose(name, q)
    fd = gpu_world(capi, w, q, qd, u)
    _, _, gqdd = fd.batch_get_state()
    a, t, r, f = fd.batch_get_contact()
    assert (fd.batch_get_status() == 0).all()
    ow = oracle.OracleWorld(w)
    nvol, worst = 0, 0.0
    for b in range(B):
        e = ow.env(); e.set_state(q[b], qd[b]); e.set_motor_input(u[b])
        ref = e.eval(True)
        npl, ty, wr, ce = e.volume()
        worst = max(worst, relerr(gqdd[b], ref))
        for p in range(len(npl)):
            if npl[p] <= 0 or not a[b][8 * p:8 * p + 8].any():
                continue
            nvol += 1
            got = f[b][8 * p:8 * p + 3].reshape(-1)
            assert np.allclose(got[:6], wr[p], rtol=1e-8, atol=1e-8 * max(1.0, np.abs(wr[p]).max())), (name, b, p)
            assert np.allclose(got[6:9], ce[p], atol=1e-10)
    print("volume %s: %d contact volumes, max rel err of q'' %.2e" % (name, nvol, worst))
    # relaxation 1e-4 (contactinfo.ztk) makes the QP Hessian ill conditioned (cond ~ 1e5): rounding differences of the
    # fused multiply-adds are amplified, 1e-7 there; 1e-9 (north_star) with the solver's own default contact info
    assert nvol > 0 and worst < (1e-7 if name.endswith("_ci") else 1e-9)
    fd.destroy()


@pytest.mark.parametrize("name", list(VOLUME_WORLDS))
def test_volume_short_trajectory(capi, oracle, name):
    w = VOLUME_WORLDS[name]()
    B, nsteps = 128, 20
    q, qd, u = ch.sample_state(w, B, seed=9)
    q = volume_pose(name, q)
    fd = gpu_world(capi, w, q, qd, u)
    fd.update_n(nsteps)
    gq, gqd, _ = fd.batch_get_state()
    assert (fd.batch_get_status() == 0).all()
    oq, oqd, _, _ = oracle.OracleWorld(w).batch_run(q, qd, u, nsteps=nsteps)
    err = np.array([relerr(gq[b], oq[b]) for b in range(B)])
    print("volume trajectory %s: %d/%d envs within 1e-6 (max %.2e)" % (name, (err < 1e-6).sum(), B, err.max()))
    assert (err < 1e-6).mean() >= 0.97
    fd.destroy()


# ---- edge cases: ragged batch sizes, worlds at the limits, nothing to do
@pytest.mark.parametrize("B", [1, 31, 33, 513])
@pytest.mark.parametrize("name", ["c3", "c4_volume", "c5_mlcp"])
def test_ragged_env_counts(capi, oracle, name, B):
    """Environment counts that fill neither a warp nor a block (the engine pads to whole blocks with zero-state
    environments): the real environments still match the oracle and no padding environment leaks into the results."""
    w = {"c3": lambda: ch.world_c3(base_z=0.1), "c4_volume": ch.world_c4_volume,
         "c5_mlcp": lambda: ch.world_c5(base_z=0.45, solver="MLCP")}[name]()
    q, qd, u = (ch.sample_c4_standing if name == "c4_volume" else ch.sample_state)(w, B, seed=77)
    fd = gpu_world(capi, w, q, qd, u)
    fd.update_n(5)
    gq, gqd, gqdd = fd.batch_get_state()
    assert gq.shape == (B, w.nq) and (fd.batch_get_status() == 0).all()
    oq, oqd, oqdd, _ = oracle.OracleWorld(w).batch_run(q, qd, u, nsteps=5)
    tq, tv = (1e-8, 1e-6) if name == "c4_volume" else (1e-9, 1e-8)      # Volume: the QP amplifies rounding (measured 1e-11-class per evaluation)
    for b in range(B):
        assert relerr(gq[b], oq[b]) < tq and relerr(gqd[b], oqd[b]) < tv, (name, B, b)
    fd.destroy()


def test_world_without_moving_chain_and_zero_steps(capi):
    """Only a static chain registered: UpdateInit succeeds or reports, nothing crashes; update_n(0) is a no-op."""
    w = ch.world_c3(base_z=0.1)
    q, qd, u = ch.sample_state(w, 64, seed=1)
    fd = gpu_world(capi, w, q, qd, u)
    before = fd.batch_get_state()
    n0 = fd.launch_count
    fd.update_n(0)
    after = fd.batch_get_state()
    assert fd.launch_count == n0 and all(np.array_equal(a, b) for a, b in zip(before, after))
    fd.destroy()


def test_set_dis_vel_and_motor_input_reach_a_running_simulator(capi, oracle):
    """rkFDChainSetDis / SetVel / rkJointMotorSetInput between two rkFDUpdate calls change what the next step integrates
    from (the reference's cell windows alias fd->dis/vel, rkfd_sim.c:277-287) - teleport / reset callers."""
    w = ch.World(chains=[ch.arm_2dof(), ch.box(), ch.floor_soft()], contact_info=[ch.ContactInfo("soft", "body", "elastic", E=1000.0, V=10.0)])
    fd = capi.RkFD()
    for ci in w.contact_info:
        fd.contact_info_add(ci)
    c_arm = fd.chain_reg(w.chains[0]); c_box = fd.chain_reg(w.chains[1]); fd.chain_reg(w.chains[2])
    q0 = np.array([0.3, -0.4, 0.0, 0.0, 0.2, 0.1, 0.2, 0.3])
    fd.chain_set_dis(c_arm, q0[:2]); fd.chain_set_dis(c_box, q0[2:])
    fd.update_init()
    e = oracle.OracleWorld(w).env(); e.set_state(q0, np.zeros(8)); e.update_init()
    for _ in range(5):
        fd.update(); e.update()
    # teleport the box, give the arm a velocity, switch a motor on
    newbox = np.array([0.1, -0.1, 0.08, 0.0, 0.3, 0.0]); newvel = np.array([1.5, -0.5])
    fd.chain_set_dis(c_box, newbox); fd.chain_set_vel(c_arm, newvel)
    c_arm.joint_motor_set_input(1, 3.0)
    oq, oqd, _ = e.get_state(); oq[2:] = newbox; oqd[:2] = newvel
    e.set_state(oq, oqd); u = np.zeros(w.nl); u[1] = 3.0; e.set_motor_input(u)
    for _ in range(5):
        fd.update(); e.update()
    oq, oqd, oqdd = e.get_state()
    assert relerr(fd.dis, oq) < 1e-9 and relerr(fd.vel, oqd) < 1e-9 and relerr(fd.acc, oqdd) < 1e-9
    assert not fd.chain_unreg(c_box)              # refused while the engine lives (as registration is)
    fd.update_destroy()
    assert fd.chain_unreg(c_box)
    fd.destroy()


def test_batch_stats(capi):
    w = ch.world_c3(base_z=0.1)
    B = 5000
    q, qd, u = ch.sample_state(w, B, seed=3)
    fd = gpu_world(capi, w, q, qd, u)
    fd.update_n(20)
    _, gqd, gqdd = fd.batch_get_state()
    a, _, _, _ = fd.batch_get_contact()
    s = fd.batch_stats()
    assert s[0] == B and s[1] == (a.sum(1) > 0).sum() and s[2] == a.sum() and s[3] == (fd.batch_get_status() != 0).sum()
    assert s[4] == np.abs(gqdd).max() and s[5] == np.abs(gqd).max()
    fd.destroy()


@pytest.mark.parametrize("name,soft,solver", [("mighty_on_floor", True, None), ("arm_box_floor", True, None), ("mighty_on_floor", False, "Volume"),
                                              ("boxdrop_hardsoft", False, "Vert"), ("crawler_on_hardsoft", False, None)])
def test_reference_model_files(capi, oracle, name, soft, solver):
    """The reference's own models (tests/golden/flat_*.txt = what rkFDChainRegFile + rkFDUpdateInit make of example/model/*.ztk,
    checked in tests/test_capi_host.py where the reference tree exists): mighty.ztk (25 links, 26 DoF, 701 collision vertices
    in 22 flag words; BASELINE config C4's model) standing on floor.ztk under the Volume solver and with penalty contact,
    arm_2DoF.ztk + box.ztk + floor.ztk (example/chain/arm_box_test.c) with penalty contact, box.ztk on floor_hardsoft.ztk
    (example/chain/boxdrop_hardsoft_test.c), crawler.ztk with both tracks in slide mode on the soft half of floor_hardsoft.ztk (the
    reference's fake crawler): one committing evaluation (1e-9) and 50 free-running steps."""
    w, q0 = flat_world(name, solver=solver, soft=soft)
    B = 256
    if name == "boxdrop_hardsoft":
        q, qd, u = ch.sample_state(w, B, seed=3); q[:, 2] = np.linspace(0.0, 0.12, B); q[:, 1] = np.linspace(-0.4, 0.4, B)
    else:
        q, qd, u = flat_states(name, w, q0, B)
    fd = gpu_world(capi, w, q, qd, u)
    _, _, gqdd = fd.batch_get_state()
    a, t, r, f = fd.batch_get_contact()
    o = oracle.OracleWorld(w).batch_run_state(q, qd, u, nsteps=0)
    assert (a == o[3]).all() and o[3].sum() > 0 and (fd.batch_get_status() == 0).all()
    err = np.abs(gqdd - o[2]).max(1) / np.maximum(np.abs(o[2]).max(1), 1e-12)
    assert (err < 1e-9).mean() >= (0.99 if name == "boxdrop_hardsoft" else 1.0), (np.sort(err)[-5:])
    fd.update_n(50)
    gq, _, _ = fd.batch_get_state()
    oq = oracle.OracleWorld(w).batch_run_state(q, qd, u, nsteps=50)[0]
    errq = np.abs(gq - oq).max(1) / np.abs(oq).max(1)
    print("reference model %s (%s): q'' max rel err %.2e; after 50 steps %d/%d envs within 1e-7 (max %.2e)" % (
        name, w.solver if not soft else "penalty", err.max(), (errq < 1e-7).sum(), B, errq.max()))
    assert (errq < 1e-7).mean() >= (1.0 if soft or name.startswith("crawler") else 0.9)
    if name.startswith("crawler"):
        fd.update_n(250)
        assert (fd.batch_get_state()[1][:, 0] > 0.2).all()         # it drives: forward at about the belt speed (0.3 m/s)
    fd.destroy()


@pytest.mark.parametrize("name", ["c3", "c5_mlcp", "arm_box_floor", "c5_vert", "c4_volume"])
def test_environment_resort_is_invisible(capi, name):
    """The engine re-orders its slots by contact count - under the Vert / Volume solvers by the work class the step kernel leaves
    per environment (StateDev::work) - while stepping (rkFDBatchSetResortInterval): every host-side result - state, accelerations,
    contact flags / anchors / forces, friction pivots, status - is bit-identical to a run without it, also when state and motor
    inputs are written between the sorts.  The Volume world sorts every step (its default), the Vert world every 4."""
    intervals = (0, 7)
    if name == "arm_box_floor":
        w, q0 = flat_world(name, soft=True)
        B = 3000
        q, qd, u = flat_states(name, w, q0, B)
    elif name == "c4_volume":
        w = ch.world_c4_volume(); B = 6000; intervals = (0, 1)
        q, qd, u = ch.sample_c4_standing(w, B, seed=5)
    else:
        w = ch.world_c3(base_z=0.3) if name == "c3" else ch.world_c5(base_z=0.3, solver="MLCP" if name == "c5_mlcp" else "Vert")
        B = 20000
        if name == "c5_vert": intervals = (0, 4)
        q, qd, u = ch.sample_state(w, B, seed=11)
    out = []
    for interval in intervals:
        fd, _ = capi.create_world(w, B=B)
        fd.batch_set_resort_interval(interval)
        fd.batch_set_state(q, qd); fd.batch_set_motor_input(u); fd.update_init()
        for seg in range(6):
            for _ in range(20 if name != "c4_volume" else 6):
                fd.update()
            if seg == 2:       # inputs written mid-run go to the right environments
                u2 = u.copy(); u2[::3] *= -1.0
                fd.batch_set_motor_input(u2)
            if seg == 3:
                gq, gqd, _ = fd.batch_get_state(); gq[::5] += 0.01
                fd.batch_set_state(gq, gqd)
        res = list(fd.batch_get_state()) + list(fd.batch_get_contact()) + list(fd.batch_get_pivot()) + [fd.batch_get_status()]
        out.append((res, fd.resort_count))
        fd.destroy()
    assert out[0][1] == 0 and out[1][1] >= 10
    a_act = out[0][0][3]
    assert a_act.sum() > 0
    for x, y in zip(out[0][0], out[1][0]):
        if x.ndim == 3:            # anchors / forces: compared on active slots (inactive ones keep stale values)
            m = (a_act == 1)[:, :, None]
            assert np.array_equal(x * m, y * m)
        else:
            assert np.array_equal(x, y)


@pytest.mark.parametrize("kind", ["box_stack", "arm_pushes_box"])
def test_moving_vs_moving_contact(capi, oracle, kind):
    """SURVEY.md section 8(f)3: cells of two MOVING links in contact (vertices of one against a box primitive of the other,
    relative velocity of both links rkfd_util.c:42-60, force on one and its opposite on the other rkfd_util.c:268-282):
    three free boxes landing on each other (example/chain/boxdrop_test.c) and an arm pushing a free box
    (example/chain/arm_box_test.c), penalty contact, 200 free-running steps against the oracle."""
    w = mm_world(kind)
    B = 512
    q, qd, u = mm_states(kind, w, B)
    fd = gpu_world(capi, w, q, qd, u)
    assert fd.slot_num == w.nslot
    fd.update_n(200)
    gq, gqd, _ = fd.batch_get_state()
    a, t, r, f = fd.batch_get_contact()
    o = oracle.OracleWorld(w).batch_run_state(q, qd, u, nsteps=200)
    nstat = sum(v.shape[0] for l in w.flat_links() for v in l.cells()) * len(w.boxes)
    assert (fd.batch_get_status() == 0).all()
    err = np.abs(gq - o[0]).max(1) / np.abs(o[0]).max(1)
    same = (a == o[3]).all(1)
    print("moving-vs-moving %s: %d/%d envs within 1e-8 after 200 steps (max %.2e), contact flags equal in %d, moving-pair contacts at the end: %d" % (
        kind, (err < 1e-8).sum(), B, err.max(), same.sum(), o[3][:, nstat:].sum()))
    assert (err < 1e-8).mean() >= 0.99 and same.mean() >= 0.99
    fd.destroy()


@pytest.mark.parametrize("kind,solver", [("box_stack_rigid", "MLCP"), ("arm_pushes_box_rigid", "MLCP"), ("arm_pushes_box_rigid", "Vert")])
def test_rigid_moving_vs_moving_contact(capi, oracle, kind, solver):
    """SURVEY.md section 8(f)3, the rigid half: RIGID contact info between two moving links (what the reference's default contact
    info gives example/chain/arm_box_test.c and boxdrop_test.c) - A couples the two links / chains (rkfd_vert.c:125-185,
    rkfd_mlcp.c:76-142): relative point acceleration / velocity (rkfd_util.c:42-60, 103-118), probes with the opposite unit force
    on the partner, opposite wrenches.  The committing evaluation and 100 free-running steps against the oracle."""
    w = mm_world(kind, solver)
    # the dense Vert QP serves the environments of a warp one after the other, every active-set iteration with a Jacobi
    # eigen-decomposition in the per-warp workspace: small batch (two boxes lying flat on each other - 8 rigid contacts,
    # up to 64 active pyramid rows - are covered on the host harness, tests/test_kernel_core_host.py)
    B = 256 if solver == "MLCP" else 32
    q, qd, u = mm_states(kind, w, B, seed=3)
    ow = oracle.OracleWorld(w)
    # states with the moving pair in contact: 60 oracle steps in
    o60 = ow.batch_run_state(q, qd, u, nsteps=60)
    fd = gpu_world(capi, w, q, qd, u)
    assert fd.slot_num == w.nslot
    fd.update_n(60)
    g60 = fd.batch_get_state(); a60 = fd.batch_get_contact()[0]
    nstat = sum(v.shape[0] for l in w.flat_links() for v in l.cells()) * len(w.boxes)
    ok = np.isfinite(o60[0]).all(1)
    err60 = np.abs(g60[0] - o60[0]).max(1) / np.maximum(np.abs(o60[0]).max(1), 1e-12)
    fd.update_n(40)
    gq = fd.batch_get_state()[0]; a = fd.batch_get_contact()[0]
    o = ow.batch_run_state(q, qd, u, nsteps=100)
    ok &= np.isfinite(o[0]).all(1)
    err = np.abs(gq - o[0]).max(1) / np.maximum(np.abs(o[0]).max(1), 1e-12)
    same = (a == o[3]).all(1)
    print("rigid moving-vs-moving %s/%s: %d/%d envs within 1e-8 after 60 steps, %d after 100 (max %.2e), flags equal in %d, moving-pair contacts: %d / %d" % (
        kind, solver, (err60[ok] < 1e-8).sum(), ok.sum(), (err[ok] < 1e-8).sum(), err[ok].max(), same[ok].sum(), o60[3][:, nstat:].sum(), o[3][:, nstat:].sum()))
    assert o60[3][:, nstat:].sum() + o[3][:, nstat:].sum() > 0
    # mode flips at zTOL-sized margins split trajectories; the dense Vert path finds its multipliers by a Jacobi pseudo-inverse
    # where the oracle refines zLESolveMP to rounding (measured on the B200: MLCP 256/256, Vert 27/32 within 1e-8 after 60 steps)
    share = 0.95 if solver == "MLCP" else 0.75
    assert (err60[ok] < 1e-8).mean() >= share and (err[ok] < 1e-7).mean() >= share - 0.1 and same[ok].mean() >= share - 0.1
    fd.destroy()


@pytest.mark.parametrize("name", ["belt_registered_second_penalty", "belt_registered_first_penalty", "crawler_box_on_plain_floor_penalty",
                                  "belt_mlcp", "belt_registered_first_vert"])
def test_slide_mode(capi, oracle, name):
    """SURVEY.md section 8(f)4, the slide mode ("fake crawler", rkfd_sim.c:386-440): set through the reference's own calls
    (rkFDShape3DSetSlideMode / -Vel / -Axis on a shape of the registered chain), belt velocity in the relative contact velocity
    (rkfd_util.c:26-40), anchors of sticking contacts riding on the belt (:218-237); penalty, MLCP and Vert; 400 steps against
    the oracle."""
    w = slide_worlds()[name]()
    B = 256
    q, qd, u = slide_states(w, B)
    fd = gpu_world(capi, w, q, qd, u)
    fd.update_n(400)
    gq = fd.batch_get_state()[0]; a = fd.batch_get_contact()[0]
    o = oracle.OracleWorld(w).batch_run_state(q, qd, u, nsteps=400)
    err = np.abs(gq - o[0]).max(1) / np.maximum(np.abs(o[0]).max(1), 1e-12)
    print("slide mode %s: max rel err of q after 400 steps %.2e, flags equal in %d/%d, mean x %.4f" % (name, err.max(), (a == o[3]).all(1).sum(), B, o[0][:, 0].mean()))
    assert (fd.batch_get_status() == 0).all() and np.abs(o[0][:, 0]).mean() > 0.005
    tol = 1e-9 if "vert" not in name else 1e-6
    assert (err < tol).mean() >= (1.0 if "vert" not in name else 0.97) and (a == o[3]).all(1).mean() >= 0.97
    fd.destroy()


def test_breakable_float_joint(capi, oracle):
    """SURVEY.md section 8(f)2: the breakable float joint of example/model/wall.ztk:51-95 ([EXT A-17]): a cantilever of three
    bricks whose middle joint gives way under gravity; 400 steps against the oracle."""
    w = brick_wall_world([200.0, 4.0, 10.0], [200.0, 0.3, 10.0])
    B = 256
    rng = np.random.default_rng(0)
    q = np.zeros((B, w.nq)); qd = np.zeros((B, w.nq)); u = np.zeros((B, w.nl))
    q[:, 9:12] = rng.uniform(-0.05, 0.05, (B, 3))
    fd = gpu_world(capi, w, q, qd, u)
    assert (fd.batch_get_pivot()[0][:, [0, 6, 12]] == [0, 1, 0]).all()        # broken flag = pivot bit of the joint's first dof
    fd.update_n(400)
    gq, gqd, _ = fd.batch_get_state()
    o = oracle.OracleWorld(w).batch_run_state(q, qd, u, nsteps=400)
    assert (fd.batch_get_status() == 0).all()
    assert np.abs(gq - o[0]).max() < 1e-9 and (gq[:, 8] < -0.5).all() and (gq[:, :6] == q[:, :6]).all()
    fd.destroy()
