"""World builders and state samplers the test modules share: the reference's own model files, moving-vs-moving and slide-mode
worlds, the brick wall, random trees for the kinematics walk with the oracle's frames to compare against, the workloads of the
external-wrench and mass-property tests, and the catalogue of the GPU batch tests."""
import copy
import os

import numpy as np

import rokifd_b200  # noqa: F401
from rokifd_b200 import chains as ch
from oracle.oracle import OracleWorld

NDOF = {"fixed": 0, "revolute": 1, "prismatic": 1, "cylindrical": 2, "hooke": 2, "spherical": 3, "float": 6, "breakablefloat": 6}
ALL_JOINTS = ("revolute", "prismatic", "spherical", "float", "cylindrical", "hooke", "breakablefloat")


# ---- the reference's own model files (tests/golden/flat_*.txt: what the C-ABI makes of example/model/*.ztk) -------------
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def flat_world(name, solver=None, soft=False):
    desc = ch.load_flat(os.path.join(GOLD, "flat_%s.txt" % name))
    w = ch.world_from_flat(desc)
    if solver:
        w.solver = solver
    if soft:      # every pair elastic (contactinfo.ztk's soft/body record): the penalty path on the reference's geometry
        for ci in w.contact_info:
            ci.type, ci.E, ci.V = "elastic", 1000.0, 10.0
    return w, np.array(desc["init.q[0]"])


def flat_states(name, w, q0, B, seed=0):
    rng = np.random.default_rng(seed)
    q = np.tile(q0, (B, 1)); qd = rng.uniform(-0.05, 0.05, (B, w.nq)); u = np.zeros((B, w.nl))
    if name.startswith("crawler"):         # crawler.ztk on the SOFT half of floor_hardsoft.ztk (y < 0), tracks on the floor
        q[:, 0:2] = np.array([0.0, -1.0]) + rng.uniform(-0.05, 0.05, (B, 2)); q[:, 2] = rng.uniform(-0.002, 0.004, B)    # (the body's frame: already holds z = 0.13)
        q[:, 3:6] = rng.uniform(-0.02, 0.02, (B, 3))
    elif name.startswith("mighty"):        # the humanoid near its registered standing pose, soles on the floor
        q[:, 6:] += 0.002 * rng.uniform(-1, 1, (B, w.nq - 6))
    else:                                  # arm_box_test.c: arm swung down towards the floor, box dropped next to it
        q[:, :2] = rng.uniform(-0.3, 0.3, (B, 2)) + np.array([np.pi / 2, 0.0]); qd[:, :2] = rng.uniform(-2, 2, (B, 2))
        q[:, 2:5] = np.array([0.0, 0.6, 0.06]) + rng.uniform(-0.02, 0.02, (B, 3)); q[:, 5:8] = rng.uniform(-0.3, 0.3, (B, 3))
    return q, qd, u


# ---- moving-vs-moving collision (SURVEY.md section 8(f)3): vertices of a cell against a box carried by another link ----------
def mm_box(name, stuff="body"):
    """box.ztk as a `type: box` shape: 8 collision vertices AND a box target for other bodies' vertices."""
    return ch.ChainModel(name, [ch.Link(name="link#00", jtype="float", mass=0.5, stuff=stuff, inertia=np.eye(3) * 8.33e-4,
                                        boxes=[((0.0, 0.0, 0.0), 0.1, 0.1, 0.1)])])


MM_CI = [ch.ContactInfo("soft", "body", "elastic", E=1000.0, V=10.0, SF=0.5, KF=0.3),
         ch.ContactInfo("body", "body", "elastic", E=2000.0, V=20.0, SF=0.5, KF=0.3)]


# the same bodies with RIGID contact info between them (what the reference's default contact info gives arm_box_test.c and
# boxdrop_test.c): the pair couples two chains in A (rkfd_vert.c:125-185, rkfd_mlcp.c:76-142)
MM_CI_RIGID = [ch.ContactInfo("soft", "body", "elastic", E=1000.0, V=10.0, SF=0.5, KF=0.3),
               ch.ContactInfo("body", "body", "rigid", K=1000.0, L=0.01, SF=0.5, KF=0.3)]


def mm_world(kind, solver="Vert"):
    rigid = kind.endswith("_rigid")
    ci = MM_CI_RIGID if rigid else MM_CI
    if kind.startswith("box_stack"):          # example/chain/boxdrop_test.c: boxes landing on each other (self pairs unregistered)
        nb = 2 if rigid else 3                # rigid: 2 boxes (3 x 8 x 2 + 16 = 32 slots is the limit of the vertex solvers)
        return ch.World(chains=[mm_box(n) for n in "abc"[:nb]] + [ch.floor_soft()], contact_info=ci, solver=solver)
    arm = ch.arm_2dof()              # example/chain/arm_box_test.c: the arm pushes a free box lying on the floor
    arm.links[2].boxes = [((0.2, 0.0, 0.0), 0.3, 0.1, 0.1)]
    return ch.World(chains=[arm, mm_box("box"), ch.floor_soft()], contact_info=ci, solver=solver)


def mm_states(kind, w, B, seed=0):
    rng = np.random.default_rng(seed)
    q = np.zeros((B, w.nq)); qd = np.zeros((B, w.nq)); u = np.zeros((B, w.nl))
    if kind.startswith("box_stack"):
        for k in range(w.nq // 6):
            o = 6 * k
            q[:, o:o + 2] = rng.uniform(-0.02, 0.02, (B, 2)); q[:, o + 2] = 0.05 + 0.105 * k + rng.uniform(0.0, 0.01, B)
            q[:, o + 3:o + 6] = rng.uniform(-0.1, 0.1, (B, 3)); qd[:, o:o + 6] = rng.uniform(-0.2, 0.2, (B, 6))
    else:
        q[:, 0] = rng.uniform(-0.3, 0.3, B); q[:, 1] = rng.uniform(-0.3, 0.3, B); qd[:, :2] = rng.uniform(-1, 1, (B, 2))
        # the free box starts in the path of the forearm's box primitive (link 2, centre (0.2, 0, 0) in its frame)
        ow = OracleWorld(w)
        for b in range(B):
            e = ow.env(); e.set_state(q[b], qd[b]); e.eval(False)
            Rs, ps = e.link_frames(); R, p = Rs[2], ps[2]
            q[b, 2:5] = p + R @ np.array([0.2, 0.0, 0.0]) + R @ np.array([0.0, 0.09, 0.0]) + rng.uniform(-0.005, 0.005, 3)
        q[:, 5:8] = rng.uniform(-0.2, 0.2, (B, 3))
        u[:, 1:3] = rng.uniform(-6, 6, (B, 2))
    return q, qd, u


# ---- the brick wall: breakable float joints ---------------------------------------------------------------------------
def brick_wall(fth, tth):
    """wall.ztk-like: a fixed base and three bricks sticking out sideways, held by breakable float joints (example/model/wall.ztk:51-95)."""
    links = [ch.Link(name="base", jtype="fixed", mass=1.0, inertia=np.eye(3) * 1e-2, org_p=np.array([0, 0, 1.0]), stuff="wall")]
    for k in range(3):
        links.append(ch.Link(name="b%d" % k, jtype="breakablefloat", parent=k, mass=0.25, com=np.array([0.05, 0, 0]),
                             inertia=np.diag([2.6e-4, 4.2e-4, 2.6e-4]), org_p=np.array([0.1, 0, 0]), stuff="wall",
                             break_force=fth[k], break_torque=tth[k], shapes=[ch.box_verts(0.1, 0.05, 0.05, center=(0.05, 0, 0))]))
    return ch.ChainModel("wall", links)


def brick_wall_world(fth, tth):
    """the brick wall with break forces fth and torques tth over the soft floor"""
    return ch.World(chains=[brick_wall(fth, tth), ch.floor_soft()],
                    contact_info=[ch.ContactInfo("soft", "wall", "elastic", E=1000.0, V=10.0)])


def brick_wall_states(w, B, seed):
    rng = np.random.default_rng(seed)
    q = np.zeros((B, w.nq)); qd = np.zeros((B, w.nq)); u = np.zeros((B, w.nl))
    q[:, 9:12] = rng.uniform(-0.05, 0.05, (B, 3))
    return q, qd, u


# ---- slide mode of collision cells --------------------------------------------------------------------------------------------
def slide_worlds():
    def belt(stuff, vel):       # a conveyor: static box whose link origin lies far below it, belt axis y -> surface velocity +x
        l = ch.Link(name="belt", jtype="fixed", stuff=stuff, org_p=np.array([0, 0, -100.0]), boxes=[((0, 0, 100 - 0.2), 50.0, 5.0, 0.4)])
        l.slides = {0: (vel, (0.0, 1.0, 0.0))}
        return ch.ChainModel("belt", [l])

    def mbox(name, slide=None):
        l = ch.Link(name="b", jtype="float", mass=0.5, stuff="body", inertia=np.eye(3) * 8.33e-4, shapes=[ch.box_verts(0.1, 0.1, 0.1)])
        if slide:
            l.slides = {0: slide}
        return ch.ChainModel(name, [l])
    el = [ch.ContactInfo("soft", "body", "elastic", E=1000.0, V=10.0, SF=0.5, KF=0.3)]
    rg = [ch.ContactInfo("soft", "body", "rigid", K=1000.0, L=0.01, SF=0.5, KF=0.3)]
    return {
        "belt_registered_second_penalty": lambda: ch.World(chains=[mbox("box"), belt("soft", 0.5)], contact_info=el),
        "belt_registered_first_penalty": lambda: ch.World(chains=[belt("soft", 0.5), mbox("box")], contact_info=el),
        "crawler_box_on_plain_floor_penalty": lambda: ch.World(chains=[mbox("box", (0.3, (0.0, 1.0, 0.0))), ch.floor_soft()], contact_info=el),
        "belt_mlcp": lambda: ch.World(chains=[mbox("box"), belt("soft", 0.5)], contact_info=rg, solver="MLCP"),
        "belt_registered_first_vert": lambda: ch.World(chains=[belt("soft", 0.5), mbox("box")], contact_info=rg, solver="Vert"),
    }


def slide_states(w, B, seed=1):
    rng = np.random.default_rng(seed)
    q = np.zeros((B, 6)); q[:, 2] = 0.05 + rng.uniform(0, 0.01, B); q[:, 3:6] = rng.uniform(-0.05, 0.05, (B, 3))
    return q, rng.uniform(-0.2, 0.2, (B, 6)), np.zeros((B, w.nl))


# ---- the kinematics walk: random trees and the oracle's frames at a state --------------------------------------------------
def as_broken(world, broken):
    """a copy of `world` in which the breakable-float joints of the flat link indices `broken` are float joints - what a
    broken joint is - so that the oracle holds them broken"""
    w = copy.deepcopy(world)
    k = 0
    for chn in w.moving_chains():
        for l in chn.links:
            if k in broken:
                assert l.jtype == "breakablefloat"
                l.jtype = "float"
            k += 1
    return w


def broken_links(world, piv_type):
    """per environment: the flat link indices whose breakable-float joint is broken (pivot bit of the joint's first dof)"""
    out, o = [[] for _ in range(piv_type.shape[0])], 0
    for k, l in enumerate(world.flat_links()):
        if l.jtype == "breakablefloat":
            for e in np.nonzero(piv_type[:, o])[0]:
                out[e].append(k)
        o += NDOF[l.jtype]
    return [tuple(b) for b in out]


def oracle_frames(world, q, qd, broken=None):
    """frames (B, nl, 12) and world-axis velocities (B, nl, 6) of the oracle at states (q, qd)"""
    B, nl = q.shape[0], world.nl
    fr, vel, worlds = np.zeros((B, nl, 12)), np.zeros((B, nl, 6)), {}
    for e in range(B):
        key = broken[e] if broken is not None else ()
        if key not in worlds:
            worlds[key] = OracleWorld(as_broken(world, key))
        env = worlds[key].env()
        env.set_state(q[e], qd[e])
        env.eval(False)
        R, p = env.link_frames()
        v = env.link_vel()                          # link axes
        fr[e, :, :9], fr[e, :, 9:] = R.reshape(nl, 9), p
        vel[e, :, :3] = np.einsum("kij,kj->ki", R, v[:, :3])
        vel[e, :, 3:] = np.einsum("kij,kj->ki", R, v[:, 3:])
    return fr, vel


def assert_frames_close(fr, vel, ofr, ovel, what):
    """R within 1e-12, p within 1e-12 (1 + |p|), velocities within 1e-11 (1 + |v|)"""
    dR = np.abs(fr[..., :9] - ofr[..., :9]).max()
    assert dR <= 1e-12, "%s: R differs by %.3g" % (what, dR)
    dp = (np.abs(fr[..., 9:] - ofr[..., 9:]) / (1 + np.abs(ofr[..., 9:]))).max()
    assert dp <= 1e-12, "%s: p differs by %.3g" % (what, dp)
    if vel is not None:
        dv = (np.abs(vel - ovel) / (1 + np.abs(ovel))).max()
        assert dv <= 1e-11, "%s: velocity differs by %.3g" % (what, dv)


def structured(rng, chain):
    """quarter-turn and identity org rotations (the structured transforms of the revolute joint) and org positions on the
    parent's z axis on some links"""
    for l in chain.links[1:]:
        r = rng.integers(5)
        if r == 0:
            l.org_R = np.eye(3)
        elif r == 1:
            l.org_R = ch.rot_x(np.pi / 2)
        elif r == 2:
            l.org_R = ch.rot_x(-np.pi / 2)
        if rng.integers(3) == 0:
            l.org_p = np.array([0.0, 0.0, rng.uniform(-0.3, 0.3)])
    return chain


def random_world(seed):
    """three chains (a floating-root tree, a fixed-root tree, a breakable-float root with a revolute arm), within the 32 dofs
    of the pivot word"""
    rng = np.random.default_rng(seed)
    while True:
        chains = [structured(rng, ch.random_chain(rng, n_links=6, jtypes=ALL_JOINTS, root="float", branching=True, name="a")),
                  structured(rng, ch.random_chain(rng, n_links=6, jtypes=ALL_JOINTS, root="fixed", branching=True, name="b")),
                  structured(rng, ch.random_chain(rng, n_links=3, jtypes=("revolute",), root="breakablefloat", name="c"))]
        w = ch.World(chains=chains)
        jts = {l.jtype for l in w.flat_links()}
        if w.nq <= 32 and len(jts) >= 5:
            return w


# ---- external wrenches and mass properties ------------------------------------------------------------------------------
def free_body(com=(0.03, -0.02, 0.05)):
    I = np.array([[0.02, 0.003, -0.001], [0.003, 0.03, 0.002], [-0.001, 0.002, 0.04]])
    return ch.World(chains=[ch.ChainModel("body", [ch.Link(name="b", jtype="float", mass=1.7, com=np.array(com), inertia=I)])])


def workload(name):
    """(world, links, sampler(B, seed) -> (q, qd, u, W), tolerance on q and q' relative to their largest entry)"""
    if name == "arm_box_floor":
        w, q0 = flat_world(name, soft=True)
        links = [3, 2]

        def sample(B, seed):
            q, qd, u = flat_states(name, w, q0, B, seed=seed)
            return q, qd, u, np.random.default_rng(seed).uniform(-3, 3, (B, 2, 6))
        return w, links, sample, 1e-9
    if name == "c4_volume":
        w = ch.world_c4_volume()

        def sample(B, seed):
            q, qd, u = ch.sample_c4_standing(w, B, seed=seed)
            W = np.zeros((B, 1, 6)); W[:, 0, :2] = np.random.default_rng(seed).uniform(-40, 40, (B, 2))   # a shove on the trunk
            return q, qd, u, W
        return w, [0], sample, 1e-6
    if name.startswith("c5"):
        w = ch.world_c5(base_z=0.3, solver="MLCP" if name == "c5_mlcp" else "Vert")

        def sample(B, seed):
            q, qd, u = ch.sample_state(w, B, seed=seed)
            W = np.random.default_rng(seed).uniform(-1, 1, (B, 2, 6)); W[:, 0, 2] -= 30.0      # the tip pushed into the floor
            return q, qd, u, W
        return w, [7, 4], sample, 1e-9 if name == "c5_mlcp" else 1e-7
    w = ch.world_c3(base_z=0.3)

    def sample(B, seed):
        q, qd, u = ch.sample_state(w, B, seed=seed)
        W = np.random.default_rng(seed).uniform(-10, 10, (B, 2, 6)); W[:, 0, 2] -= 20.0
        return q, qd, u, W
    return w, [7, 3], sample, 1e-9


# ---- the GPU batch tests ------------------------------------------------------------------------------------------------
def world(name):
    """(world, sampler(B, seed) -> (q, qd, u)) of a batch workload ("c4" is "c4_penalty")"""
    if name == "arm_box_floor":
        w, q0 = flat_world(name, soft=True)
        return w, lambda B, seed: flat_states(name, w, q0, B, seed=seed)
    if name == "brick_wall":
        w = brick_wall_world([200.0, 4.0, 10.0], [200.0, 0.3, 10.0])
        return w, lambda B, seed: brick_wall_states(w, B, seed)
    if name == "random_tree":
        w = random_world(11)
        return w, lambda B, seed: ch.sample_state(w, B, seed=seed)
    if name in ("c4", "c4_penalty", "c4_volume"):
        w = ch.world_c4_volume() if name == "c4_volume" else ch.world_c4_penalty()
        return w, lambda B, seed: ch.sample_c4_standing(w, B, seed=seed)
    w = {"c2": ch.world_c2, "c3": lambda: ch.world_c3(base_z=0.3), "c5_mlcp": lambda: ch.world_c5(base_z=0.3, solver="MLCP"),
         "c5_vert": lambda: ch.world_c5(base_z=0.3, solver="Vert")}[name]()
    return w, lambda B, seed: ch.sample_state(w, B, seed=seed)
