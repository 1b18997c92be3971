"""The step-kernel variant matrix: every compiled instantiation of rkfd_step_kernel (roki-fd_b200/csrc/Makefile VARIANTS,
RKFD_VARIANT_LIST in rkfd_engine.cu), written (block, gscr, rigid, spec, minb), mapped to a world that selects it, a state
sampler and the tuning variables that force it.  One table for the host tests (tests/test_variant_matrix_host.py: the lists
agree, every specialisation id is covered and matches its world) and the GPU tests (tests/test_gpu_variants.py: the engine
reports the tuple, and the variant agrees with the generic kernel and the oracle)."""
import os
import re
from collections import namedtuple

import numpy as np

from rokifd_b200 import chains as ch

CSRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "roki-fd_b200", "csrc")

# the tuning variables Engine::Engine reads when it picks a variant
TUNING_VARS = ("RKFD_SPEC", "RKFD_FORCE_BLOCK", "RKFD_FORCE_MINB", "RKFD_FORCE_GSCR", "RKFD_FORCE_SMEM", "RKFD_SMEM_PAD")

SOFT = ch.ContactInfo("soft", "body", "elastic", E=1000.0, V=10.0, SF=0.5, KF=0.3)
RIGID = ch.ContactInfo("ground", "body", "rigid", K=1000.0, L=0.001, SF=0.5, KF=0.3)


def cell_min_z(chain, q):
    """Lowest world z of the cell vertices of the last link of a fixed-base serial revolute chain, per state (R_i =
    R_parent Ro_i Rz(q_i), p_i = p_parent + R_parent po_i)."""
    v = chain.links[-1].cells()[0]
    out = np.zeros(q.shape[0])
    for b in range(q.shape[0]):
        R, p, j = np.eye(3), np.zeros(3), 0
        for l in chain.links:
            p = p + R @ l.org_p
            R = R @ l.org_R
            if l.jtype == "revolute":
                R = R @ ch.rot_z(q[b, j])
                j += 1
        out[b] = (p + v @ R.T)[:, 2].min()
    return out


def _pose_base(chain, q, share):
    """Lifts the fixed base so that the cube of the last link dips below the floor in `share` of the states q (shallowly:
    the base height is a quantile of the states' lowest vertex)."""
    lo = cell_min_z(chain, q)
    chain.links[0].org_p = chain.links[0].org_p + np.array([0.0, 0.0, -np.quantile(lo, share)])
    return chain


def _sample_arm(w, B, seed):
    return ch.sample_state(w, B, seed=seed)


def arm6_cube():
    """The 7-DoF arm cut to 6 quarter-turn revolute joints, the cube of box.ztk on link 6, the soft floor (spec 6)."""
    a = ch.arm7(base_z=0.0, contact_cube=False)
    a.links = a.links[:7]
    a.links[6].shapes = [ch.box_verts(0.1, 0.1, 0.1, center=(0, 0, 0.1))]
    w = ch.World(chains=[a, ch.floor_soft()], contact_info=[SOFT])
    _pose_base(a, ch.sample_state(w, 256, seed=1)[0], 0.35)
    return w


def arm2dof_cube():
    """arm_2DoF.ztk with the cube of box.ztk at the tip of link 2, the soft floor (specs 2 and 4)."""
    a = ch.arm_2dof()
    a.links[2].shapes = [ch.box_verts(0.1, 0.1, 0.1, center=(0.4, 0, 0))]
    w = ch.World(chains=[a, ch.floor_soft()], contact_info=[SOFT])
    _pose_base(a, ch.sample_state(w, 256, seed=1)[0], 0.35)
    return w


def general_arm_cube(nlinks):
    """A random fixed-base serial revolute arm with general constant frames (DC motors, joint friction), the cube of box.ztk
    on its last link, posed over the soft floor (specs 8, 9, 10: 2, 6 and 7 joints)."""
    rng = np.random.default_rng(100 + nlinks)
    a = ch.random_chain(rng, nlinks, jtypes=("revolute",), motors=True, shapes=True)
    w = ch.World(chains=[a, ch.floor_soft()], contact_info=[SOFT])
    _pose_base(a, ch.sample_state(w, 256, seed=1)[0], 0.35)
    return w


def biped_pose(q):
    """The random trunk pose of sample_state made a standing one (both soles near the floor)."""
    q[:, 2] = 0.44; q[:, 3:6] *= 0.1; q[:, 6:] *= 0.3
    return q


def _sample_biped(w, B, seed):
    q, qd, u = ch.sample_state(w, B, seed=seed)
    return biped_pose(q), qd, u


def _sample_box(w, B, seed):
    """The box nearly flat and slow, its lowest corners within 1 cm of the floor: rigid contacts that last"""
    q, qd, u = ch.sample_state(w, B, seed=seed)
    q[:, 3:6] *= 0.1; qd *= 0.1
    q[:, 2] = np.linspace(0.04, 0.06, B)
    q[:, 1] = np.linspace(-0.3, 0.3, B)
    return q, qd, u


def _sample_c4(w, B, seed):
    return ch.sample_c4_standing(w, B, seed=seed)


# name -> (world builder, state sampler (world, B, seed), class).  Classes: "penalty" (vertex penalty contact: the kernels
# agree to rounding), "mlcp" (rigid contact, MLCP), "vert" (rigid contact, Vert QP: ill-conditioned KKT systems), "volume"
World_ = namedtuple("World_", "make sample cls")
WORLDS = {
    "c3": World_(lambda: ch.world_c3(base_z=0.1), _sample_arm, "penalty"),
    "arm6_cube": World_(arm6_cube, _sample_arm, "penalty"),
    "arm2dof_cube": World_(arm2dof_cube, _sample_arm, "penalty"),
    "general_arm3_cube": World_(lambda: general_arm_cube(3), _sample_arm, "penalty"),
    "general_arm7_cube": World_(lambda: general_arm_cube(7), _sample_arm, "penalty"),
    "general_arm8_cube": World_(lambda: general_arm_cube(8), _sample_arm, "penalty"),
    "biped_penalty": World_(ch.world_c4_penalty, _sample_biped, "penalty"),
    "c5_mlcp": World_(lambda: ch.world_c5(base_z=0.1, solver="MLCP"), _sample_arm, "mlcp"),
    "c5_vert": World_(lambda: ch.world_c5(base_z=0.3, solver="Vert"), _sample_arm, "vert"),
    "box_mlcp": World_(lambda: ch.World(chains=[ch.box(), ch.floor()], contact_info=ch.contact_info_table(), solver="MLCP"), _sample_box, "mlcp"),
    "biped_rigid_mlcp": World_(lambda: ch.World(chains=[ch.biped(), ch.floor()], contact_info=[RIGID], solver="MLCP"), _sample_c4, "mlcp"),
    "c4_volume": World_(ch.world_c4_volume, _sample_c4, "volume"),
}

Row = namedtuple("Row", "variant world env")


def _row(variant, world, **env):
    return Row(tuple(variant), world, {k: str(v) for k, v in env.items()})


# one row per compiled variant; env: the tuning variables that select it (none: the engine's own choice for that world)
MATRIX = [
    # unrolled 7-DoF arm, scratch in tensor memory
    _row((128, 0, 0, 3, 4), "c3", RKFD_SPEC=3, RKFD_FORCE_BLOCK=128, RKFD_FORCE_MINB=4),
    _row((128, 0, 0, 3, 3), "c3", RKFD_SPEC=3, RKFD_FORCE_BLOCK=128, RKFD_FORCE_MINB=3),
    _row((256, 0, 0, 3, 2), "c3", RKFD_SPEC=3, RKFD_FORCE_BLOCK=256, RKFD_FORCE_MINB=2),
    _row((512, 0, 0, 3, 1), "c3", RKFD_SPEC=3, RKFD_FORCE_BLOCK=512, RKFD_FORCE_MINB=1),
    # unrolled 7-DoF arm, shared memory
    _row((128, 0, 0, 1, 1), "c3", RKFD_SPEC=1, RKFD_FORCE_BLOCK=128),
    _row((256, 0, 0, 1, 1), "c3", RKFD_SPEC=1, RKFD_FORCE_BLOCK=256),
    # rolled quarter-turn arms
    _row((128, 0, 0, 5, 4), "c3", RKFD_SPEC=5, RKFD_FORCE_BLOCK=128, RKFD_FORCE_MINB=4),
    _row((256, 0, 0, 5, 2), "c3", RKFD_SPEC=5, RKFD_FORCE_BLOCK=256, RKFD_FORCE_MINB=2),
    _row((512, 0, 0, 5, 1), "c3", RKFD_SPEC=5, RKFD_FORCE_BLOCK=512, RKFD_FORCE_MINB=1),
    _row((256, 0, 0, 6, 2), "arm6_cube", RKFD_SPEC=6),
    # unrolled arm_2DoF, shared / tensor memory
    _row((128, 0, 0, 2, 1), "arm2dof_cube", RKFD_SPEC=2),
    _row((128, 0, 0, 4, 4), "arm2dof_cube", RKFD_SPEC=4),
    # rolled general-frame arms
    _row((128, 0, 0, 8, 4), "general_arm3_cube", RKFD_SPEC=8),
    _row((128, 0, 0, 9, 4), "general_arm7_cube", RKFD_SPEC=9),
    _row((128, 0, 0, 10, 4), "general_arm8_cube", RKFD_SPEC=10),
    # generic kernel, T space in tensor memory
    _row((128, 0, 0, 11, 2), "biped_penalty", RKFD_SPEC=11),
    # generic kernel, shared memory (C3's generic column is 110 doubles: 225 KB at 256 threads)
    _row((128, 0, 0, 0, 1), "c3", RKFD_SPEC=0, RKFD_FORCE_BLOCK=128),
    _row((256, 0, 0, 0, 1), "c3", RKFD_SPEC=0, RKFD_FORCE_BLOCK=256),
    _row((64, 0, 0, 0, 1), "biped_penalty", RKFD_SPEC=0, RKFD_FORCE_BLOCK=64),
    _row((32, 0, 0, 0, 1), "biped_penalty", RKFD_SPEC=0, RKFD_FORCE_BLOCK=32),
    # generic kernel, scratch in device memory
    _row((64, 1, 0, 0, 1), "biped_penalty", RKFD_SPEC=0, RKFD_FORCE_GSCR=1, RKFD_FORCE_BLOCK=64),
    # rolled rigid 7-DoF arm: scratch in device memory (the default) and in shared memory
    _row((128, 1, 1, 7, 2), "c5_mlcp"),
    _row((128, 0, 1, 7, 2), "c5_vert", RKFD_FORCE_SMEM=1),
    _row((64, 0, 1, 7, 4), "c5_mlcp", RKFD_FORCE_SMEM=1, RKFD_FORCE_BLOCK=64),
    # generic rigid kernel, shared memory
    _row((128, 0, 1, 0, 1), "c5_mlcp", RKFD_SPEC=0, RKFD_FORCE_BLOCK=128),
    _row((64, 0, 1, 0, 1), "c5_mlcp", RKFD_SPEC=0, RKFD_FORCE_BLOCK=64),
    _row((32, 0, 1, 0, 1), "c5_mlcp", RKFD_SPEC=0, RKFD_FORCE_BLOCK=32),
    _row((256, 0, 1, 0, 1), "box_mlcp", RKFD_SPEC=0, RKFD_FORCE_BLOCK=256),
    # generic rigid kernel, scratch in device memory: the biped's 291-double column (the default) and the Volume solver
    _row((64, 1, 1, 0, 1), "biped_rigid_mlcp"),
    _row((256, 1, 1, 0, 1), "c4_volume"),
]


def row_id(row):
    return "%d_%d_%d_%d_%d" % row.variant


def makefile_variants():
    """The VARIANTS of roki-fd_b200/csrc/Makefile as tuples."""
    src = open(os.path.join(CSRC, "Makefile")).read().replace("\\\n", " ")
    m = re.search(r"^VARIANTS\s*:=(.*)$", src, re.M)
    return [tuple(int(x) for x in v.split("_")) for v in m.group(1).split()]


def engine_variants():
    """RKFD_VARIANT_LIST of rkfd_engine.cu as tuples."""
    src = open(os.path.join(CSRC, "rkfd_engine.cu")).read().replace("\\\n", " ")
    m = re.search(r"#define RKFD_VARIANT_LIST\(X\)(.*)", src)
    return [tuple(int(x) for x in g.split(",")) for g in re.findall(r"X\(([\d,\s]+)\)", m.group(1))]


def spec_table_ids():
    """Specialisation ids of RKFD_SPEC_TABLE, RKFD_SPEC_ROLLED_TABLE (rkfd_core.cuh) and the generic tensor-memory kernel."""
    src = open(os.path.join(CSRC, "rkfd_core.cuh")).read()
    ids = []
    for name in ("RKFD_SPEC_TABLE", "RKFD_SPEC_ROLLED_TABLE"):
        m = re.search(r"#define %s\(X\)(.*)" % name, src)
        ids += [int(g) for g in re.findall(r"X\((\d+),", m.group(1))]
    ids.append(int(re.search(r"SPEC_GENERIC_TM\s*=\s*(\d+)", src).group(1)))
    return ids
