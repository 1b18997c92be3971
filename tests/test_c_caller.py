"""A plain C program written against include/roki_fd/rkfd_b200.h in the style of the reference's example callers
(reference example/chain/boxdrop_test.c): it must compile as C99 with gcc, link against librokifd_b200.so only, and -
on a GPU box - reproduce the oracle's trajectory of the same world for each of the three solver plugins."""
import os
import subprocess

import numpy as np
import pytest

import rokifd_b200  # noqa: F401
from rokifd_b200 import chains as ch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.path.join(ROOT, "tests", "c_callers", "boxdrop.c")
LIBDIR = os.path.join(ROOT, "roki-fd_b200")
GOLD = os.path.join(ROOT, "tests", "golden")


def build(tmp_path):
    exe = str(tmp_path / "boxdrop")
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Wextra", "-Werror", "-I" + os.path.join(ROOT, "include"), SRC,
                           "-L" + LIBDIR, "-lrokifd_b200", "-Wl,-rpath," + LIBDIR, "-o", exe])
    return exe


def test_c_caller_compiles_and_links_without_cuda_headers(tmp_path):
    exe = build(tmp_path)
    needed = subprocess.check_output(["readelf", "-d", exe], text=True)
    assert "librokifd_b200.so" in needed and "libcuda" not in needed and "libcudart" not in needed
    src = open(SRC).read()
    assert "cuda" not in src.lower().replace("no cuda in sight", "")


@pytest.mark.gpu
@pytest.mark.parametrize("solver,contacts,z0,cube", [("Volume", "-", 0.049, "cube.ztk"), ("Vert", "-", 0.049, "cube.ztk"),
                                                     ("MLCP", "contacts.ztk", 0.049, "cube.ztk"),
                                                     ("Volume", "-", 0.049, "cube_poly.ztk")])     # polyhedron-described box
def test_c_caller_matches_oracle(tmp_path, oracle, solver, contacts, z0, cube):
    exe = build(tmp_path)
    nsteps = 60
    args = [exe, os.path.join(GOLD, cube), os.path.join(GOLD, "rigidfloor.ztk"),
            "-" if contacts == "-" else os.path.join(GOLD, contacts), solver, str(nsteps), repr(z0)]
    out = subprocess.check_output(args, text=True)
    final = [l for l in out.splitlines() if l.startswith("final:")][0].split()
    got = np.array([float(x) for x in final[1:7]])
    t = float(final[7].split("=")[1])
    assert abs(t - nsteps * 0.001) < 1e-12
    ci = [] if contacts == "-" else [ch.ContactInfo("soft", "body", "elastic", E=1000.0, V=10.0, SF=0.5, KF=0.3),
                                     ch.ContactInfo("ground", "body", "rigid", K=1000.0, L=0.0001, SF=0.6, KF=0.4)]
    w = ch.World(chains=[ch.box(), ch.floor()], contact_info=ci, solver=solver)
    e = oracle.OracleWorld(w).env()
    q = np.zeros(6); q[2] = z0; q[3] = 0.05; q[4] = 0.02
    qd = np.zeros(6); qd[0] = 0.3
    e.set_state(q, qd); e.set_motor_input(np.zeros(w.nl)); e.update_init()
    for _ in range(nsteps):
        e.update()
    ref = e.get_state()[0]
    assert np.abs(got - ref).max() < 1e-9 * max(1.0, np.abs(ref).max()), (got, ref)


# ---- the reference's own example programs, compiled UNMODIFIED ---------------------------------------------------------
# they come from a source tree of the reference (mi-lib/roki-fd) that ROKIFD_REFERENCE names; the repository holds none of them
REF = os.environ.get("ROKIFD_REFERENCE", "")
REF_EX = os.path.join(REF, "example", "chain")
needs_reference = pytest.mark.skipif(not REF or not os.path.isdir(REF_EX), reason="no reference tree (set ROKIFD_REFERENCE)")
EXAMPLES = ["boxdrop_hardsoft_test", "boxdrop_test", "arm_box_test", "arm_box_trq_test", "arm_wall_test"]


def build_reference_example(name, outdir):
    exe = os.path.join(str(outdir), name)
    subprocess.check_call(["gcc", "-std=gnu99", "-I" + os.path.join(ROOT, "include"), os.path.join(REF_EX, name + ".c"),
                           "-L" + LIBDIR, "-lrokifd_b200", "-Wl,-rpath," + LIBDIR, "-o", exe])
    return exe


@needs_reference
@pytest.mark.parametrize("name", EXAMPLES)
def test_reference_examples_compile_unmodified(tmp_path, name):
    """example/chain/*.c of the reference, straight from its tree (nothing is copied into the repo), against
    include/roki_fd/roki_fd.h and librokifd_b200.so: every type, macro and function they touch exists (rkFD by value,
    rkFDSetSolver / rkFDODE2Assign* macros, rkChain / rkJoint accessors, zVec, zRandF, eprintf, zVecFPrint ...)."""
    exe = build_reference_example(name, tmp_path)
    needed = subprocess.check_output(["readelf", "-d", exe], text=True)
    assert "librokifd_b200.so" in needed and "libcuda" not in needed


def _splitmix(seed):
    s = seed
    while True:
        s = (s + 0x9E3779B97F4A7C15) & 0xFFFFFFFFFFFFFFFF
        z = s
        z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & 0xFFFFFFFFFFFFFFFF
        z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & 0xFFFFFFFFFFFFFFFF
        yield ((z ^ (z >> 31)) >> 11) / 9007199254740992.0


@pytest.mark.gpu
@needs_reference
def test_reference_boxdrop_hardsoft_runs_unmodified(tmp_path, oracle):
    """The reference's example/chain/boxdrop_hardsoft_test.c (compiled unmodified as in the test above) dropping ONE box
    (argv[1] = 1) on the hard/soft floor under the Volume solver: it opens ../model/{contactinfo,box,floor_hardsoft}.ztk
    (stand-ins with the reference's constants under tests/c_callers/model), steps 5 s and prints the joint displacements
    every step; compared with the oracle."""
    import shutil
    exe = build_reference_example("boxdrop_hardsoft_test", tmp_path)
    shutil.copytree(os.path.join(ROOT, "tests", "c_callers", "model"), tmp_path / "model")
    cwd = tmp_path / "chain"
    cwd.mkdir()
    seed = 12345
    subprocess.run([exe, "1"], cwd=cwd, env=dict(os.environ, ROKIFD_ZRAND_SEED=str(seed)), check=True,
                   stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL, timeout=600)
    rows = [l.split() for l in open(os.path.join(cwd, "1.zvs"))]
    traj = np.array([[float(x) for x in r[3:9]] for r in rows])           # "dt size ( q0 .. q5 )"
    assert traj.shape == (5000, 6) and all(r[1] == "6" for r in rows[:3])
    g = _splitmix(seed)
    q = np.zeros(6); q[2] = 0.1
    for k in (3, 4, 5):
        q[k] = np.deg2rad(-90.0 + 180.0 * next(g))
    w = ch.World(chains=[ch.ChainModel("box", [ch.Link(name="link#00", jtype="float", mass=0.5, stuff="body", inertia=np.eye(3) * 8.33e-4,
                                                       boxes=[((0.0, 0.0, 0.0), 0.1, 0.1, 0.1)])]), ch.floor_hardsoft()],
                 contact_info=[ch.ContactInfo("ground", "body", "rigid", K=1000.0, L=0.0001), ch.ContactInfo("body", "body", "rigid", K=1000.0, L=0.05),
                               ch.ContactInfo("soft", "body", "elastic", E=100.0, V=1.0)], solver="Volume")
    e = oracle.OracleWorld(w).env()
    e.set_state(q, np.zeros(6)); e.set_motor_input(np.zeros(w.nl)); e.update_init()
    ref = []
    for _ in range(600):
        e.update(); ref.append(e.get_state()[0].copy())
    ref = np.array(ref)
    err = np.abs(traj[:600] - ref).max(1)
    print("boxdrop_hardsoft_test: max |q - q_oracle| over the first 100 / 300 / 600 steps: %.2e / %.2e / %.2e (printed with 10 digits)" % (
        err[:100].max(), err[:300].max(), err.max()))
    assert err[:300].max() < 1e-8
    assert np.isfinite(traj).all() and abs(traj[-1, 2]) < 0.2          # after 5 s the box lies on the floor
