"""Host-side tests of the C-ABI library that need no GPU: the library loads, exports every symbol
include/roki_fd/rkfd_b200.h declares, mirrors the reference's registration bookkeeping, reads ZTK
files, and fails loudly (no CPU fallback) when no device exists."""
import ctypes as C
import os
import re

import numpy as np
import pytest

import rokifd_b200  # noqa: F401
from rokifd_b200 import capi, chains as ch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")
# a source tree of the reference (mi-lib/roki-fd), when ROKIFD_REFERENCE names one: the tests that read its own files run then
REF = os.environ.get("ROKIFD_REFERENCE", "")
REF_MODELS = os.path.join(REF, "example", "model")
needs_reference = pytest.mark.skipif(not REF or not os.path.isdir(REF_MODELS), reason="no reference tree (set ROKIFD_REFERENCE)")


def test_library_exports_every_declared_symbol():
    hdr = open(os.path.join(ROOT, "include", "roki_fd", "rkfd_b200.h")).read()
    hdr = "\n".join(l for l in hdr.splitlines() if not l.lstrip().startswith("#"))
    names = re.findall(r"__ROKI_FD_EXPORT\s+[^;(]*?\b(\w+)\s*\(", hdr)
    assert len(names) > 80
    L = C.CDLL(capi.LIB_PATH)
    missing = [n for n in names if not hasattr(L, n)]
    assert not missing, missing


def test_registration_bookkeeping():
    """fd->size, cell offsets and state windows after Reg / Unreg (reference rkfd_sim.c:79-155, 188-255)."""
    fd = capi.RkFD()
    c_arm = fd.chain_reg(ch.arm_2dof())
    c_box = fd.chain_reg(ch.box())
    c_flr = fd.chain_reg(ch.floor())
    assert fd.size == 2 + 6 and fd.link_num == 3 + 1
    fd.chain_set_dis(c_arm, [0.1, 0.2])
    fd.chain_set_dis(c_box, [1, 2, 3, 4, 5, 6])
    fd.chain_set_vel(c_box, [6, 5, 4, 3, 2, 1])
    assert np.allclose(fd.dis, [0.1, 0.2, 1, 2, 3, 4, 5, 6])
    assert np.allclose(fd.vel, [0, 0, 6, 5, 4, 3, 2, 1])
    assert fd.chain_unreg(c_arm)
    assert fd.size == 6 and np.allclose(fd.dis, [1, 2, 3, 4, 5, 6])     # state of the remaining chains is kept
    assert not fd.chain_unreg(capi.RkFDCell(c_flr.h + 8))                # unknown handle -> false
    fd.destroy()


def test_defaults_and_solver_table():
    """rkFDCreate defaults (rkfd_property.c:10-18) and the per-solver default contact info."""
    L = capi.lib()
    fd = capi.RkFD()

    class Prp(C.Structure):
        _fields_ = [("dt", C.c_double), ("pyramid", C.c_int), ("fw", C.c_double), ("max_iter", C.c_int), ("vel_eps", C.c_double)]

    class Head(C.Structure):
        _fields_ = [("t", C.c_double), ("prp", Prp)]

    h = C.cast(fd.h, C.POINTER(Head)).contents
    assert (h.t, h.prp.dt, h.prp.pyramid, h.prp.fw, h.prp.max_iter, h.prp.vel_eps) == (0.0, 0.001, 8, 100.0, 10, 1e-8)
    for s in ("Vert", "MLCP", "Volume"):
        fd.set_solver(s)
    fd.prp_set(dt=0.002, pyramid=6)
    h = C.cast(fd.h, C.POINTER(Head)).contents
    assert h.prp.dt == 0.002 and h.prp.pyramid == 6
    fd.destroy()


def test_no_cpu_fallback():
    if capi.device_count() > 0:
        pytest.skip("a GPU is present")
    fd, _ = capi.create_world(ch.world_c2(), B=4)
    with pytest.raises(RuntimeError, match="no CUDA device"):
        fd.update_init()
    # without an engine rkFDUpdate returns NULL, says so on every call and pushes the time to +inf, so that the reference
    # idiom `while( rkFDTime(&fd) < T ) rkFDUpdate(&fd);` ends instead of spinning on a time that never advances
    for _ in range(2):
        with pytest.raises(RuntimeError, match="no device engine"):
            fd.update()
    assert fd.time == float("inf")
    with pytest.raises(RuntimeError):
        fd.batch_get_state()
    fd.destroy()


def test_ztk_reader():
    c = capi.RkChain(ztk=os.path.join(GOLD, "arm2.ztk"))
    assert c.link_num == 3 and c.joint_size == 2
    L = capi.lib()
    v = L.zVecAlloc(2)
    L.rkChainGetJointDisAll.restype = C.c_void_p
    L.rkChainGetJointDisAll.argtypes = [C.c_void_p, C.c_void_p]
    L.rkChainGetJointDisAll(c.h, v)
    buf = C.cast(C.cast(v, C.POINTER(C.c_void_p))[1], C.POINTER(C.c_double))
    assert np.allclose([buf[0], buf[1]], np.deg2rad([30, -45]))
    L.zVecFree(v)
    c.destroy()
    with pytest.raises(RuntimeError):
        capi.RkChain(ztk=os.path.join(GOLD, "missing.ztk"))
    fd = capi.RkFD()
    assert fd.contact_info_scan_file(os.path.join(GOLD, "contacts.ztk"))
    assert not fd.contact_info_scan_file(os.path.join(GOLD, "missing.ztk"))
    assert fd.chain_reg_file(os.path.join(GOLD, "cube.ztk")) is not None
    assert fd.chain_reg_file(os.path.join(GOLD, "softfloor.ztk")) is not None
    assert fd.chain_reg_file(os.path.join(GOLD, "missing.ztk")) is None
    assert fd.size == 6
    assert np.allclose(fd.dis, [0.1, -0.2, 0.3] + list(np.deg2rad([10, 20, 30])))
    fd.destroy()


@needs_reference
def test_ztk_reader_on_reference_models():
    """The reader accepts the reference's own model files unmodified (SURVEY.md section 8f.1)."""
    d = REF_MODELS
    expect = {"box.ztk": (1, 6), "floor.ztk": (1, 0), "floor_hardsoft.ztk": (2, 0), "arm_2DoF.ztk": (3, 2),
              "arm_2DoF_trq.ztk": (3, 2), "puma.ztk": (7, 6), "mighty.ztk": (25, 26), "arm.ztk": (6, 12), "dualarm.ztk": (None, None),
              "wall.ztk": (4, 18), "crawler.ztk": (None, None), "box_small.ztk": (1, 6)}      # wall.ztk: three breakable float joints
    for f, (nl, nq) in expect.items():
        c = capi.RkChain(ztk=os.path.join(d, f))
        if nl is not None:
            assert (c.link_num, c.joint_size) == (nl, nq), f
        c.destroy()
    fd = capi.RkFD()
    assert fd.contact_info_scan_file(os.path.join(d, "contactinfo.ztk"))
    fd.destroy()


def test_world_errors_are_reported_before_the_device_is_needed():
    """rkFDUpdateInit checks the world (limits, cell shapes under the Volume solver) before it looks for a device: the
    message reaches the caller on any machine."""
    import numpy as np
    rng = np.random.default_rng(0)
    blob = ch.ChainModel("blob", [ch.Link(name="l", jtype="float", mass=1.0, stuff="body", inertia=np.eye(3) * 1e-2,
                                          shapes=[rng.normal(size=(8, 3)) * 0.1])])
    fd, _ = capi.create_world(ch.World(chains=[blob, ch.floor()], solver="Volume"), B=4)
    with pytest.raises(RuntimeError, match="Volume solver"):
        fd.update_init()
    fd.destroy()


def _flattened(fd):
    try:
        fd.update_init()          # flattens and checks the world, then looks for a device (none in the CPU container)
    except RuntimeError as e:
        assert "no CUDA device" in str(e), e
    return fd.describe_model()


def _same_model(ma, mb, keys=None):
    ma = {k: v for k, v in ma.items() if not k.startswith("init.")}      # the registered initial state is not part of the model
    mb = {k: v for k, v in mb.items() if not k.startswith("init.")}
    ks = set(ma) if keys is None else {k for k in ma if k.split("[")[0] in keys}
    assert (set(ma) == set(mb) or keys is not None) and len(ks) > 3
    for k in ks:
        assert len(ma[k]) == len(mb[k]), k
        assert np.allclose(ma[k], mb[k], rtol=1e-12, atol=1e-13), (k, ma[k], mb[k])


REF_WORLDS = {   # the reference's example programs: model files, solver
    "boxdrop_hardsoft": (["box.ztk", "floor_hardsoft.ztk"], "Vert"),          # example/chain/boxdrop_hardsoft_test.c
    "arm2dof_on_floor": (["arm_2DoF.ztk", "floor.ztk"], "MLCP"),
    "arm_box_floor": (["arm_2DoF.ztk", "box.ztk", "floor.ztk"], "Volume"),     # example/chain/arm_box_test.c
    "mighty_on_floor": (["mighty.ztk", "floor.ztk"], "Volume"),                # BASELINE config C4's model
    # the fake crawler (rkfd_sim.c:386-440): both tracks of crawler.ztk in slide mode, belt axis y, 0.3 m/s; over floor_hardsoft.ztk
    "crawler_on_hardsoft": (["crawler.ztk", "floor_hardsoft.ztk"], "Volume"),
}
REF_SLIDES = {"crawler_on_hardsoft": [(0, 1, 0, 0.3, (0.0, 1.0, 0.0)), (0, 2, 0, 0.3, (0.0, 1.0, 0.0))]}     # (chain, link, shape, speed, axis)


def reference_world_description(name):
    d = REF_MODELS
    files, solver = REF_WORLDS[name]
    fa = capi.RkFD()
    assert fa.contact_info_scan_file(os.path.join(d, "contactinfo.ztk"))
    cells = []
    for f in files:
        cells.append(fa.chain_reg_file(os.path.join(d, f)))
        assert cells[-1] is not None, f
    L = capi.lib()
    L.rkLinkShape.restype = C.c_void_p; L.rkLinkShape.argtypes = [C.c_void_p, C.c_int, C.c_int]
    for fn, at in (("rkFDShape3DSetSlideMode", C.c_bool), ("rkFDShape3DSetSlideVel", C.c_double), ("rkFDShape3DSetSlideAxis", C.POINTER(C.c_double))):
        getattr(L, fn).restype = C.c_void_p; getattr(L, fn).argtypes = [C.c_void_p, C.c_void_p, at]
    for (c, link, k, vel, axis) in REF_SLIDES.get(name, []):       # the reference's own calls on a shape of the registered chain
        sh = L.rkLinkShape(cells[c].chain_handle, link, k)
        assert sh and L.rkFDShape3DSetSlideMode(fa.h, sh, True) and L.rkFDShape3DSetSlideVel(fa.h, sh, vel) and L.rkFDShape3DSetSlideAxis(fa.h, sh, (C.c_double * 3)(*axis))
    fa.set_solver(solver)
    desc = _flattened(fa)
    fa.destroy()
    return desc


def flat_description(name):
    """tests/golden/flat_<name>.txt: the device model the reference's own files of world `name` flatten to (written by
    tests/golden/make_flat_models.py from a reference tree; checked against it by the test below when one is given)."""
    return ch.load_flat(os.path.join(GOLD, "flat_%s.txt" % name))


@pytest.mark.parametrize("name", list(REF_WORLDS))
def test_reference_model_files_flatten_and_round_trip(name):
    """The reference's own model files, registered through rkFDChainRegFile / rkFDContactInfoScanFile, flatten to a device
    model (mighty.ztk: 25 links, 26 DoF, 701 collision vertices on the floor) that `chains.world_from_flat` turns back
    into a World which flattens to the same tables: what the oracle and the parity tests step (tests/golden/flat_*.txt,
    written by tests/golden/make_flat_models.py from these files) IS what the C-ABI makes of the reference's files."""
    if name == "arm2dof_on_floor":
        pytest.skip("152 contact slots: the rigid vertex solvers take 32")
    desc = flat_description(name)
    if REF and os.path.isdir(REF_MODELS):
        _same_model(reference_world_description(name), desc)
    fb, _ = capi.create_world(ch.world_from_flat(desc), B=1)
    _same_model(desc, _flattened(fb))
    fb.destroy()


def test_reference_model_files_match_the_transcribed_worlds():
    """rokifd_b200.chains transcribes box.ztk / floor*.ztk / arm_2DoF.ztk / contactinfo.ztk by hand: the transcriptions
    flatten to the same tables as the files (tests/golden/flat_*.txt; arm_2DoF: the link tables of the arm in
    arm_box_floor, where it is registered first; its collision shapes are not transcribed)."""
    _same_model(flat_description("boxdrop_hardsoft"), _flattened(capi.create_world(ch.world_c1_box(), B=1)[0]))
    mb = _flattened(capi.create_world(ch.world_c1_serial(), B=1)[0])
    ma = {k: v for k, v in flat_description("arm_box_floor").items() if k in mb}
    for m in (ma, mb):
        for k in m:
            if k.startswith("link.topo"):
                m[k] = m[k][:5]            # parent, joint type, motor type, dofs, offset (not the cell range)
    assert all("link.mass[%d]" % i in ma for i in range(3))
    _same_model(ma, mb, keys={"link.topo", "link.Ro", "link.po", "link.mass", "link.joint"})


def test_ztk_shape_sugar_and_automatic_mass_properties():
    """loop / arc / prism polyhedra (puma.ztk:67-88), box axes, spheres, `COM: auto` / `inertia: auto` / `density:`
    (arm.ztk:79-80): vertices and mass properties of tests/golden/sugar.ztk against an independent evaluation (scipy's
    convex hull for the prism, closed forms for the primitives)."""
    from scipy.spatial import ConvexHull
    fd = capi.RkFD()
    cell = fd.chain_reg_file(os.path.join(GOLD, "sugar.ztk"))
    assert cell is not None
    capi.lib().rkCDPairChainUnreg(None, cell.chain_handle)      # as the reference's example programs do: the self pairs of the chain (rigid by default) are not wanted here
    m = _flattened(fd)
    fd.destroy()
    verts = np.array([m["vert[%d]" % i] for i in range(int(m["dims"][6]))])
    cells = [[int(v) for v in m["cell[%d]" % i]] for i in range(int(m["dims"][2]))]

    def link(i):
        mp = m["link.mass[%d]" % i]
        Io = np.array([[mp[4], mp[5], mp[6]], [mp[5], mp[7], mp[8]], [mp[6], mp[8], mp[9]]])
        c = np.array(mp[10:13])
        return mp[0], c, Io - mp[0] * (c @ c * np.eye(3) - np.outer(c, c))
    # --- the prism: 6 corners + 11 arc points per ring, two rings; convex, so the hull is the solid
    pv = verts[cells[0][1]:cells[0][1] + cells[0][2]]
    assert pv.shape[0] == 2 * (6 + 11) and np.allclose(sorted(set(np.round(pv[:, 2], 12))), [0.01, 0.05])
    arc = pv[1:12]
    assert np.allclose(np.hypot(arc[:, 0] - (-0.05 + np.sqrt(0.08 ** 2 - 0.06 ** 2)), arc[:, 1]), 0.08) and (arc[:, 0] < -0.05).all()
    hull = ConvexHull(pv)
    vol, vc, xx = 0.0, np.zeros(3), np.zeros((3, 3))
    o = pv.mean(0)
    for s in hull.simplices:                      # tetrahedra (o, a, b, c), 4-point degree-2 rule
        a, b, c = pv[s] - o
        v = abs(np.dot(a, np.cross(b, c))) / 6.0
        S = a + b + c
        vol += v; vc += v * 0.25 * S
        xx += v / 20.0 * (np.outer(a, a) + np.outer(b, b) + np.outer(c, c) + np.outer(S, S))
    assert abs(vol - hull.volume) < 1e-12
    com = o + vc / vol
    X = 2.0 / vol * xx - 2.0 * np.outer(vc / vol, vc / vol)      # density * second moments about the centroid
    mass, c, Ic = link(0)
    assert mass == 2.0 and np.allclose(c, com, atol=1e-12) and np.allclose(Ic, np.trace(X) * np.eye(3) - X, atol=1e-12)
    # --- the tilted box: corners on the rotated axes, inertia R diag R^T
    bv = verts[cells[1][1]:cells[1][1] + 8]
    R = np.array([[0.8, -0.6, 0], [0.6, 0.8, 0], [0, 0, 1.0]])
    loc = (bv - np.array([0.1, 0, 0.05])) @ R
    assert np.allclose(np.abs(loc), [0.1, 0.05, 0.03])
    mass, c, Ic = link(1)
    d = np.array([0.2, 0.1, 0.06])
    assert np.allclose(c, [0.1, 0, 0.05]) and np.allclose(Ic, R @ np.diag(1.5 / 12 * (d @ d - d * d)) @ R.T, atol=1e-14)
    # --- density: sphere + cone
    Vs, Vc = 4 / 3 * np.pi * 0.03 ** 3, np.pi * 0.02 ** 2 * 0.08 / 3
    mass, c, Ic = link(2)
    assert abs(mass - 1000 * (Vs + Vc)) < 1e-12
    cs, cc = np.array([0, 0.1, 0]), np.array([0, 0, 0.04])
    assert np.allclose(c, (Vs * cs + Vc * cc) / (Vs + Vc), atol=1e-14)
    Is = 1000 * Vs * 0.4 * 0.03 ** 2 * np.eye(3)
    Icn = 1000 * Vc * np.diag([3 / 80 * (4 * 0.02 ** 2 + 0.08 ** 2)] * 2 + [0.3 * 0.02 ** 2])
    tot = np.zeros((3, 3))
    for mi, ci, Ii in ((1000 * Vs, cs, Is), (1000 * Vc, cc, Icn)):
        r = ci - c
        tot += Ii + mi * (r @ r * np.eye(3) - np.outer(r, r))
    assert np.allclose(Ic, tot, atol=1e-14)


@needs_reference
def test_ztk_reader_fills_the_gaps_of_the_reference_models():
    """puma.ztk's loop/prism shapes give collision vertices, arm.ztk's `COM: auto` links get mass properties, no shape of
    the reference's model directory is dropped."""
    d = REF_MODELS
    fd = capi.RkFD(); assert fd.chain_reg_file(os.path.join(d, "puma.ztk")) is not None
    m = _flattened(fd); fd.destroy()
    assert int(m["dims"][2]) == 7 and int(m["dims"][6]) > 300           # 7 cells: base, post, shoulder, upperarm, forearm, hand ...
    fd = capi.RkFD(); assert fd.chain_reg_file(os.path.join(d, "arm.ztk")) is not None
    m = _flattened(fd); fd.destroy()
    Vs, Vc = 4 / 3 * np.pi * 0.02 ** 3, np.pi * 0.01 ** 2 * 0.11
    assert abs(m["link.mass[1]"][12] - Vc * 0.075 / (Vs + Vc)) < 1e-12 and m["link.mass[4]"][4] == pytest.approx(0.6 * 0.4 * 0.02 ** 2)


def test_volume_kernel_keeps_its_warp_barriers():
    """DESIGN.md section 3.1, "Reconvergence the compiler cannot delete": nvcc drops __syncwarp() / the sync of __any_sync at loop
    heads it takes for convergent, and lanes that skipped a divergent body then run ahead through the block barriers (seen on
    the B200 as a warp out-of-range address).  DevCtx::hsync()/hany() use a mask the compiler cannot evaluate; the SASS of the
    Volume variant must therefore hold the guarded warp barrier (active mask compared with the mask, divergent branch to a
    WARPSYNC) at the candidate loop and before the friction LPs.  Checked on the object file the build leaves in-tree."""
    import shutil, subprocess
    obj = os.path.join(os.path.dirname(capi.LIB_PATH), "csrc", "build", "rkfd_kernel_256_1_1_0_1.o")
    cuobjdump = shutil.which("cuobjdump") or shutil.which("cuobjdump", path=os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin"))
    if cuobjdump is None or not os.path.exists(obj):
        pytest.skip("no cuobjdump / no object file of the Volume variant")
    sass = subprocess.run([cuobjdump, "-sass", obj], capture_output=True, text=True, timeout=300).stdout
    assert sass.count("BRA.DIV") >= 3 and "WARPSYNC.EXCLUSIVE" in sass
    src = open(os.path.join(os.path.dirname(capi.LIB_PATH), "csrc", "rkfd_volume.cuh")).read()
    assert src.count("c.hsync()") >= 2 and "c.hany(ci < ncand)" in src
