"""The step-kernel variant matrix (tests/variant_matrix.py) on the host: the compiled variant lists agree with the matrix, every
model specialisation id is covered by a world that matches it, and every specialisation steps like the generic core and
the oracle under each integrator of the menu (the kernel core compiled by the test-only harness tests/hostsim).  The
device half is tests/test_gpu_variants.py."""
import ctypes as C

import numpy as np
import pytest

import rokifd_b200  # noqa: F401
from hostsim_py import HostSim
import variant_matrix as vm

INTEGRATORS = ["RKG", "RK4", "Euler", "Heun"]


def relerr(a, b):
    a, b = np.asarray(a, float), np.asarray(b, float)
    return np.abs(a - b).max() / max(np.abs(b).max(), 1e-12)


def test_variant_lists_agree_with_the_matrix():
    """The Makefile compiles, the engine lists and the matrix tests the same 30 variants, each exactly once: a variant added
    to the build without a matrix row fails here."""
    mk, eng = vm.makefile_variants(), vm.engine_variants()
    rows = [r.variant for r in vm.MATRIX]
    assert len(mk) == len(set(mk)) and len(eng) == len(set(eng)) and len(rows) == len(set(rows))
    assert set(mk) == set(eng) == set(rows)
    assert len(rows) == 30
    for r in vm.MATRIX:
        assert r.world in vm.WORLDS and set(r.env) <= set(vm.TUNING_VARS), r


SPEC_IDS = sorted(set(vm.spec_table_ids()))


def spec_world(sid):
    """The world of the first matrix row that runs specialisation `sid`."""
    return next(r.world for r in vm.MATRIX if r.variant[3] == sid)


def test_every_specialisation_id_is_covered():
    assert SPEC_IDS == list(range(1, 12))
    for sid in SPEC_IDS:
        w = vm.WORLDS[spec_world(sid)].make()
        # HostSim(spec=id) refuses a model that the specialisation does not match (the engine would fall back to the generic kernel)
        hs = HostSim(w, 1, spec=sid)
        assert sid == 11 or hs.spec_mask >> sid & 1, sid
    for r in vm.MATRIX:
        if r.variant[3] > 0:
            assert r.env.get("RKFD_SPEC", str(r.variant[3])) == str(r.variant[3]), r


def host_run(w, q, qd, u, spec, nsteps):
    """Committing evaluation, nsteps steps one at a time (contact-vertex count after each), then one non-committing
    evaluation: (q, q', q'' after the steps, q'' of the last evaluation, contact flags, pivots, active vertices per
    environment after the evaluation and after every step)."""
    hs = HostSim(w, q.shape[0], spec=spec or None)
    hs.set_state(q, qd, u)
    hs.eval(ref=True)
    counts = [hs.get_contact()[0].sum(1)]
    for _ in range(nsteps):
        hs.step(1)
        counts.append(hs.get_contact()[0].sum(1))
    sq, sqd, sqdd = (x.copy() for x in hs.get_state())
    a = hs.get_contact()[0].copy()
    piv = hs.get_pivot()[0].copy()
    hs.eval(ref=False)
    return sq, sqd, sqdd, hs.get_state()[2].copy(), a, piv, np.array(counts)


def oracle_run(oracle, w, q, qd, u, nsteps):
    ow = oracle.OracleWorld(w)
    out = []
    for b in range(q.shape[0]):
        e = ow.env(); e.set_state(q[b], qd[b]); e.set_motor_input(u[b]); e.update_init()
        for _ in range(nsteps):
            e.update()
        oq, oqd, oqdd = e.get_state()
        out.append((oq, oqd, oqdd, e.eval(False)))
    return [np.array(x) for x in zip(*out)]


@pytest.mark.parametrize("integ", INTEGRATORS)
@pytest.mark.parametrize("sid", SPEC_IDS)
def test_specialisation_under_each_integrator(oracle, sid, integ):
    """Each specialisation on its matrix world under RKG, RK4, Euler and Heun (the fused outward walk changes its stage
    sequence with the number of stages): a committing evaluation, 15 steps and a non-committing evaluation, bit-identical to
    the generic core (spec 7 - the rigid contact solve in the wrench space of the last link - within 1e-12), and against
    the oracle within 1e-9 on q and q'', 1e-8 on q'.  Worlds with cells are in contact at the committing
    evaluation and during the steps (penalty contact: after every step)."""
    name = spec_world(sid)
    W = vm.WORLDS[name]
    w = W.make()
    w.integrator = integ
    B, nsteps = (400 if W.cls == "mlcp" else 24), 15     # C5: about 7 % of the states start in contact
    q, qd, u = W.sample(w, B, 31)
    nq = w.nq
    gen = host_run(w, q, qd, u, 0, nsteps)
    spc = host_run(w, q, qd, u, sid, nsteps)
    fin = np.isfinite(gen[0]).all(1) & (np.abs(gen[0]).max(1) < 1e3)     # C5: a cube that starts deep in the floor blows up
    assert fin.mean() >= 0.97
    counts = gen[6][:, fin].sum(1)
    if w.nslot:       # rigid contacts push the cells out within a few steps; penalty contacts last
        live = counts > 0
        assert live[0] and live[1:].any() and (W.cls == "mlcp" or live.all()), (name, counts)
        assert (spc[6][:, fin] == gen[6][:, fin]).all()
    if sid == 7:
        for x, y in zip(spc[:4], gen[:4]):
            assert relerr(x[fin], y[fin]) < 1e-12
        assert (spc[4][fin] == gen[4][fin]).all()
    else:
        for x, y in zip(spc[:6], gen[:6]):
            assert np.array_equal(x, y)
    oq, oqd, oqdd, oqdd_eval = oracle_run(oracle, w, q, qd, u, nsteps)
    err = np.array([[relerr(spc[0][b, :nq], oq[b]), relerr(spc[1][b, :nq], oqd[b]), relerr(spc[2][b, :nq], oqdd[b]), relerr(spc[3][b, :nq], oqdd_eval[b])]
                    for b in np.where(fin)[0]])
    ok = (err < [1e-9, 1e-8, 1e-9, 1e-9]).all(1)
    print("spec %d on %s, %s: %d/%d envs within tolerance of the oracle, worst rel err q %.1e q' %.1e q'' %.1e q'' (eval) %.1e; "
          "active contact vertices %s" % (sid, name, integ, ok.sum(), len(ok), *err.max(0), counts.tolist()))
    # rigid contact: a contact or friction mode decided at a zTOL-sized margin splits a trajectory (as in test_kernel_core_host)
    assert ok.mean() >= (0.97 if W.cls == "mlcp" else 1.0)


def test_kernel_variant_query_without_an_engine_is_refused():
    """rkFDBatchKernelVariant before rkFDUpdateInit (and on no simulator at all) returns an error, writes nothing."""
    from rokifd_b200 import capi
    from rokifd_b200 import chains as ch
    L = capi.lib()
    fd = capi.RkFD()
    fd.chain_reg(ch.arm7())
    v = (C.c_int * 5)(-7, -7, -7, -7, -7)
    assert L.rkFDBatchKernelVariant(fd.h, 0, v) != 0
    assert "rkFDUpdateInit" in fd.last_error() and list(v) == [-7] * 5
    with pytest.raises(RuntimeError, match="rkFDUpdateInit"):
        fd.kernel_variant()
    assert L.rkFDBatchKernelVariant(None, 0, v) != 0 and list(v) == [-7] * 5
    fd.destroy()
