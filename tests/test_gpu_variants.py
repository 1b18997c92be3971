"""Every compiled step-kernel variant on the B200 (-m gpu), one row of tests/variant_matrix.py each: the engine reports the
variant the row forces (rkFDBatchKernelVariant), the whole ragged batch agrees with a different variant of the generic
kernel, and its first 48 environments and those of its last, partial block agree with the oracle - under RKG, RK4, Euler and
Heun.  The tensor-memory variants also run the divergent slow paths of sincos against the generic kernel.  The worst errors
are printed per variant and integrator."""
import numpy as np
import pytest

import rokifd_b200  # noqa: F401
import variant_matrix as vm
from gpu_batch import capi  # noqa: F401

pytestmark = pytest.mark.gpu

INTEGRATORS = ["RKG", "RK4", "Euler", "Heun"]
NSTEPS, CHUNK = 25, 5
NORACLE = 48
# reference variants, tried in order until one differs from the row's: the generic kernel at its default choice, the generic
# kernel with its scratch in device memory, the generic kernel in shared memory only
REFERENCES = [{"RKFD_SPEC": "0"}, {"RKFD_SPEC": "0", "RKFD_FORCE_GSCR": "1", "RKFD_FORCE_BLOCK": "64"},
              {"RKFD_SPEC": "0", "RKFD_FORCE_SMEM": "1"}]


@pytest.fixture(scope="module")
def sms():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def relerr(a, b):
    a, b = np.asarray(a, float), np.asarray(b, float)
    return np.abs(a - b).max() / max(np.abs(b).max(), 1e-12) if a.size else 0.0


def env_relerr(a, b):
    return np.abs(a - b).max(1) / np.maximum(np.abs(b).max(1), 1e-12)


def batch_size(world, sms):
    """At least four CTAs per SM of the largest block among the world's rows, plus a partial block; the Vert and Volume worlds
    (a data-dependent rigid solve per environment) run the batches of test_gpu_parity.py."""
    if vm.WORLDS[world].cls in ("vert", "volume"):
        return 4096 + 37
    return sms * 4 * max(r.variant[0] for r in vm.MATRIX if r.world == world) + 37


def variants_of(fd):
    out, s = [], 0
    while True:
        try:
            out.append(fd.kernel_variant(s))
        except RuntimeError:
            return out
        s += 1


def run(capi, monkeypatch, w, q, qd, u, env, nsteps=NSTEPS, chunk=CHUNK):
    """Committing evaluation + nsteps steps (in launches of `chunk`) under the tuning variables env: reported variants,
    state, contacts and status after the evaluation and after the steps, environments in contact after each launch."""
    for k in vm.TUNING_VARS:
        monkeypatch.delenv(k, raising=False)
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    fd, _ = capi.create_world(w, B=q.shape[0])
    try:
        fd.batch_set_state(q, qd); fd.batch_set_motor_input(u); fd.update_init()
        out = {"variants": variants_of(fd)}

        def snap():
            s = [x.copy() for x in fd.batch_get_state()]
            a, t, r, f = fd.batch_get_contact()
            return {"q": s[0], "qd": s[1], "qdd": s[2], "a": a.astype(np.int8), "t": t.astype(np.int8), "r": r, "f": f,
                    "status": fd.batch_get_status()}
        out["init"] = snap()
        counts = [fd.batch_stats()[1]]
        for _ in range(nsteps // chunk):
            fd.update_n(chunk)
            counts.append(fd.batch_stats()[1])
        out["final"] = snap()
        out["counts"] = counts
    finally:
        fd.destroy()
    return out


_REF = {}


def reference(capi, monkeypatch, world, integ, k, q, qd, u):
    """Reference k of REFERENCES for (world, integrator), cached for the current world only (the C3 batch is large)."""
    if any(key[0] != world for key in _REF):
        _REF.clear()
    key = (world, integ, k)
    if key not in _REF:
        w = vm.WORLDS[world].make(); w.integrator = integ
        _REF[key] = run(capi, monkeypatch, w, q, qd, u, REFERENCES[k])
    return _REF[key]


def compare_batch(cls, got, ref, stage):
    """Whole batch: the row's variant against the reference variant.  Returns the worst errors for the report."""
    g, r = got[stage], ref[stage]
    fin = np.isfinite(r["q"]).all(1) & (np.abs(r["q"]).max(1) < 1e3) & np.isfinite(r["qd"]).all(1)
    assert fin.mean() > 0.9
    eq, eqd, eqdd = (relerr(g[k][fin], r[k][fin]) for k in ("q", "qd", "qdd"))
    same = (g["a"] == r["a"]).all(1)
    m = (g["a"] == 1) & (r["a"] == 1) & (same & fin)[:, None]          # forces and anchors: slots active in both runs
    fmax = max(np.abs(r["f"][m]).max(), 1.0) if m.any() else 1.0
    ef = np.abs(g["f"][m] - r["f"][m]).max() / fmax if m.any() else 0.0
    er = np.abs(g["r"][m] - r["r"][m]).max() if m.any() else 0.0
    assert (g["status"] == r["status"]).all()
    if cls == "penalty":
        # the same equations, products contracted differently by the compiler: agreement to rounding
        assert eq < 1e-11 and eqd < 1e-10 and eqdd < 1e-8, (stage, eq, eqd, eqdd)
        assert same.mean() >= 0.9999
        assert ef < 1e-8 and er < 1e-9, (stage, ef, er)
    elif cls == "mlcp":
        d = np.abs(g["q"][fin] - r["q"][fin]).max(1)
        if stage == "init":
            assert (g["a"] == r["a"]).all() and eqdd < 1e-9, eqdd
            assert ef < 1e-8 and er < 1e-9, (stage, ef, er)
        assert (d < 1e-8).mean() > 0.995, (stage, (d < 1e-8).mean())
    else:
        # Vert / Volume: KKT and QP systems of condition 1e5-1e7 amplify rounding (test_gpu_parity.py: Vert 99.9 % of the contact
        # environments within 1e-9 per evaluation; 97 % of the environments within 1e-6 after 20 steps)
        e = env_relerr(g["qdd" if stage == "init" else "q"][fin], r["qdd" if stage == "init" else "q"][fin])
        assert same.mean() >= 0.999
        assert (e < (1e-9 if stage == "init" else 1e-6)).mean() >= (0.999 if stage == "init" else 0.97), (stage, np.sort(e)[-5:])
    return eq, eqd, eqdd, ef


def compare_oracle(oracle, cls, w, q, qd, u, got, idx):
    """The checked environments against the oracle: q'' of the committing evaluation, the state after the steps."""
    oi = oracle.OracleWorld(w).batch_run(q[idx], qd[idx], u[idx], nsteps=0)[2]
    oq, oqd, _, _ = oracle.OracleWorld(w).batch_run(q[idx], qd[idx], u[idx], nsteps=NSTEPS)
    gi, gq, gqd = got["init"]["qdd"][idx], got["final"]["q"][idx], got["final"]["qd"][idx]
    ei = env_relerr(gi, oi)
    ofin = np.isfinite(oq).all(1) & (np.abs(oq).max(1) < 1e3)
    eq, eqd = env_relerr(gq[ofin], oq[ofin]), env_relerr(gqd[ofin], oqd[ofin])
    if cls == "penalty":
        assert ei.max() < 1e-9, ei.max()
        # test_kernel_variants_agree / test_integrator_menu: 1e-9 on q, 1e-8 on q' over the checked environments
        assert ofin.all() and relerr(gq, oq) < 1e-9 and relerr(gqd, oqd) < 1e-8, (relerr(gq, oq), relerr(gqd, oqd))
    elif cls == "volume":
        assert ei.max() < 1e-9, ei.max()
        assert (eq < 1e-6).mean() >= 0.97, np.sort(eq)[-5:]
    else:
        # rigid contact: a contact or friction mode decided at a zTOL-sized margin splits a trajectory (test_rigid_short_trajectory)
        assert (ei < 1e-9).mean() >= 0.97, np.sort(ei)[-5:]
        assert ofin.mean() > 0.9 and (eq < 1e-6).mean() >= 0.97, np.sort(eq)[-5:]
    return ei.max(), eq.max(), eqd.max()


ROWS = sorted(vm.MATRIX, key=lambda r: list(vm.WORLDS).index(r.world))


@pytest.mark.parametrize("integ", INTEGRATORS)
@pytest.mark.parametrize("row", ROWS, ids=vm.row_id)
def test_variant_matches_generic_kernel_and_oracle(capi, oracle, monkeypatch, sms, row, integ):
    W = vm.WORLDS[row.world]
    w = W.make(); w.integrator = integ
    B = batch_size(row.world, sms)
    q, qd, u = W.sample(w, B, 21)
    got = run(capi, monkeypatch, w, q, qd, u, row.env)
    assert got["variants"] and all(v == row.variant for v in got["variants"]), (got["variants"], row.variant)
    k = 0
    while True:
        ref = reference(capi, monkeypatch, row.world, integ, k, q, qd, u)
        if ref["variants"][0] != row.variant:
            break
        k += 1
    # every matrix world has cells: contacts in the committing evaluation and during the steps (rigid contacts push the cells
    # out within a few steps: some launch ends with contacts; penalty contacts: every launch)
    assert got["init"]["a"].sum() > 0 and got["counts"][0] > 0
    assert (min(got["counts"][1:]) if W.cls == "penalty" else max(got["counts"][1:])) > 0, got["counts"]
    bi = compare_batch(W.cls, got, ref, "init")
    bf = compare_batch(W.cls, got, ref, "final")
    block = row.variant[0]
    idx = np.r_[np.arange(NORACLE), np.arange(B - (B % block or block), B)]
    eo = compare_oracle(oracle, W.cls, w, q, qd, u, got, idx)
    print("variant %s on %s (%s, B=%d) vs %s: q'' %.1e after the evaluation; after %d steps q %.1e q' %.1e q'' %.1e f %.1e; "
          "oracle: q'' %.1e, q %.1e q' %.1e; envs in contact %s" % (
              vm.row_id(row), row.world, integ, B, "%d_%d_%d_%d_%d" % ref["variants"][0], bi[2], NSTEPS, *bf, *eo,
              [int(c) for c in got["counts"]]))


TM_ROWS = [r for r in ROWS if r.variant[3] >= 3]       # specialisations 3-11 keep their T space in tensor memory


@pytest.mark.parametrize("row", TM_ROWS, ids=vm.row_id)
def test_tensor_memory_variant_with_divergent_slow_paths(capi, monkeypatch, row):
    """test_divergent_slow_paths_keep_tensor_memory_accesses_converged for every tensor-memory variant: lanes of a warp take
    different branches around the warp-collective tensor-memory accesses (huge joint angles - the slow argument reduction
    of sincos - and velocities so large that the stage-to-stage angle addition falls back to sincos).  Same finite
    environments as the generic kernel, q' within 1e-9."""
    W = vm.WORLDS[row.world]
    w = W.make()
    B = 512
    q, qd, u = W.sample(w, B, 77)
    rng = np.random.default_rng(5)
    o = 6 if row.world in ("biped_penalty", "biped_rigid_mlcp", "c4_volume") else 0       # the joints, not the floating trunk
    big = rng.random(B) < 0.3
    q[big, o:] += rng.uniform(-3e6, 3e6, (big.sum(), w.nq - o))
    fast = rng.random(B) < 0.3
    qd[fast, o:] = rng.uniform(-400, 400, (fast.sum(), w.nq - o))
    got = run(capi, monkeypatch, w, q, qd, u, row.env, nsteps=3, chunk=3)
    ref = run(capi, monkeypatch, w, q, qd, u, REFERENCES[0], nsteps=3, chunk=3)
    assert got["variants"][0] == row.variant and ref["variants"][0] != row.variant
    fin = np.isfinite(ref["final"]["q"]).all(1) & np.isfinite(ref["final"]["qd"]).all(1)
    gfin = np.isfinite(got["final"]["q"]).all(1) & np.isfinite(got["final"]["qd"]).all(1)
    # C5 states whose cube starts deep in the rigid floor blow up in every kernel (|q'| 1e46 after 3 steps, on the host harness
    # too): compared are the environments whose velocities stay bounded
    ok = fin & (np.abs(ref["final"]["qd"]).max(1) < 1e3)
    e = relerr(got["final"]["qd"][ok], ref["final"]["qd"][ok])
    print("divergent slow paths, variant %s on %s: %d/%d finite, %d bounded, q' %.1e" % (vm.row_id(row), row.world, fin.sum(), B, ok.sum(), e))
    assert ok.mean() > 0.9 and (gfin == fin).all()
    assert e < 1e-9
