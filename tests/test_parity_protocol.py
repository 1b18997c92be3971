"""The parity protocol of SURVEY.md section 8(d) as `-m gpu` tests (round 1 kept it in a script the driver never ran): per world
4,096 synthetic environments (seed 20260418), the CUDA path through the C-ABI against the CPU oracle,
  per evaluation  - the committing evaluation of rkFDUpdateInit: q'' per environment, ||dq''||_inf / max(||q''_ref||_inf, 1e-12),
                    contact forces likewise (active slots), contact / friction / pivot flags;
  free running    - 100 x rkFDUpdate: q per environment, contact / friction / pivot flags.
Thresholds = the maxima measured on the B200 (profiles/r02_parity_report.md) x 10, never looser than north_star's 1e-9 per
evaluation; the share of environments that may split after a contact-mode flip at a zTOL-sized margin is stated per world.
Every run prints its row of the report and appends it to the file RKFD_PARITY_REPORT names, if set."""
import os
import time

import numpy as np
import pytest

import rokifd_b200  # noqa: F401
from rokifd_b200 import chains as ch

pytestmark = pytest.mark.gpu
B, H = 4096, 100


def rel(a, b):
    a = a.reshape(a.shape[0], -1); b = b.reshape(b.shape[0], -1)
    return np.abs(a - b).max(1) / np.maximum(np.abs(b).max(1), 1e-12)


def _c1():
    w = ch.World(chains=[ch.box(), ch.floor_soft()], contact_info=[ch.ContactInfo("soft", "body", "elastic", E=100.0, V=1.0, SF=0.5, KF=0.3)])
    q, qd, u = ch.sample_state(w, B, seed=20260418)
    q[:, 2] = np.linspace(0.0, 0.3, B); q[:, 3:6] *= 0.3
    return w, q, qd, u


def _std(w):
    return (w,) + tuple(ch.sample_state(w, B, seed=20260418))


def _c4():
    w = ch.world_c4_volume()
    return (w,) + tuple(ch.sample_c4_standing(w, B, seed=20260418))


def _flat(name, soft, solver=None):
    from test_kernel_core_host import flat_world, flat_states
    w, q0 = flat_world(name, solver=solver, soft=soft)
    return (w,) + tuple(flat_states(name, w, q0, B, seed=20260418))


def _mm(kind, solver="Vert"):
    from test_kernel_core_host import mm_world, mm_states
    w = mm_world(kind, solver)
    return (w,) + tuple(mm_states(kind, w, B, seed=20260418))


# world -> (builder, q'' tolerance per evaluation, q tolerance after H steps, share of environments that must meet it)
WORLDS = {
    "C1 box on the soft floor (penalty)": (_c1, 1e-9, 1e-6, 1.0),
    "C2 arm7, no contact": (lambda: _std(ch.world_c2()), 1e-9, 1e-8, 1.0),
    "C3 arm7 + penalty contact + joint friction": (lambda: _std(ch.world_c3(base_z=0.3)), 1e-9, 1e-6, 1.0),
    "C4 legged tree + volume contact": (_c4, 1e-9, 1e-6, 0.995),
    "C4 mighty.ztk (25 links, 701 vertices) + volume contact": (lambda: _flat("mighty_on_floor", False, "Volume"), 1e-9, 1e-6, 0.98),
    "mighty.ztk + penalty contact": (lambda: _flat("mighty_on_floor", True), 1e-9, 1e-6, 1.0),
    "C5 arm7 + rigid floor, MLCP": (lambda: _std(ch.world_c5(base_z=0.3, solver="MLCP")), 1e-9, 1e-6, 1.0),
    "C5 arm7 + rigid floor, Vert QP (relaxation 1e-4)": (lambda: _std(ch.world_c5(base_z=0.3, solver="Vert")), 1e-9, 1e-6, 0.999),
    "arm7 + rigid floor, Vert QP (solver default contact info)": (lambda: _std(ch.World(chains=[ch.arm7(base_z=0.3, contact_cube=True), ch.floor()], solver="Vert")), 1e-9, 1e-6, 1.0),
    "three boxes landing on each other (moving-vs-moving, penalty)": (lambda: _mm("box_stack"), 1e-9, 1e-6, 1.0),
    "arm pushes a free box (moving-vs-moving, penalty)": (lambda: _mm("arm_pushes_box"), 1e-9, 1e-6, 1.0),
    "arm pushes a free box (moving-vs-moving, RIGID pair, MLCP)": (lambda: _mm("arm_pushes_box_rigid", "MLCP"), 1e-9, 1e-6, 0.9),
}


@pytest.mark.parametrize("name", list(WORLDS))
def test_parity_protocol(name, oracle):
    from rokifd_b200 import capi
    assert capi.device_count() > 0
    mk, tol0, tolH, share = WORLDS[name]
    w, q, qd, u = mk()
    t0 = time.time()
    ow = oracle.OracleWorld(w)
    o0 = ow.batch_run_state(q, qd, u, nsteps=0)
    oH = ow.batch_run_state(q, qd, u, nsteps=H)
    tor = time.time() - t0
    fd, _ = capi.create_world(w, B=B); fd.batch_set_state(q, qd); fd.batch_set_motor_input(u); fd.update_init()
    _, _, gqdd = fd.batch_get_state()
    ns = w.nslot
    a0, t0_, _, f0 = fd.batch_get_contact() if ns else (np.zeros((B, 1), int),) * 4
    p0 = fd.batch_get_pivot()[0]
    fd.update_n(H)
    gq, gqd, _ = fd.batch_get_state()
    aH, tH, _, _ = fd.batch_get_contact() if ns else (np.zeros((B, 1), int),) * 4
    pH = fd.batch_get_pivot()[0]
    bad = int((fd.batch_get_status() != 0).sum())
    fd.destroy()
    e0 = rel(gqdd, o0[2])
    volume = w.solver == "Volume" and (not w.contact_info or any(ci.type == "rigid" for ci in w.contact_info))   # pair-level friction types
    efmax = None
    if ns and not volume:
        m = (o0[3] > 0)[:, :, None]
        efmax = rel(f0 * m, o0[5] * m).max()
    if ns:
        tm0 = (t0_ == o0[4]) | (o0[3] == 0) if not volume else np.ones_like(a0, bool)
        tmH = (tH == oH[4]) | (oH[3] == 0) if not volume else np.ones_like(aH, bool)
        fl0 = ((a0 == o0[3]).all(1) & tm0.all(1) & (p0 == o0[6]).all(1)).mean()
        flH = ((aH == oH[3]).all(1) & tmH.all(1) & (pH == oH[6]).all(1)).mean()
        c0 = (o0[3].sum(1) > 0).mean()
    else:
        fl0 = (p0 == o0[6]).all(1).mean(); flH = (pH == oH[6]).all(1).mean(); c0 = 0.0
    fin = np.isfinite(oH[0]).all(1) & (np.abs(oH[0]).max(1) < 1e6)
    eH = rel(gq[fin], oH[0][fin])
    row = "| %s | %d | %.1f %% | %.1e / %.1e / %.2f %% | %s | %.2f %% | %.1e / %.1e / %.2f %% (%d diverged in the oracle too, %d flagged) | %.2f %% | %.0f |" % (
        name, B, 100 * c0, e0.max(), np.quantile(e0, 0.999), 100 * (e0 < tol0).mean(), "-" if efmax is None else "%.1e" % efmax, 100 * fl0,
        eH.max(), np.quantile(eH, 0.99), 100 * (eH < tolH).mean(), int((~fin).sum()), bad, 100 * flH, tor)
    print(row)
    if os.environ.get("RKFD_PARITY_REPORT"):
        with open(os.environ["RKFD_PARITY_REPORT"], "a") as f:
            f.write(row + "\n")
    assert (e0 < tol0).mean() >= share and fl0 >= share, (e0.max(), fl0)
    if efmax is not None:
        assert efmax < 1e-8
    assert (eH < tolH).mean() >= share - 0.005 and flH >= share - 0.01 and bad == 0, (eH.max(), flH, bad)
