"""Tuning aid: step time of worlds with RIGID contact between two moving links (dense vertex solvers)."""
import sys, os, time; sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__)))); sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests"))
import numpy as np, rokifd_b200
from rokifd_b200 import capi, chains as ch
from workloads import mm_world, mm_states
B = int(sys.argv[1]) if len(sys.argv) > 1 else 32
for kind, solver in (("arm_pushes_box_rigid", "MLCP"), ("box_stack_rigid", "MLCP"), ("arm_pushes_box_rigid", "Vert"), ("box_stack_rigid", "Vert")):
    w = mm_world(kind, solver)
    q, qd, u = mm_states(kind, w, B, seed=3)
    fd, _ = capi.create_world(w, B=B); fd.batch_set_state(q, qd); fd.batch_set_motor_input(u); fd.update_init()
    for n in (10, 30, 20):
        t0 = time.time(); fd.update_n(n); fd.batch_sync(); dt = time.time() - t0
        a = fd.batch_get_contact()[0]
        print("%s %s B=%d: %d steps %.3f s (%.2f ms/step), active slots per env %.2f max %d" % (kind, solver, B, n, dt, 1e3 * dt / n, a.sum(1).mean(), a.sum(1).max()), flush=True)
    fd.destroy()
