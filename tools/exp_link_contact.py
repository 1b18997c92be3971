"""Measurement: cost of the link contact-wrench calls (rkFDBatchGetLinkContactWrench, rkFDBatchGetLinkContactWrenchDevice) next
to the step time, on three settled workloads: C3 (262,144 environments, tip link), C4 Volume (131,072, both soles) and C5 MLCP
(131,072, tip link).  CUDA events on the engine's stream (rkFDBatchSetStream), mean over --reps calls after one warm-up call
per case (the host variant allocates its device buffer on the first call).  The host variant is also timed with the host
clock: it is synchronous and includes the copy to pageable host memory.

The HBM bound is the least time for the minimal bytes: the q rows of the walked dofs, perm and the piv word read once, the cf
rows of the listed slots read once, each output double written once, at the 6,553 GB/s of DESIGN.md section 3.4.

    python tools/exp_link_contact.py [--reps 50] [--settle 700] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

import rokifd_b200  # noqa: E402,F401
from rokifd_b200 import capi, chains as ch  # noqa: E402

HBM_GBS = 6553.0


def walked_dofs(w, links):
    """dofs of the links the readout walks: the requested links with contact and their ancestors"""
    fl = w.flat_links()
    ndof = {"fixed": 0, "revolute": 1, "prismatic": 1, "cylindrical": 2, "hooke": 2, "spherical": 3, "float": 6, "breakablefloat": 6}
    need = set()
    for i in links:
        while i >= 0 and i not in need:
            need.add(i); i = fl[i].parent
    return sum(ndof[fl[i].jtype] for i in need)


def slots_of(w, links):
    """contact slots the readout reads on static-floor worlds: the cells of the links against every static box (the Volume
    solver reads the first three slots of a box pair)"""
    nbox = sum(len(l.boxes) for c in w.chains if c.is_static for l in c.links)
    n = 0
    for i in set(links):
        for v in w.flat_links()[i].cells():          # (nvert, 3)
            n += nbox * (3 if w.solver == "Volume" else len(v))
    return n


def case(label, w, B, sample, links, settle, reps, st, e0, e1):
    q, qd, u = sample(B)
    fd, _ = capi.create_world(w, B=B)
    fd.batch_set_state(q, qd); fd.batch_set_motor_input(u); fd.update_init()
    fd.batch_set_stream(st.cuda_stream)
    fd.update_n(settle)
    for _ in range(20):
        fd.update()
    torch.cuda.synchronize()
    e0.record(st)
    for _ in range(20):
        fd.update()
    e1.record(st); torch.cuda.synchronize()
    step_ms = e0.elapsed_time(e1) / 20
    n = len(links)
    tw = torch.empty((B, n, 6), dtype=torch.float64, device="cuda")
    fd.batch_get_link_contact_wrench_device(0, links, tw.data_ptr())
    torch.cuda.synchronize()
    e0.record(st)
    for _ in range(reps):
        fd.batch_get_link_contact_wrench_device(0, links, tw.data_ptr())
    e1.record(st); torch.cuda.synchronize()
    dev_ms = e0.elapsed_time(e1) / reps
    fd.batch_get_link_contact_wrench(links)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(reps):
        fd.batch_get_link_contact_wrench(links)
    host_ms = (time.perf_counter() - t0) * 1e3 / reps
    per_env = 8 * walked_dofs(w, links) + 4 + 4 + 8 * 3 * slots_of(w, links) + 8 * 6 * n
    bound_ms = per_env * B / (HBM_GBS * 1e9) * 1e3
    fd.destroy()
    r = {"case": label, "B": B, "links": links, "step_ms": step_ms, "device_ms": dev_ms, "share_of_step": dev_ms / step_ms,
         "bytes_per_env": per_env, "hbm_bound_ms": bound_ms, "share_of_bound": bound_ms / dev_ms, "host_call_ms": host_ms}
    print("%-12s %d envs: step %.4f ms; device call %.4f ms (%.1f %% of a step; HBM bound %.4f ms for %d B per env: %.0f %%); "
          "host variant %.3f ms per call" % (label, B, step_ms, dev_ms, 100 * dev_ms / step_ms, bound_ms, per_env,
                                             100 * bound_ms / dev_ms, host_ms), flush=True)
    return r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--settle", type=int, default=700)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert args.reps >= 50
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True).stdout.strip()
    print(gpu, flush=True)
    st = torch.cuda.current_stream()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    c3, c4, c5 = ch.world_c3(), ch.world_c4_volume(), ch.world_c5(base_z=0.3, solver="MLCP")
    cases = [("C3 tip", c3, 262144, lambda B: ch.sample_state(c3, B, seed=20260418), [c3.nl - 1]),
             ("C4 Volume soles", c4, 131072, lambda B: ch.sample_c4_standing(c4, B, seed=20260418), [3, 6]),
             ("C5 MLCP tip", c5, 131072, lambda B: ch.sample_state(c5, B, seed=20260418), [c5.nl - 1])]
    out = {"gpu": gpu, "settle": args.settle, "reps": args.reps, "hbm_GBs": HBM_GBS, "cases": []}
    for label, w, B, sample, links in cases:
        out["cases"].append(case(label, w, B, sample, links, args.settle, args.reps, st, e0, e1))
    print(json.dumps(out))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
