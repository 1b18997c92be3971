"""Measurement: cost of an environment reset (rkFDBatchResetEnvs, rkFDBatchResetEnvsDevice) on settled C3 with 262,144
environments, next to the step time.  CUDA events on the engine's stream (rkFDBatchSetStream); every list length is run once
before timing (the first call allocates the reset's sub-state).  The host variant is also timed with the host clock: it is
synchronous and includes the host-side split of the list and the copies of the states.

    python tools/exp_reset.py [--reps 20] [--settle 700]
"""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

import rokifd_b200  # noqa: E402,F401
from rokifd_b200 import capi, chains as ch  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--B", type=int, default=262144)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--settle", type=int, default=700)
    ap.add_argument("--steps", type=int, default=100)
    args = ap.parse_args()
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True).stdout.strip()
    w, B = ch.world_c3(), args.B
    q, qd, u = ch.sample_state(w, B, seed=20260418)
    fd, _ = capi.create_world(w, B=B)
    fd.batch_set_state(q, qd); fd.batch_set_motor_input(u); fd.update_init()
    st = torch.cuda.current_stream(); fd.batch_set_stream(st.cuda_stream)
    fd.update_n(args.settle)
    for _ in range(20):
        fd.update()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record(st)
    for _ in range(args.steps):
        fd.update()
    e1.record(st); torch.cuda.synchronize()
    step_ms = e0.elapsed_time(e1) / args.steps
    out = {"gpu": gpu, "B": B, "settle": args.settle, "step_ms": step_ms, "resets": []}
    print("%s: C3, %d envs, settled %d steps: %.4f ms per step" % (gpu, B, args.settle, step_ms), flush=True)
    rng = np.random.default_rng(1)
    nq_, nqd_, nu_ = ch.sample_state(w, 26214, seed=7)
    for n in (262, 2621, 26214):
        envs = rng.permutation(B)[:n].astype(np.int32)
        a, b, c = nq_[:n].copy(), nqd_[:n].copy(), nu_[:n].copy()
        fd.batch_reset_envs(envs, a, b, c)                       # allocation
        torch.cuda.synchronize()
        t0 = time.perf_counter(); e0.record(st)
        for _ in range(args.reps):
            fd.batch_reset_envs(envs, a, b, c)
        e1.record(st); torch.cuda.synchronize(); t1 = time.perf_counter()
        host_ms, host_ev = (t1 - t0) * 1e3 / args.reps, e0.elapsed_time(e1) / args.reps
        # the device variant: ids and states already on the GPU, nothing waits for the host
        te = torch.from_numpy(envs).cuda()
        tq, tqd, tu = [torch.from_numpy(x).cuda() for x in (a, b, c)]
        torch.cuda.synchronize()
        fd.batch_reset_envs_device(0, n, te.data_ptr(), tq.data_ptr(), tqd.data_ptr(), tu.data_ptr())
        e0.record(st)
        for _ in range(args.reps):
            fd.batch_reset_envs_device(0, n, te.data_ptr(), tq.data_ptr(), tqd.data_ptr(), tu.data_ptr())
        e1.record(st); torch.cuda.synchronize()
        dev_ms = e0.elapsed_time(e1) / args.reps
        r = {"n": n, "host_call_ms": host_ms, "host_events_ms": host_ev, "device_ms": dev_ms}
        out["resets"].append(r)
        print("reset %6d envs: host variant %.4f ms per call (host clock; %.4f ms between events), device variant %.4f ms "
              "(%.2f / %.2f steps)" % (n, host_ms, host_ev, dev_ms, host_ms / step_ms, dev_ms / step_ms), flush=True)
    # steps after the resets run at the settled rate again (the reset environments are in their first steps)
    torch.cuda.synchronize(); e0.record(st)
    for _ in range(args.steps):
        fd.update()
    e1.record(st); torch.cuda.synchronize()
    out["step_ms_after"] = e0.elapsed_time(e1) / args.steps
    print("steps after the resets: %.4f ms per step" % out["step_ms_after"])
    print(json.dumps(out))
    fd.destroy()


if __name__ == "__main__":
    main()
