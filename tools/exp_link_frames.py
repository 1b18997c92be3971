"""Measurement: cost of the link kinematics calls (rkFDBatchGetLinkFrames, rkFDBatchGetLinkFramesDevice) on settled C3 with
262,144 environments, next to the step time.  CUDA events on the engine's stream (rkFDBatchSetStream), mean over --reps calls
after one warm-up call per case (the host variant allocates its device buffer on the first call).  The host variant is also
timed with the host clock: it is synchronous and includes the copies to pageable host memory.

The HBM bound is the least time for the minimal bytes: q and q' (nq rows) and perm read once, each output double written
once, at the 6,553 GB/s of DESIGN.md section 3.4.

    python tools/exp_link_frames.py [--reps 50] [--settle 700] [--out FILE]
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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--B", type=int, default=262144)
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--settle", type=int, default=700)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert args.reps >= 20
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
    out = {"gpu": gpu, "B": B, "settle": args.settle, "step_ms": step_ms, "hbm_GBs": HBM_GBS, "cases": []}
    print("%s: C3, %d envs, settled %d steps: %.4f ms per step" % (gpu, B, args.settle, step_ms), flush=True)
    nq, nl = w.nq, w.nl
    cases = [("tip, frames", [nl - 1], True, False), ("all links, frames", None, True, False),
             ("all links, frames + velocities", None, True, True)]
    for label, links, want_f, want_v in cases:
        n = nl if links is None else len(links)
        # the device variant: outputs in torch tensors on the engine's device
        tf = torch.empty((B, n, 12), dtype=torch.float64, device="cuda") if want_f else None
        tv = torch.empty((B, n, 6), dtype=torch.float64, device="cuda") if want_v else None
        pf, pv = (tf.data_ptr() if want_f else None), (tv.data_ptr() if want_v else None)
        fd.batch_get_link_frames_device(0, links, pf, pv)
        torch.cuda.synchronize()
        e0.record(st)
        for _ in range(args.reps):
            fd.batch_get_link_frames_device(0, links, pf, pv)
        e1.record(st); torch.cuda.synchronize()
        dev_ms = e0.elapsed_time(e1) / args.reps
        # the host variant
        fd.batch_get_link_frames(links, frames=want_f, vel=want_v)
        torch.cuda.synchronize()
        t0 = time.perf_counter(); e0.record(st)
        for _ in range(args.reps):
            fd.batch_get_link_frames(links, frames=want_f, vel=want_v)
        e1.record(st); torch.cuda.synchronize(); t1 = time.perf_counter()
        host_ms, host_ev = (t1 - t0) * 1e3 / args.reps, e0.elapsed_time(e1) / args.reps
        per_env = 2 * nq * 8 + 4 + n * ((12 if want_f else 0) + (6 if want_v else 0)) * 8
        bound_ms = per_env * B / (HBM_GBS * 1e9) * 1e3
        r = {"case": label, "nlink": n, "device_ms": dev_ms, "host_call_ms": host_ms, "host_events_ms": host_ev,
             "bytes_per_env": per_env, "total_MB": per_env * B / 1e6, "hbm_bound_ms": bound_ms, "share_of_bound": bound_ms / dev_ms}
        out["cases"].append(r)
        print("%-32s device %.4f ms (%.1f %% of a step; HBM bound %.4f ms for %d B per env, %.0f MB: %.0f %%), host variant "
              "%.3f ms per call (host clock; %.3f ms between events)" % (label, dev_ms, 100 * dev_ms / step_ms, bound_ms, per_env,
                                                                        per_env * B / 1e6, 100 * bound_ms / dev_ms, host_ms, host_ev), flush=True)
        del tf, tv
    print(json.dumps(out))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(out, f, indent=1)
    fd.destroy()


if __name__ == "__main__":
    main()
