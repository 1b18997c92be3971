"""Measurement: what a declared external wrench costs.  C3 at 262,144 environments with a tip wrench (generic tensor-memory
kernel) against the undeclared world (rolled arm specialisation); C4 (Volume) at 131,072 environments with and without a
trunk wrench (generic kernel in both); the call time of rkFDBatchSetExtWrenchDevice and rkFDBatchSetExtWrench.  CUDA events on
the engine's stream (rkFDBatchSetStream) after --warmup steps, the same seeded states for both worlds of a pair, the two
worlds alternating --rounds times.

    python tools/exp_ext_wrench.py [--steps 100] [--warmup 30] [--rounds 3] [--out FILE]
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


def make(w, q, qd, u, links, W):
    fd, _ = capi.create_world(w, B=q.shape[0])
    if links:
        fd.batch_set_ext_wrench_links(links); fd.batch_set_ext_wrench(W)
    fd.batch_set_state(q, qd); fd.batch_set_motor_input(u); fd.update_init()
    fd.batch_set_stream(torch.cuda.current_stream().cuda_stream)
    return fd


def step_ms(fd, steps):
    st = torch.cuda.current_stream()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize(); e0.record(st)
    for _ in range(steps):
        fd.update()
    e1.record(st); torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def pair(label, w, B, sample, links, wscale, args):
    q, qd, u = sample(B)
    W = np.zeros((B, len(links), 6)); W[:, :, :3] = np.random.default_rng(1).uniform(-wscale, wscale, (B, len(links), 3))
    runs = {"undeclared": make(w, q, qd, u, None, None), "declared": make(w, q, qd, u, links, W)}
    res = {k: {"variant": fd.kernel_variant(), "ms": []} for k, fd in runs.items()}
    for fd in runs.values():
        for _ in range(args.warmup):
            fd.update()
    for _ in range(args.rounds):
        for k, fd in runs.items():
            res[k]["ms"].append(step_ms(fd, args.steps))
    for k in res:
        print("%-5s %-10s variant %s: %s ms per step" % (label, k, res[k]["variant"], " ".join("%.4f" % x for x in res[k]["ms"])), flush=True)
    out = {"case": label, "B": B, "links": links, **{k: {"variant": v["variant"], "ms": v["ms"], "median_ms": float(np.median(v["ms"]))} for k, v in res.items()}}
    return out, runs, W


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=30)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True).stdout.strip()
    print(gpu, flush=True)
    out = {"gpu": gpu, "cases": []}
    w3 = ch.world_c3()
    r, runs, W = pair("C3", w3, 262144, lambda B: ch.sample_state(w3, B, seed=20260418), [7], 5.0, args)
    out["cases"].append(r)
    # setter call times on the declared C3 batch
    fd = runs["declared"]; st = torch.cuda.current_stream()
    tw = torch.from_numpy(W).cuda(); torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    fd.batch_set_ext_wrench_device(0, tw.data_ptr()); torch.cuda.synchronize()
    e0.record(st)
    for _ in range(args.reps):
        fd.batch_set_ext_wrench_device(0, tw.data_ptr())
    e1.record(st); torch.cuda.synchronize()
    dev_ms = e0.elapsed_time(e1) / args.reps
    fd.batch_set_ext_wrench(W)
    t0 = time.perf_counter()
    for _ in range(args.reps):
        fd.batch_set_ext_wrench(W)
    host_ms = (time.perf_counter() - t0) * 1e3 / args.reps
    out["setters"] = {"B": 262144, "nlink": 1, "device_ms": dev_ms, "host_ms": host_ms}
    print("setters at 262144 envs, 1 link: device %.4f ms (events), host %.3f ms per call (host clock, synchronous)" % (dev_ms, host_ms), flush=True)
    for x in runs.values():
        x.destroy()
    w4 = ch.world_c4_volume()
    r, runs, _ = pair("C4", w4, 131072, lambda B: ch.sample_c4_standing(w4, B), [0], 20.0, args)
    out["cases"].append(r)
    for x in runs.values():
        x.destroy()
    print(json.dumps(out))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
