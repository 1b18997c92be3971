"""Tuning aid: A/B of two builds of the library on one GPU.  Runs `bench.py --no-cpu-baseline` alternately with library A
and library B (ROKIFD_B200_LIB), `--reps` times each, and prints the median / min / max of ms_per_step per build with the
card's name and power limit.  Alternating spreads the drift of a shared machine over both builds.

    python tools/ab_bench.py --a roki-fd_b200/exp/librokifd_b200_base.so --b roki-fd_b200/librokifd_b200.so [--config C3]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def bench_line(lib, args):
    env = dict(os.environ, ROKIFD_B200_LIB=os.path.abspath(lib))
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--no-cpu-baseline", "--config", args.config,
           "--steps", str(args.steps), "--warmup", str(args.warmup)]
    out = subprocess.run(cmd, env=env, cwd=ROOT, check=True, capture_output=True, text=True).stdout
    return json.loads([ln for ln in out.splitlines() if ln.startswith("{")][-1])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--a", required=True, help="library A (e.g. the parent commit's build)")
    ap.add_argument("--b", required=True, help="library B")
    ap.add_argument("--config", default="C3")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--out", help="also write all lines and the summary as JSON")
    args = ap.parse_args()
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True).stdout.strip()
    runs = {"a": [], "b": []}
    for r in range(args.reps):
        for k in ("a", "b"):
            line = bench_line(getattr(args, k), args)
            runs[k].append(line)
            print("rep %d %s: %.4f ms/step" % (r, k, line["ms_per_step"]), flush=True)
    summary = {"gpu": gpu, "config": args.config, "steps": args.steps, "warmup": args.warmup}
    for k in ("a", "b"):
        ms = [ln["ms_per_step"] for ln in runs[k]]
        summary[k] = {"lib": getattr(args, k), "median": statistics.median(ms), "min": min(ms), "max": max(ms), "ms": ms}
    summary["b_over_a"] = summary["b"]["median"] / summary["a"]["median"]
    print(json.dumps(summary))
    if args.out:
        with open(args.out, "w") as f:
            json.dump({"summary": summary, "lines": runs}, f, indent=1)


if __name__ == "__main__":
    main()
