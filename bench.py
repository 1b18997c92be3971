#!/usr/bin/env python
"""bench.py - env-steps/s of the batched FD+contact step (BASELINE.json metric) on N B200s.

Default workload (config.workload): C3 of SURVEY.md section 8d - 7-DoF arm with an 8-vertex end-effector on a soft
floor (vertex penalty contact + joint friction + DC motors), 262,144 environments per GPU, synthetic
randomised initial states (numpy default_rng(20260418)), dt = 1e-3, Runge-Kutta-Gill.  One "step" =
one rkFDUpdate for every environment (5 dynamics evaluations + RKG combination, one kernel launch).
--config {C2,C3,C4,C5-mlcp,C5-vert} selects another BASELINE.json configuration (same JSON line).

  python bench.py --gpus N --steps K --warmup W              the CUDA engine (one process per GPU)
  python bench.py --impl reference --gpus N --steps K ...    the CPU restatement of the reference on all
                                                             host cores (the reference itself is un-buildable
                                                             here: ZEDA/ZM/Zeo/RoKi absent)
  python bench.py ... --dump-outputs DIR                     also writes what the last timed step computed as
                                                             DIR/<name>.npy (seeded inputs: runs of two builds
                                                             compare output for output)
Prints ONE JSON line on rank 0.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SEED = 20260418
METRIC = "env-steps/sec (batched FD+contact step)"
UNIT = "env-steps/s"


def _c4_states(world, ch, B, seed):
    return ch.sample_c4_standing(world, B, seed=seed)


def _mighty_states(world, ch, B, seed):
    """mighty.ztk near its registered standing pose ([roki::chain::init]: trunk at z = 0.3667, soles on the floor)."""
    q0 = np.array(ch.load_flat(os.path.join(ROOT, "tests", "golden", "flat_mighty_on_floor.txt"))["init.q[0]"])
    rng = np.random.default_rng(seed)
    q = np.tile(q0, (B, 1)); q[:, 6:] += 0.002 * rng.uniform(-1, 1, (B, world.nq - 6))
    return q, rng.uniform(-0.05, 0.05, (B, world.nq)), np.zeros((B, world.nl))


def _default_states(world, ch, B, seed):
    return ch.sample_state(world, B, seed=seed)


# BASELINE.json configurations that fit one GPU (SURVEY.md section 8d).  Per config: the world, environments per GPU,
# untimed settle steps from the synthetic initial states, ALGORITHMIC bytes / flop per env-step (section 8d's figures; None
# where the survey gives no closed formula), the CPU samples (environments per host core, steps) of the cpu_baseline leg
# and of one "step" of the reference arm; `slow` marks steps of tens of ms.  C3 is the configuration BASELINE.json's metric
# is quoted on: the default.
CONFIGS = {
    "C2": dict(label="C2: arm7 (7-DoF, DC motors, joint friction), no contact (pure ABA kernel)",
               world=lambda ch: ch.world_c2(), envs=65536, settle=0, states=_default_states,
               alg_bytes=462.0, alg_flop=16351.0, cpu=(1024, 400), ref=(512, 100)),
    "C3": dict(label="C3: arm7 (7-DoF, DC motors, joint friction) + 8-vertex penalty ground contact",
               world=lambda ch: ch.world_c3(), envs=262144, settle=700, states=_default_states,
               alg_bytes=1054.0, alg_flop=20471.0, cpu=(1024, 400), ref=(512, 100)),
    "C4": dict(label="C4: legged tree (floating trunk + two 3-joint legs, 12 DoF, box soles) standing, volume-based contact (rkfd_volume)",
               world=lambda ch: ch.world_c4_volume(), envs=131072, settle=10, states=_c4_states,
               alg_bytes=66.0 * 12 + 74.0 * 16, alg_flop=None, cpu=(8, 40), ref=(4, 10), slow=True),
    "C4-mighty": dict(label="C4 on the reference's own model: mighty.ztk (25 links, 26 DoF, 701 collision vertices; tests/golden/flat_mighty_on_floor.txt) "
                            "standing on floor.ztk, volume-based contact (rkfd_volume) on the soles",
                      world=lambda ch: ch.world_from_flat(ch.load_flat(os.path.join(ROOT, "tests", "golden", "flat_mighty_on_floor.txt"))),
                      envs=32768, settle=10, states=lambda world, ch, B, seed: _mighty_states(world, ch, B, seed),
                      alg_bytes=66.0 * 26 + 74.0 * 701, alg_flop=None, cpu=(8, 40), ref=(4, 10), slow=True),
    "C5-mlcp": dict(label="C5: arm7 + 8-vertex cube on the rigid floor (K=1000, L=1e-4), MLCP/PGS max_iter=10; 1M envs over 8 GPUs = 131,072 per GPU",
                    world=lambda ch: ch.world_c5(base_z=0.45, solver="MLCP"), envs=131072, settle=500, states=_default_states,
                    alg_bytes=1054.0, alg_flop=106191.0, cpu=(256, 400), ref=(128, 100)),
    "C5-vert": dict(label="C5: arm7 + 8-vertex cube on the rigid floor (K=1000, L=1e-4), Vert active-set QP pyramid=8; 1M envs over 8 GPUs = 131,072 per GPU",
                    world=lambda ch: ch.world_c5(base_z=0.45, solver="Vert"), envs=131072, settle=500, states=_default_states,
                    alg_bytes=1054.0, alg_flop=None, cpu=(128, 400), ref=(64, 100)),
}


def workload_string(cfg, envs):
    return "%s, %d envs/GPU, states after %d settle steps from the random initial states" % (cfg["label"], envs, cfg["settle"])


def host_threads():
    """Every host thread this process may use.  Passed EXPLICITLY to the oracle: torchrun exports OMP_NUM_THREADS=1,
    which made the round-1 reference arm run on one core for N > 1."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return os.cpu_count() or 1


def kernel_source_hash():
    """Identity of the kernel sources a profiles/traffic.json entry was captured for."""
    import hashlib
    h = hashlib.sha256()
    d = os.path.join(ROOT, "roki-fd_b200", "csrc")
    for f in ("rkfd_core.cuh", "rkfd_kernel.cuh", "rkfd_math.cuh", "rkfd_types.h", "rkfd_volume.cuh", "rkfd_kernel_variant.cu"):
        with open(os.path.join(d, f), "rb") as fh:
            h.update(fh.read())
    return h.hexdigest()[:16]


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return json.load(f).get("hbm_gbs", 6650.0), "measured"
    return 6650.0, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled while the device runs the benchmark load (settle + warm-up + timed steps)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.rows, self.proc, self.gpu = [], None, gpu_index
        self.t0, self.t1, self.note = None, None, None

    def mark_begin(self):      # the device is under the benchmark's load from here ...
        self.t0 = time.time()

    def mark_end(self):        # ... to here: only samples in between are reported
        self.t1 = time.time()

    def _loaded(self):
        t0 = self.t0 if self.t0 is not None else 0.0
        t1 = self.t1 if self.t1 is not None else float("inf")
        return [r for (t, r) in self.rows if t0 + 0.15 <= t <= t1]      # +0.15 s: a sample reports the preceding interval

    def loaded_samples(self):
        return len(self._loaded())

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [c.strip() for c in line.split(",")]))

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        for r in self._loaded():
            try:
                sm.append(float(r[1])); mx = float(r[2])
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        out = {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
               "samples": len(sm)}
        if self.note:
            out["note"] = self.note
        return out


DUMP_BYTES = 64 * 10**6      # --dump-outputs: all files together, .npy headers included


def step_outputs(fd, world):
    """What a caller of the step path reads back after a step, one row per environment: the state (rkFDBatchGetState),
    the status word and, in worlds with contact slots, the contact state and forces."""
    q, qd, qdd = fd.batch_get_state()
    out = {"q": q, "qd": qd, "qdd": qdd, "status": fd.batch_get_status()}
    if world.nslot:
        out["contact_active"], out["contact_type"], out["contact_ref"], out["contact_force"] = fd.batch_get_contact()
    return out


def dump_outputs(path, arrays, seed=SEED):
    """Writes `arrays` (first axis: environment) as <path>/<name>.npy in float64, with env_index.npy naming the environments
    written.  Beyond DUMP_BYTES in all, every array keeps the same fixed sample of environments (drawn from `seed`)."""
    B = len(next(iter(arrays.values())))
    per_env = 8 * (1 + sum(a[0].size for a in arrays.values()))
    room = DUMP_BYTES - 4096 * (len(arrays) + 1)
    idx = np.arange(B)
    if B * per_env > room:
        idx = np.sort(np.random.default_rng(seed).choice(B, room // per_env, replace=False))
    out = {name: np.asarray(a, np.float64)[idx] for name, a in arrays.items()}
    out["env_index"] = idx.astype(np.float64)
    os.makedirs(path, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(path, name + ".npy"), a)


def cpu_settled_state(world, ch, cfg, n_envs, seed=SEED):
    """Initial states of the CPU sample: the same synthetic states, settled by the oracle itself (untimed)."""
    from oracle import oracle as orc
    ow = orc.OracleWorld(world)
    q, qd, u = cfg["states"](world, ch, n_envs, seed)
    if cfg["settle"] > 0:
        q, qd, _, _ = ow.batch_run(q, qd, u, nsteps=cfg["settle"], nthreads=host_threads())
    return ow, q, qd, u


def cpu_baseline_run(ow, q, qd, u, n_steps, threads):
    """The oracle (CPU restatement of the reference's algorithm) on the host cores: env-steps/s."""
    t0 = time.perf_counter()
    _, _, _, used = ow.batch_run(q, qd, u, nsteps=n_steps, nthreads=threads)
    dt = time.perf_counter() - t0
    # batch_run also performs rkFDUpdateInit's evaluation per env: count it as 1/5 of a step
    return q.shape[0] * (n_steps + 0.2) / dt, used, dt


CPU_NOTE = "CPU restatement of RoKi-FD's algorithm (oracle/); reference un-buildable (ZEDA/ZM/Zeo/RoKi absent)"


def cpu_baseline_leg(world, ch, cfg):
    threads = host_threads()
    n_envs, n_steps = cfg["cpu"][0] * threads, cfg["cpu"][1]       # ~10-30 s of CPU work on every host core (settling included)
    ow, cq, cqd, cu = cpu_settled_state(world, ch, cfg, n_envs)
    v, used, dt = cpu_baseline_run(ow, cq, cqd, cu, n_steps, threads)
    return {"value": v, "unit": UNIT, "cores": used, "kind": "port",
            "sample": "%d envs x %d steps of the same workload, settled %d steps first (timed %.1f s)" % (n_envs, n_steps, cfg["settle"], dt),
            "note": CPU_NOTE}


def run_reference(args, emit):
    """--impl reference: the reference's own CPU implementation of the path.  The reference cannot be
    compiled (its dependencies are absent), so this times the oracle port with every host thread.  One "step" of this
    arm = a bounded sample of the workload: cfg["ref"][0] environments per host thread x cfg["ref"][1] rkFDUpdate calls."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import rokifd_b200  # noqa: F401
    from rokifd_b200 import chains as ch
    cfg = CONFIGS[args.config]
    world = cfg["world"](ch)
    threads = host_threads()
    n_envs, n_sub = cfg["ref"][0] * threads, cfg["ref"][1]
    ow, q, qd, u = cpu_settled_state(world, ch, cfg, n_envs)
    for _ in range(min(args.warmup, 2)):
        cpu_baseline_run(ow, q, qd, u, n_sub, threads)
    t0 = time.perf_counter()
    done, used = 0.0, threads
    for _ in range(args.steps):
        _, used, _ = cpu_baseline_run(ow, q, qd, u, n_sub, threads)
        done += n_envs * (n_sub + 0.2)
    dt = time.perf_counter() - t0
    value = done / dt
    sample = "per step: %d envs x %d rkFDUpdate (+ the UpdateInit evaluation), %d timed steps, %.1f s" % (n_envs, n_sub, args.steps, dt)
    out = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
           "warmup": args.warmup, "ms_per_step": 1e3 * dt / max(args.steps, 1), "higher_is_better": True, "scaling": "weak",
           "vs_baseline": None, "dtype": "f64", "data": "synthetic",
           "config": {"workload": workload_string(cfg, args.envs or cfg["envs"]), "cpu_sample": sample},
           "cpu_baseline": {"value": value, "unit": UNIT, "cores": used, "kind": "port", "sample": sample, "note": CPU_NOTE},
           "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(out)


def _json_only_stdout():
    """Everything but the result line goes to stderr: native libraries (NCCL prints its version banner) write to file
    descriptor 1 directly, and the contract is ONE JSON line on stdout.  Returns the function that prints it."""
    sys.stdout.flush()
    real = os.dup(1)
    os.dup2(2, 1)

    def emit(obj):
        sys.stdout.flush()
        os.write(real, (json.dumps(obj) + "\n").encode())
    return emit


def _cpulist(text):
    cpus = set()
    for part in text.strip().split(","):
        if not part:
            continue
        lo, _, hi = part.partition("-")
        cpus.update(range(int(lo), int(hi or lo) + 1))
    return cpus


def gpu_numa_node(torch, device_index):
    """NUMA node the GPU hangs off: sysfs first, `nvidia-smi topo -m` ("NUMA Affinity" column) when sysfs says -1."""
    try:
        pr = torch.cuda.get_device_properties(device_index)
        bdf = "%04x:%02x:%02x.0" % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)
        with open("/sys/bus/pci/devices/%s/numa_node" % bdf) as f:
            node = int(f.read().strip())
        if node >= 0:
            return node, "sysfs"
    except Exception:
        pass
    try:
        txt = subprocess.run(["nvidia-smi", "topo", "-m"], capture_output=True, text=True, timeout=20).stdout
        lines = [l for l in txt.splitlines() if l.strip()]
        head = [h.strip() for h in lines[0].split("\t")]
        col = [i for i, h in enumerate(head) if "NUMA Affinity" in h]
        for l in lines[1:]:
            cells = [c.strip() for c in l.split("\t")]
            if cells and cells[0] == "GPU%d" % device_index and col and col[0] < len(cells):
                v = cells[col[0]].split(",")[0].split("-")[0]
                if v.isdigit():
                    return int(v), "nvidia-smi topo"
    except Exception:
        pass
    return None, "unknown"


def bind_to_gpu_numa_node(torch, device_index):
    """Places this process's future allocations (the pinned host buffers of the end-to-end leg) on the NUMA node the GPU
    hangs off: set_mempolicy(MPOL_PREFERRED, node) - which needs no CPU affinity - and, where the node's CPUs are in our
    affinity mask, the CPU affinity as well.  8 ranks on a two-socket box otherwise push half of their PCIe traffic
    across the socket interconnect.  Best effort: returns (node or None, how)."""
    node, how = gpu_numa_node(torch, device_index)
    if node is None:
        return None, how
    done = []
    try:
        import ctypes
        libc = ctypes.CDLL(None, use_errno=True)
        mask = (ctypes.c_ulong * 16)()
        mask[node // 64] = 1 << (node % 64)
        SYS_set_mempolicy, MPOL_PREFERRED = 238, 1      # x86_64
        if libc.syscall(SYS_set_mempolicy, MPOL_PREFERRED, mask, 16 * 64 + 1) == 0:
            done.append("set_mempolicy")
    except Exception:
        pass
    try:
        with open("/sys/devices/system/node/node%d/cpulist" % node) as f:
            cpus = _cpulist(f.read()) & os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            done.append("cpu affinity")
    except Exception:
        pass
    return (node if done else None), how + (": " + "+".join(done) if done else ": not applied")


def main():
    emit = _json_only_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="C3", choices=list(CONFIGS), help="BASELINE.json configuration (default: C3, the one the metric is quoted on)")
    ap.add_argument("--envs", type=int, default=0, help="environments per GPU (default: the configuration's)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--e2e-upload-state", action="store_true", help="e2e leg: also re-send (q, q') host->device every step")
    ap.add_argument("--e2e-outputs", default="q,qd", help="e2e leg: what the caller reads back every step, of q,qd,qdd (default q,qd: what the "
                    "feedback loop of the reference's example/chain/arm_box_test.c:10-23 reads - rkJointGetDis/GetVel - before it sets the motor inputs)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed (state, status, contacts of rank 0's "
                    "environments; a fixed sample of them beyond 64 MB) as DIR/<name>.npy in float64")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the CUDA engine (--impl b200)")
    if args.impl == "reference":
        return run_reference(args, emit)
    if args.warmup < 3:
        args.warmup = 3
    cfg = CONFIGS[args.config]

    import torch
    import rokifd_b200  # noqa: F401
    from rokifd_b200 import capi, chains as ch, multi

    rank = int(os.environ.get("RANK", "0"))
    world_size = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    affinity0 = host_threads()                           # before the NUMA binding narrows it: the CPU leg uses all of them
    all_cpus = os.sched_getaffinity(0)
    torch.cuda.set_device(local_rank)
    numa, numa_how = bind_to_gpu_numa_node(torch, local_rank)     # before any pinned allocation: host buffers next to the GPU
    dist = None
    if world_size > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    sampler = ClockSampler(local_rank)      # started early: the first nvidia-smi of a fresh box can take seconds to report
    sampler.start()
    world = cfg["world"](ch)
    B = args.envs or cfg["envs"]
    q, qd, u = cfg["states"](world, ch, B, SEED + rank)      # weak scaling: every rank its own synthetic states
    fd, _ = capi.create_world(world, B=B, devices=[local_rank])
    fd.batch_set_state(q, qd)
    fd.batch_set_motor_input(u)
    fd.update_init()
    stream = torch.cuda.current_stream()
    fd.batch_set_stream(stream.cuda_stream)       # kernels run on torch's current stream: torch events bracket them

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident throughput ("value") --------------------------------------------------------
    # settle (untimed, ~1 s of GPU load: also lets nvidia-smi deliver samples of the loaded device), then warm-up
    sampler.mark_begin()
    settle = cfg["settle"]
    fd.update_n(settle // 2)
    torch.cuda.synchronize()
    fd.update_n(settle - settle // 2)
    for _ in range(args.warmup):
        fd.update()
    barrier()
    l0 = fd.launch_count
    r0 = fd.resort_count
    rk0 = fd.resort_kernel_count
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
    ev[0].record(stream)
    for s in range(args.steps):
        fd.update()
        ev[s + 1].record(stream)
    barrier()
    launches = fd.launch_count - l0
    resorts = fd.resort_count - r0
    resort_kernels = fd.resort_kernel_count - rk0
    sampler.mark_end()
    outputs = step_outputs(fd, world) if args.dump_outputs and rank == 0 else None     # before any further step
    if sampler.loaded_samples() == 0:
        # nvidia-smi delivered nothing inside the timed region (slow start): keep the same load on the device until it does
        t_wait = time.time()
        while sampler.loaded_samples() == 0 and time.time() - t_wait < 5.0:
            fd.update_n(5 if cfg.get("slow") else 100); torch.cuda.synchronize()
        sampler.mark_end()
        sampler.note = "no nvidia-smi sample fell inside the loaded region (settle + warm-up + timed steps); sampled under the same load right after it"
    clocks = sampler.stop()
    total_ms = ev[0].elapsed_time(ev[-1])
    per_launch_ms = [ev[s].elapsed_time(ev[s + 1]) for s in range(args.steps)]
    if os.environ.get("RKFD_BENCH_DEBUG"):
        print("rank %d: total %.3f ms, per-launch min/median/max %.3f/%.3f/%.3f ms" % (rank, total_ms, min(per_launch_ms), float(np.median(per_launch_ms)), max(per_launch_ms)), file=sys.stderr)
    total_ms = multi.max_over_ranks(dist, total_ms, device="cuda")      # the job's time is the slowest rank's
    value = multi.job_throughput(B, world_size, args.steps, total_ms)
    nbad = int((fd.batch_get_status() != 0).sum())
    assert nbad == 0 or args.config != "C3", "non-finite accelerations in the timed run"
    contact_frac = mean_active = None
    if world.nslot:
        ca, _, _, _ = fd.batch_get_contact()
        contact_frac, mean_active = float((ca.sum(1) > 0).mean()), float(ca.sum(1).mean())
    q, qd, _ = (np.ascontiguousarray(x) for x in fd.batch_get_state())     # settled states: inputs of the e2e leg

    # ---- end to end through the C-ABI with HOST buffers ("e2e") -----------------------------------------
    nq, nl = world.nq, world.nl
    hq = torch.from_numpy(q.copy()).pin_memory(); hqd = torch.from_numpy(qd.copy()).pin_memory()
    hu = torch.from_numpy(u.copy()).pin_memory()
    oq = torch.empty((B, nq), dtype=torch.float64).pin_memory(); oqd = torch.empty_like(oq).pin_memory()
    oqdd = torch.empty_like(oq).pin_memory()
    e2e_steps = max(3, min(args.steps, 20))
    outs = [o for o in args.e2e_outputs.split(",") if o in ("q", "qd", "qdd")]
    assert outs, "--e2e-outputs needs at least one of q,qd,qdd"

    def e2e_step():
        # every step: this step's inputs host->device from pinned memory, the step, its result device->host.
        # A step's inputs are what the reference's callers set between two rkFDUpdate calls - the motor inputs
        # (rkJointMotorSetInput, example/chain/arm_box_test.c:21); the simulator owns the state, as the reference's
        # rkFD does.  Its result is the state the caller reads back: q, q', q''.  --e2e-upload-state also re-sends
        # (q, q') every step (rkFDChainSetDis/SetVel before every update).
        # The calls are asynchronous (copy streams + staging ring), so the transfers of neighbouring steps overlap
        # the step kernel; rkFDBatchJoin + the closing event make the timed region cover all of them.
        if args.e2e_upload_state:
            fd.batch_set_state_async(hq.data_ptr(), hqd.data_ptr())
        fd.batch_set_motor_input_async(hu.data_ptr())
        fd.update()
        fd.batch_get_state_async(oq.data_ptr() if "q" in outs else None, oqd.data_ptr() if "qd" in outs else None,
                                 oqdd.data_ptr() if "qdd" in outs else None)

    def e2e_time(closed_loop):
        for _ in range(3):
            e2e_step()
        fd.batch_sync()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(e2e_steps):
            e2e_step()
            if closed_loop:
                fd.batch_sync()       # the caller needs step k's state on the host before it sends step k+1's inputs
        fd.batch_join()
        e1.record(stream)
        fd.batch_sync()
        barrier()
        return multi.job_throughput(B, world_size, e2e_steps, multi.max_over_ranks(dist, e0.elapsed_time(e1), device="cuda"))

    e2e_value = e2e_time(False)
    e2e_closed = e2e_time(True)
    assert np.isfinite((oq if "q" in outs else oqd if "qd" in outs else oqdd).numpy()).all() or nbad > 0
    h2d = B * ((2 * nq if args.e2e_upload_state else 0) + nl) * 8
    d2h = B * len(outs) * nq * 8

    # ---- end-of-run reductions over the job (SURVEY.md section 8e: the only collective, after the timed region) ----
    stats = fd.batch_stats()          # per rank: envs, envs in contact, active vertices, failed envs (sums); max|q''|, max|q'| (max)
    if dist is not None:
        ssum = torch.tensor(stats[:4], dtype=torch.float64, device="cuda"); smax = torch.tensor(stats[4:6], dtype=torch.float64, device="cuda")
        dist.all_reduce(ssum, op=dist.ReduceOp.SUM); dist.all_reduce(smax, op=dist.ReduceOp.MAX)
        stats = ssum.tolist() + smax.tolist()
    job_stats = {"envs": int(stats[0]), "envs_in_contact": int(stats[1]), "active_contact_vertices": int(stats[2]),
                 "failed_envs": int(stats[3]), "max_abs_qdd": stats[4], "max_abs_qd": stats[5],
                 "how": "rkFDBatchStats per rank%s" % (" + ncclAllReduce(sum|max)" if dist is not None else "")}

    # ---- roofline of the dominant kernel (rkfd_step_kernel: the only kernel of a step) ------------------
    hbm_peak, peak_src = load_peaks()
    k_ms = float(np.mean(per_launch_ms))
    traffic, traffic_note = None, "no ncu capture on record for this configuration"
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tpath):
        with open(tpath) as f:
            tj = json.load(f).get(args.config)
        if tj:
            if tj.get("kernel_source_hash") == kernel_source_hash() and tj.get("envs") == B:
                traffic, traffic_note = tj.get("dram_bytes_per_launch"), "ncu --set full capture %s (same kernel sources, same batch)" % tj.get("capture")
            else:
                traffic_note = "stale: the capture on record (%s) was taken for other kernel sources or another batch" % tj.get("capture")
    ach_gbs = cfg["alg_bytes"] * B / (k_ms * 1e-3) / 1e9
    fp64_peak = capi.measure_fp64_tflops()
    ach_tf = cfg["alg_flop"] * B / (k_ms * 1e-3) / 1e12 if cfg["alg_flop"] else None
    hbm_roof = {"bound": "hbm", "achieved": ach_gbs, "peak": hbm_peak, "unit": "GB/s", "frac": ach_gbs / hbm_peak,
                "traffic": traffic, "traffic_note": traffic_note, "peak_source": peak_src, "kernel": "rkfd_step_kernel", "kernel_ms": k_ms,
                "algorithmic_bytes_per_env_step": cfg["alg_bytes"]}
    fp64_roof = {"bound": "fp64", "achieved": ach_tf, "peak": fp64_peak, "unit": "TFLOP/s",
                 "frac": ach_tf / fp64_peak if (fp64_peak and ach_tf) else None, "traffic": traffic, "traffic_note": traffic_note,
                 "peak_source": "measured in this run (register-resident DFMA loop on every SM; MEASURED_PEAKS.json has no fp64 figure)",
                 "kernel": "rkfd_step_kernel", "kernel_ms": k_ms, "algorithmic_flop_per_env_step": cfg["alg_flop"]}
    # the binding roof of this path is the fp64 pipe (SURVEY.md section 8d: ~19 flop per byte against a machine balance of ~5);
    # configurations without a closed flop formula (Volume, Vert QP) report against HBM only
    binding = fp64_roof if ach_tf else hbm_roof

    out = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world_size, "steps": args.steps, "warmup": args.warmup,
           "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
           "dtype": "f64", "data": "synthetic",
           "config": {"workload": workload_string(cfg, B), "name": args.config, "envs_per_gpu": B, "dt": world.dt, "integrator": "RKG", "solver": world.solver,
                      "settle_steps": settle, "envs_in_contact": contact_frac, "mean_active_vertices": mean_active, "flagged_envs": nbad,
                      "numa_node": numa, "numa_how": numa_how,
                      "env_resorts_in_timed_region": int(resorts),       # the engine re-orders its slots by contact count every 16 steps (rkFDBatchSetResortInterval)
                      "l2": "per-GPU state (%.0f MB) is larger than the 126 MB L2" % (B * 8 * 140 / 1e6) if B * 8 * 140 > 126e6 else
                            "per-GPU state %.0f MB: fits the 126 MB L2 (the configuration's batch is what BASELINE.json names)" % (B * 8 * 140 / 1e6)},
           "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "steps": e2e_steps,
                   "closed_loop_value": e2e_closed,
                   "io": "per step: motor inputs u[B][%d] host->device%s, rkFDUpdate, (%s)[B][%d] device->host; pinned host buffers, "
                         "asynchronous copies on their own streams.  value: pipelined caller (step k+1's inputs do not depend on step k's "
                         "outputs: transfers overlap the kernels); closed_loop_value: the caller waits for step k's state on the host before "
                         "sending step k+1's inputs" % (nl, " + state (q, q')" if args.e2e_upload_state else "", ", ".join(outs), nq)},
           # every kernel of this repository launched inside the timed region: one rkfd_step_kernel per step plus the kernels of the
           # environment re-sorts that fell into it (key / offsets / assign / row permutations / order; their device-to-device
           # staging copies are cudaMemcpyAsync calls, not kernels)
           "gpu_launches": int(launches + resort_kernels),
           "gpu_launches_detail": {"rkfd_step_kernel": int(launches), "resort_kernels": int(resort_kernels), "resorts": int(resorts)},
           "clocks": clocks,
           "job_stats": job_stats,
           "roofline": binding, "roofline_hbm": hbm_roof, "roofline_fp64": fp64_roof}
    if rank == 0 and not args.no_cpu_baseline:
        # the other ranks wait in the closing barrier; rank 0 takes back every host thread for the CPU leg
        try:
            os.sched_setaffinity(0, all_cpus)
        except Exception:
            pass
        assert host_threads() == affinity0
        out["cpu_baseline"] = cpu_baseline_leg(world, ch, cfg)
    if outputs is not None:
        dump_outputs(args.dump_outputs, outputs)
    fd.destroy()
    if rank == 0:
        emit(out)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
