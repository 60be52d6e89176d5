#!/usr/bin/env python
"""bench.py — unique states explored per second for VSR.tla (BASELINE.json's metric).

Workload (config.workload): BASELINE configs[1] = the reference's shipped VSR.cfg — ReplicaCount=3, ClientCount=1,
Values={v1,v2}, StartViewOnTimerLimit=2, VIEW view, SYMMETRY symmValues, INVARIANT AcknowledgedWriteNotLost,
deadlock checking off, exploration continued past the violation to the COMPLETE reachable set (1,173,992,337
distinct states, depth 47).  One "step" = one complete BFS of that state space.  Inputs are fully determined
by the config (single Init state): "synthetic" data does not apply; nothing is cached between steps — every
step clears the seen-set and starts from Init.

  value   distinct states / second, device-timed over K steps with the engine (tables allocated) resident in HBM
  e2e     the same metric through the public one-call API (ModelChecker.check -> vsr_bfs): config text in host
          memory -> parse -> allocate -> BFS -> stats and counterexample back in host memory
  --impl reference   the CPU restatement of the spec (oracle/, "port": TLC itself cannot run here — no JVM) on all
          host cores, bounded sample per step

Launch: python bench.py --gpus N --steps K --warmup W   (N>1: under torchrun, one rank per GPU, NCCL).
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOAD = dict(R=3, V=2, L=2)           # BASELINE configs[1] = vsr-revisited/paper/VSR.cfg
TABLE_CAP = 1 << int(os.environ.get("VSR_BENCH_TABLE_LOG2", "32"))  # 2^32 slots * 16 B = 64 GiB over all GPUs (1.17e9 states -> load 0.27: measured 10 %
                                                                     # less kernel time than 2^31, profiles/round2_expand_kernel.md) + 8 B of trace record per slot
FRONTIER_CAP = 140_000_000               # widest level: 120,193,500 states
EXPECT = dict(distinct=1173992337, generated=3129587684, depth=47, violation_level=28)
# a configuration BOTH arms finish: (R=3, V=2, L=1) WITHOUT SYMMETRY, complete = 697,364 distinct states, depth 30 - totals pinned to
# the spec's text (tests/golden/spec_text_results.json) - the same-config comparison beside the bounded cfg2 sample of the CPU arm
SMALL = dict(R=3, V=2, L=1, symmetry=0, distinct=697364, generated=1831657, depth=30)
# BASELINE configs[2]/[4]: README constants to the first AcknowledgedWriteNotLost violation, at every GPU count
# Sizes per GPU count (level 24 alone is 1.345e9 states of 64 B; 3.17e9 seen-set entries + trace records): one GPU holds the seen-set,
# the trace and 2 x 560 M frontier states in HBM and lets each frontier buffer continue with 850 M states in pinned host memory (spill)
CFG3 = dict(R=3, V=3, L=3, violation_level=24, distinct=3166753191,
            table_total={1: 4_000_000_000, 2: 4_400_000_000, 4: 1 << 33, 8: 1 << 33},
            frontier_total={1: 560_000_000, 2: 1_500_000_000, 4: 1_600_000_000, 8: 1_600_000_000},
            frontier_host={1: 850_000_000, 2: 0, 4: 0, 8: 0})


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region"""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx = float(f[1])
            except ValueError:
                continue
            for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


def usable_cores():
    """Threads the CPU arm may really use: the affinity mask and a cgroup CPU quota both cap os.cpu_count() in a container."""
    n = os.cpu_count() or 1
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except (AttributeError, OSError):
        pass
    for path in ("/sys/fs/cgroup/cpu.max",):
        try:
            quota, period = open(path).read().split()[:2]
            if quota != "max":
                n = min(n, max(1, int(int(quota) / int(period))))
        except (OSError, ValueError):
            pass
    try:
        q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
        p = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
        if q > 0 and p > 0:
            n = min(n, max(1, q // p))
    except (OSError, ValueError):
        pass
    return max(1, n)


def oracle_sample(seconds, workers, cfg=None):
    """CPU restatement (oracle/) on the same workload for a bounded time (0 = to completion): distinct states / s on
    `workers` threads."""
    so = os.path.join(ROOT, "oracle", "_build", "liboracle.so")
    lib = C.CDLL(so)
    lib.orc_bfs.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_uint64, C.c_double, C.c_int, C.c_int, C.c_int, C.c_char_p,
                            C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int]
    cfg = cfg or WORKLOAD
    q = (C.c_int * 8)(cfg["R"], 1, cfg["V"], cfg["L"], 0, cfg.get("symmetry", 1), 1, 0)  # invariant 0: explore, do not stop
    scal = (C.c_uint64 * 32)()
    lv = (C.c_uint64 * 512)()
    t0 = time.time()
    lib.orc_bfs(q, workers, 0, 0, float(seconds), 0, 0, 0, None, scal, lv, None, 512, None, None, 0)
    dt = time.time() - t0
    return dict(distinct=int(scal[1]), generated=int(scal[0]), depth=int(scal[3]), seconds=dt, rate=int(scal[1]) / dt)


def small_complete_cpu(cores):
    """the same-config leg of the CPU arm: (R=3, V=2, L=1) to completion on all cores"""
    s = oracle_sample(0.0, cores, SMALL)
    ok = (s["distinct"], s["generated"], s["depth"]) == (SMALL["distinct"], SMALL["generated"], SMALL["depth"])
    return {"workload": "VSR.tla ReplicaCount=3 Values={v1,v2} StartViewOnTimerLimit=1 VIEW view, no SYMMETRY: COMPLETE state space (%d distinct states, depth %d)"
                        % (SMALL["distinct"], SMALL["depth"]),
            "value": s["rate"], "unit": "states/s", "seconds": s["seconds"], "cores": cores, "kind": "port", "results_match_expected": ok}


def try_tlc(seconds):
    """BASELINE.md: if a JVM and tla2tools.jar ever appear on the box ($TLA2TOOLS_JAR) together with the spec ($VSR_TLA),
    run the REAL reference — TLC — on the same config for a bounded time and return its rate.  In this
    image there is no java, so this returns None and the CPU restatement stands in."""
    import re
    import shutil
    import tempfile
    jar, java = os.environ.get("TLA2TOOLS_JAR"), shutil.which("java")
    tla = os.environ.get("VSR_TLA")
    if not (jar and java and tla and os.path.exists(jar) and os.path.exists(tla)):
        return None
    import _pkg
    pkg = _pkg.load()
    d = tempfile.mkdtemp()
    shutil.copy(tla, os.path.join(d, "VSR.tla"))
    with open(os.path.join(d, "VSR.cfg"), "w") as f:
        f.write(pkg.cfg_text(WORKLOAD["R"], ["v1", "v2"], WORKLOAD["L"]))
    t0 = time.time()
    try:
        out = subprocess.run([java, "-cp", jar, "tlc2.TLC", "-workers", "auto", "-deadlock", "-continue", "-config", "VSR.cfg", "VSR.tla"],
                             cwd=d, capture_output=True, text=True, timeout=seconds).stdout
    except subprocess.TimeoutExpired as e:
        out = (e.stdout or b"").decode() if isinstance(e.stdout, bytes) else (e.stdout or "")
    dt = time.time() - t0
    m = re.findall(r"([\d,]+) states generated.*?([\d,]+) distinct states found", out)
    if not m:
        return None
    distinct = int(m[-1][1].replace(",", ""))
    return dict(distinct=distinct, seconds=dt, rate=distinct / dt)


def run_reference(args, rank):
    if rank != 0:
        return
    tlc = try_tlc(30.0)
    if tlc:
        cores = usable_cores()
        print(json.dumps({
            "impl": "reference", "metric": "unique states explored/sec (VSR.tla, shipped VSR.cfg constants)", "value": tlc["rate"],
            "unit": "states/s", "n_gpus": args.gpus, "steps": 1, "warmup": 0, "ms_per_step": 1e3 * tlc["seconds"], "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "u32", "data": "none (state space of the config)",
            "config": {"workload": "VSR.tla shipped VSR.cfg constants under TLC (-workers auto -deadlock -continue), bounded run"},
            "cpu_baseline": {"value": tlc["rate"], "unit": "states/s", "cores": cores, "kind": "reference",
                             "sample": "tlc2.TLC for %.0f s: %d distinct states" % (tlc["seconds"], tlc["distinct"])},
            "e2e": {"value": tlc["rate"], "unit": "states/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
        return
    cores = usable_cores()
    per_step = 10.0
    for _ in range(min(args.warmup, 1)):
        oracle_sample(2.0, cores)
    tot_states, tot_s = 0, 0.0
    sample = None
    for _ in range(args.steps):
        sample = oracle_sample(per_step, cores)
        tot_states += sample["distinct"]
        tot_s += sample["seconds"]
    v = tot_states / tot_s
    desc = "BFS of the same config from Init for %.0f s wall per step (reaches depth %d, %d distinct states)" % (
        per_step, sample["depth"], sample["distinct"])
    print(json.dumps({
        "impl": "reference", "metric": "unique states explored/sec (VSR.tla, shipped VSR.cfg constants)", "value": v, "unit": "states/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * tot_s / max(args.steps, 1),
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "u32", "data": "none (state space of the config)",
        "config": {"workload": "VSR.tla ReplicaCount=3 ClientCount=1 Values={v1,v2} StartViewOnTimerLimit=2 (BASELINE configs[1]), "
                               "bounded sample of the BFS", "note": "CPU restatement of the spec (oracle/), NOT TLC: no JVM in this image"},
        "cpu_baseline": {"value": v, "unit": "states/s", "cores": cores, "kind": "port", "sample": desc},
        "e2e": {"value": v, "unit": "states/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        # a configuration this arm FINISHES: the b200 arm's line carries the same block (same_config_small.gpu)
        "same_config_small": small_complete_cpu(cores),
    }))


def host_memory_available():
    """bytes this process may still allocate on the host: MemAvailable, capped by the cgroup's limit (a GPU box is often a slice of a
    machine: pinning past the slice's limit gets the whole job killed, not an error code)"""
    avail = None
    try:
        for ln in open("/proc/meminfo"):
            if ln.startswith("MemAvailable:"):
                avail = int(ln.split()[1]) * 1024
    except OSError:
        pass
    for mx, cur in (("/sys/fs/cgroup/memory.max", "/sys/fs/cgroup/memory.current"),
                    ("/sys/fs/cgroup/memory/memory.limit_in_bytes", "/sys/fs/cgroup/memory/memory.usage_in_bytes")):
        try:
            m = open(mx).read().strip()
            if m != "max":
                left = int(m) - int(open(cur).read().strip())
                avail = left if avail is None else min(avail, left)
        except (OSError, ValueError):
            pass
    return avail


def golden_depths(pkg, mc, eng, torch, tdist, world, dev, rank):
    """BFS depth at which each state of the reference's published 24-state counterexample (tests/golden/
    state_transfer_trace.json, generated from state_transfer_violation_trace.txt) was first seen; 0 = not in the explored set"""
    import base64
    import zlib
    fx = json.load(open(os.path.join(ROOT, "tests", "golden", "state_transfer_trace.json")))
    Flat = pkg.checker.VsrFlatState
    levels = []
    for s in fx["states"]:
        packed = mc.pack(Flat.from_buffer_copy(zlib.decompress(base64.b64decode(s["flat_zlib_b64"]))))  # canonical labels
        lvl, owner = eng.lookup(packed)
        levels.append(lvl if owner == rank else 0)
    t = torch.tensor(levels, dtype=torch.int64, device=dev)
    if world > 1:
        tdist.all_reduce(t, op=tdist.ReduceOp.MAX)
    return [int(x) for x in t.cpu().tolist()]


def sampled_state_depths(mc, eng, torch, tdist, world, dev, rank, walks=64, steps=64, seed=0):
    """BFS depth at which the seen-set holds each state of a fixed sample of the reachable set (0 = absent): the states of
    `walks` seeded random walks of `steps` steps from Init through the host's Next, successors taken in byte order so that
    the sample does not depend on the order a build lists them in"""
    import random
    rng = random.Random(seed)
    sample = []
    for _ in range(walks):
        s = mc.init_state()
        for _ in range(steps):
            sample.append(s)
            succ = sorted(t for t, _, _ in mc.successors(s))
            if not succ:
                break
            s = rng.choice(succ)
    levels = []
    for s in sample:
        lvl, owner = eng.lookup(s)
        levels.append(lvl if owner == rank else 0)
    t = torch.tensor(levels, dtype=torch.int64, device=dev)
    if world > 1:
        tdist.all_reduce(t, op=tdist.ReduceOp.MAX)
    return t.cpu().numpy()


def dump_outputs(path, res, depths):
    """what the timed path returned in its last step, as float64 .npy files (exact: every count is below 2^53)"""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    totals = [res.rc, res.generated, res.distinct, res.queue, res.depth, res.complete, res.violation_level, res.h2_ties, res.fp_collisions]
    out = {"totals": totals,  # rc, generated, distinct, queue, depth, complete, violation_level, h2_ties, fp_collisions
           "level_sizes": res.level_sizes, "level_generated": res.level_generated, "sampled_state_depths": depths}
    for name, a in out.items():
        np.save(os.path.join(path, name + ".npy"), np.asarray(a, dtype=np.float64))


def cfg3_first_violation(pkg, vdist, torch, tdist, group, rank, world, local, dev, barrier):
    """BASELINE configs[2]/[4]: the README constants (the config the reference says needs 500 GB of disk and days under TLC)
    sharded over the job's GPUs, to the first AcknowledgedWriteNotLost violation; the published trace's states must be in
    the explored set at depths 1..24 and the checker's own counterexample must be a behaviour of Next ending in the violation."""
    mc = pkg.ModelChecker.from_constants(CFG3["R"], CFG3["V"], CFG3["L"])
    pinned = 2 * CFG3["frontier_host"][world] * mc.state_bytes
    if pinned:
        avail = host_memory_available()
        if avail is None or pinned > 0.6 * avail:
            return {"skipped": "needs %.0f GB of pinned host memory for the frontier spill; %s available to this job"
                               % (pinned / 1e9, "unknown" if avail is None else "%.0f GB" % (avail / 1e9))}
    table_cap = CFG3["table_total"][world] // world
    frontier_cap = CFG3["frontier_total"][world] // world
    barrier()
    t0 = time.time()
    eng = vdist.GpuEngine(mc, rank, world, device=local, table_capacity=table_cap, frontier_capacity=frontier_cap, keep_trace=True, group=group,
                          frontier_host_capacity=CFG3["frontier_host"][world])
    t1 = time.time()
    res = eng.run(stop_on_violation=True, want_trace=True)
    barrier()
    t2 = time.time()
    gold = golden_depths(pkg, mc, eng, torch, tdist, world, dev, rank)
    out = None
    if rank == 0:
        trace = vdist.replay_trace(mc, res.trace_cands) if res.rc == 12 else []
        mc_lit = pkg.ModelChecker.from_constants(CFG3["R"], CFG3["V"], CFG3["L"], symmetry=False)
        steps_ok = bool(trace) and all(trace[i + 1][1] in [t for t, _, _ in mc_lit.successors(trace[i][1])] for i in range(len(trace) - 1))
        viol_ok = bool(trace) and mc_lit.invariant(trace[-1][1]) != 0 and all(mc_lit.invariant(s) == 0 for _, s in trace[:-1])
        out = {"workload": "VSR.tla ReplicaCount=3 Values={v1,v2,v3} StartViewOnTimerLimit=3 (README.md:13-18) to the first AcknowledgedWriteNotLost violation",
               "n_gpus": world, "frontier_states_in_host_memory_per_buffer": CFG3["frontier_host"][world], "rc": res.rc, "violation_depth": res.violation_level, "distinct_states": res.distinct, "states_generated": res.generated,
               "seconds_bfs": t2 - t1, "seconds_setup": t1 - t0, "kernel_seconds": res.kernel_ms_max / 1e3, "states_per_s": res.distinct / (t2 - t1),
               "golden_state_depths": gold, "golden_state_depths_ok": gold == list(range(1, 25)),
               "counterexample_len": len(trace), "counterexample_actions": [a for a, _ in trace],
               "counterexample_steps_are_next_steps": steps_ok, "counterexample_violates_only_at_end": viol_ok,
               "h2_ties": res.h2_ties, "fp_collisions": res.fp_collisions,
               "matches_expected": res.rc == 12 and res.violation_level == CFG3["violation_level"] and res.distinct == CFG3["distinct"]}
    eng.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-seconds", type=float, default=15.0)
    ap.add_argument("--no-cfg3", action="store_true", help="N >= 2: skip the README-constants first-violation block (BASELINE configs[2]/[4])")
    ap.add_argument("--cfg3-one-gpu", action="store_true",
                    help="N = 1: run that block too: 3.17e9 states on ONE GPU with the frontier spilling into 109 GB of pinned host memory "
                         "(off by default: a box that is a slice of a machine may not have that much)")
    ap.add_argument("--no-e2e", action="store_true", help="profiling runs: skip the end-to-end legs")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed to DIR/<name>.npy (float64): totals, level_sizes, "
                         "level_generated, and the seen-set's depth of a fixed seeded sample of states")
    ap.add_argument("--exchange", default="p2p", choices=["p2p", "staged"],
                    help="N > 1: p2p = the kernel stores remote successors into the owner's inbox over NVLink, C++ level loop (default); "
                         "staged = the baseline it replaces: local staging buffer + NCCL send/recv per step, Python level loop")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank)
        return

    import torch
    import _pkg
    pkg = _pkg.load()
    from vsr_tlaplus_b200 import dist as vdist
    import torch.distributed as tdist

    group = None
    if world > 1:
        torch.cuda.set_device(local)
        tdist.init_process_group("nccl", device_id=torch.device("cuda", local))
    assert world == args.gpus, "launch with torchrun --nproc-per-node == --gpus"
    dev = torch.device("cuda", local)
    if world > 1:
        group = vdist.Group.from_torch()   # the ranks' shared-memory barrier / all-gather (csrc/vsr_group.cpp)

    cfg = pkg.cfg_text(WORKLOAD["R"], ["v1", "v2"], WORKLOAD["L"])
    mc = pkg.ModelChecker.from_cfg_text(cfg)
    S = mc.state_bytes
    table_cap = TABLE_CAP // world
    frontier_cap = FRONTIER_CAP // world + 4_000_000
    staged = world > 1 and args.exchange == "staged"
    eng = vdist.GpuEngine(mc, rank, world, device=local, table_capacity=table_cap, frontier_capacity=frontier_cap, keep_trace=True, group=group,
                          exchange=args.exchange)
    pump = vdist.ShardedBfs(eng, rank, world) if staged else None

    def barrier():
        torch.cuda.synchronize(dev)
        if world > 1:
            tdist.barrier()
        torch.cuda.synchronize(dev)

    def one_step():
        if staged:
            r = pump.run(stop_on_violation=False, want_trace=False)
            r.launches = int(eng.stats().kernel_launches)
            return r
        return eng.run(stop_on_violation=False, want_trace=False)

    for _ in range(args.warmup):
        res = one_step()
    sampler = ClockSampler(local)
    barrier()
    if rank == 0:
        sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    launches0 = 0
    ev0.record()
    t0 = time.time()
    kernel_ms = 0.0
    insert_ms = 0.0
    exchanged = 0
    levels_ms = []
    for _ in range(args.steps):
        res = one_step()
        kernel_ms += res.kernel_ms_max
        insert_ms += res.insert_ms_max
        exchanged += res.exchanged_records
        launches0 += res.launches
        levels_ms.append(res.level_ms)
    ev1.record()
    barrier()
    wall = time.time() - t0
    dev_ms = ev0.elapsed_time(ev1)
    t = torch.tensor([wall, dev_ms / 1e3], dtype=torch.float64, device=dev)
    if world > 1:
        tdist.all_reduce(t, op=tdist.ReduceOp.MAX)
    wall = float(t[0])
    clocks = sampler.stop() if rank == 0 else None
    st = eng.stats()
    if args.dump_outputs:
        depths = sampled_state_depths(mc, eng, torch, tdist, world, dev, rank)
        if rank == 0:
            dump_outputs(args.dump_outputs, res, depths)

    ok = (res.distinct == EXPECT["distinct"] and res.generated == EXPECT["generated"] and res.depth == EXPECT["depth"] and
          res.violation_level == EXPECT["violation_level"] and res.complete)
    value = res.distinct * args.steps / wall

    # roofline of the dominant kernel (expand_kernel): algorithmic bytes per distinct state (SURVEY §8d)
    g = res.generated / res.distinct
    b_alg = 2 * S + 32 * g + 32 + 8          # read + write the packed state, one 32 B sector per probe, the CAS sector, trace record
    kern_s = kernel_ms / 1e3                 # sum over levels of the slowest rank's kernel time, all timed steps
    achieved = (res.distinct / world) * args.steps * b_alg / kern_s / 1e9
    peak, peak_src = peaks()
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "round2_traffic.json")  # ncu --set full dram bytes of one wide level of THIS configuration
    if os.path.exists(tpath):
        try:
            traffic = json.load(open(tpath))
        except ValueError:
            traffic = None

    probe = None
    eng.close()
    del eng
    torch.cuda.empty_cache()
    barrier()
    if rank == 0:
        # the seen-set's own ceiling (SURVEY §8d "probe_peak"): the BFS's insert routine alone on random keys, same table size
        eng_probe_out = (C.c_double * 3)()
        nkeys = 1 << 27
        rc = pkg.load_library().vsr_probe_bench(local, table_cap, nkeys, 0.5, 3, eng_probe_out)
        if rc == 0:
            peak_probes = eng_probe_out[2] / (eng_probe_out[0] / 1e3)
            ach_probes = int(st.probe_total) / (kern_s / args.steps)   # this rank's probes in the last timed step
            probe = {"unit": "probes/s", "peak": peak_probes, "achieved": ach_probes, "frac": ach_probes / peak_probes,
                     "how": "vsr_probe_bench: %d splitmix64 keys (50%% repeats) into a fresh table of %d slots with the BFS's own "
                            "insert routine, best of 3: %.3f ms; achieved = this rank's seen-set probes per kernel-second of the BFS"
                            % (nkeys, table_cap, eng_probe_out[0])}
    # e2e: the public one-call API with host buffers in and out: config text -> parse -> allocate (seen-set, frontiers, inboxes)
    # -> BFS -> stats and counterexample back in host memory -> teardown.  Allocating and clearing tens of GB varies with the
    # box's allocator state, so three runs, median reported, all three in the JSON.
    e2e_runs, e2e_states, h2d, d2h, e2e_parts = [], 0, 0, 0, None
    for _ in range(0 if (args.no_e2e or staged) else 3):
        barrier()
        te = time.time()
        if world == 1:
            r2 = pkg.ModelChecker.from_cfg_text(cfg).check(stop_on_violation=False, table_capacity=table_cap, frontier_capacity=frontier_cap)
            e2e_states, h2d, d2h = r2.distinct, r2.bytes_h2d + len(cfg), r2.bytes_d2h + C.sizeof(pkg.checker.VsrStats)
            ok = ok and r2.distinct == EXPECT["distinct"] and r2.rc == 12 and len(r2.trace) == EXPECT["violation_level"]
            e2e_parts = {"setup": r2.seconds_setup, "bfs_and_trace": r2.seconds_total - r2.seconds_setup}
        else:
            mc2 = pkg.ModelChecker.from_cfg_text(cfg)
            r2 = vdist.check_sharded(mc2, group, device=local, table_capacity=table_cap, frontier_capacity=frontier_cap, stop_on_violation=False)
            e2e_states, h2d, d2h = r2.distinct, r2.bytes_h2d + len(cfg), r2.bytes_d2h + C.sizeof(pkg.checker.VsrStats)
            ok = ok and r2.distinct == EXPECT["distinct"] and r2.rc == 12 and (rank != 0 or len(r2.trace) == EXPECT["violation_level"])
            e2e_parts = r2.call_seconds
        barrier()
        t = torch.tensor([time.time() - te], dtype=torch.float64, device=dev)
        if world > 1:
            tdist.all_reduce(t, op=tdist.ReduceOp.MAX)
        e2e_runs.append(float(t[0]))
    e2e_s = sorted(e2e_runs)[1] if e2e_runs else None

    cfg3 = None
    if (world > 1 and not args.no_cfg3 and not staged) or (world == 1 and args.cfg3_one_gpu):
        torch.cuda.empty_cache()
        try:
            cfg3 = cfg3_first_violation(pkg, vdist, torch, tdist, group, rank, world, local, dev, barrier)
        except pkg.VsrError as ex:
            cfg3 = {"error": str(ex)}

    small_gpu = None
    if world == 1 and rank == 0:
        mcs = pkg.ModelChecker.from_constants(SMALL["R"], SMALL["V"], SMALL["L"], symmetry=False)
        ts = time.time()
        rs = mcs.check(stop_on_violation=False, table_capacity=1 << 22, frontier_capacity=1 << 19)
        small_gpu = {"value": rs.distinct / (time.time() - ts), "unit": "states/s", "seconds": time.time() - ts, "kernel_seconds": rs.seconds_kernels,
                     "api": "ModelChecker.check() (engine creation and teardown included)",
                     "results_match_expected": (rs.distinct, rs.generated, rs.depth) == (SMALL["distinct"], SMALL["generated"], SMALL["depth"])}

    if rank == 0:
        wide = max(range(len(levels_ms[-1])), key=lambda i: levels_ms[-1][i]) if levels_ms and levels_ms[-1] else 0
        out = {
            "metric": "unique states explored/sec (VSR.tla, shipped VSR.cfg constants)", "value": value, "unit": "states/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * wall / args.steps,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "u32",
            "data": "none: the workload is the complete reachable state space of the config (single Init state)",
            "config": {"workload": "VSR.tla ReplicaCount=3 ClientCount=1 Values={v1,v2} StartViewOnTimerLimit=2 VIEW view SYMMETRY symmValues "
                                   "INVARIANT AcknowledgedWriteNotLost, deadlock check off, continued past the violation to the complete "
                                   "reachable set (BASELINE configs[1] = shipped VSR.cfg)",
                       "state_bytes": S, "distinct_states": res.distinct, "states_generated": res.generated, "depth": res.depth,
                       "first_violation_depth": res.violation_level, "parallelism": "fingerprint-sharded x%d" % world,
                       "exchange": "none" if world == 1 else "STAGED BASELINE: local staging buffer + NCCL send/recv per step, Python level loop" if staged else "expand_kernel stores each remote successor into the owner's inbox over NVLink "
                                   "(CUDA IPC peer mapping, TMA bulk store per destination run); the owner inserts it in its next launch; "
                                   "C++ level loop, shared-memory all-gather between ranks; NCCL only for the bench's own barrier/timing",
                       "l2": "working set (seen-set %.1f GiB per GPU) exceeds L2; no flush needed" % (table_cap * 16 / 2**30),
                       "results_match_expected": bool(ok),
                       "oracle_coverage": "GPU == CPU oracle as SETS for complete spaces <= 697k states and to a bounded depth of this config "
                                          "(tests/test_gpu_parity.py); the full-size totals are checked against the numbers every earlier run "
                                          "and every GPU count reproduced, not against an oracle run (the oracle does 4e5 states/s)",
                       "timing": "wall clock bracketed by barrier+synchronize, max over ranks; "
                       "device time between CUDA events on the launch stream = %.3f s" % (dev_ms / 1e3)},
            "gpu_launches": launches0,
            "kernel_seconds": kern_s,
            # N>1: the part of kernel_seconds spent in launches that only drain records received from peers (slowest rank per
            # level), and the records rank 0 pushed to its peers
            "kernel_seconds_insert": insert_ms / 1e3,
            "records_sent_rank0": exchanged,
            # the slowest rank's kernel time per BFS level (ms) in the last timed step, beside the level sizes
            "level_ms_last_step": [round(x, 4) for x in levels_ms[-1]] if levels_ms else [],
            "level_sizes": [int(x) for x in res.level_sizes],
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic.get("dram_bytes_per_launch") if traffic else None,
                         "traffic_note": (traffic.get("note") if traffic else "no ncu capture of this configuration committed yet (profiles/round2_traffic.json)"),
                         "peak_source": peak_src, "bytes_per_state": b_alg, "g": g,
                         "widest_level": {"depth": wide + 1, "ms": levels_ms[-1][wide] if levels_ms and levels_ms[-1] else None,
                                          "states_expanded": int(res.level_sizes[wide]) if res.level_sizes else None},
                         "kernel": "expand_kernel<Layout<3,2,3>> (per-GPU states x B_alg / sum of per-level kernel time, max over ranks)"},
            "e2e": ({"value": e2e_states / e2e_s, "unit": "states/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                     "seconds": e2e_s, "seconds_all_runs": e2e_runs,
                     # rank 0's wall clock of the LAST run by part: where the call's time goes beside the BFS itself
                     "seconds_by_part_rank0_last_run": e2e_parts,
                     "api": "ModelChecker.from_cfg_text(cfg).check()" if world == 1 else "dist.check_sharded(ModelChecker.from_cfg_text(cfg), group) on every rank"}
                    if e2e_s else None),
            "probe_roofline": probe,
            "clocks": clocks,
        }
        if cfg3 is not None:
            out["cfg3_first_violation"] = cfg3
        if small_gpu is not None:
            out["same_config_small"] = {"workload": "VSR.tla ReplicaCount=3 Values={v1,v2} StartViewOnTimerLimit=1 VIEW view, no SYMMETRY: COMPLETE state space (%d distinct states, depth %d)"
                                                    % (SMALL["distinct"], SMALL["depth"]), "gpu": small_gpu}
        if world == 1 and not args.no_cpu_baseline:
            try:
                cores = usable_cores()
                s = oracle_sample(args.cpu_seconds, cores)
                s1 = oracle_sample(min(3.0, args.cpu_seconds), 1) if cores > 1 else s
                out["cpu_baseline"] = {"value": s["rate"], "unit": "states/s", "cores": cores, "kind": "port",
                                       "single_thread_value": s1["rate"],  # the same BFS on one thread for 3 s: how far the all-core figure is from linear
                                       "sample": "CPU restatement (oracle/, not TLC) BFS of the same config for %.0f s: depth %d, %d distinct states"
                                                 % (args.cpu_seconds, s["depth"], s["distinct"])}
                out["same_config_small"]["cpu"] = small_complete_cpu(cores)
            except Exception as ex:  # the GPU line must not be lost to a failure of the reported CPU leg
                out["cpu_baseline"] = {"error": repr(ex)}
        print(json.dumps(out))
    if group is not None:
        group.close()
    if world > 1:
        tdist.destroy_process_group()


if __name__ == "__main__":
    try:
        main()
    except BaseException as ex:  # every rank's traceback must survive torchrun's summary: print it last, on stderr, and exit non-zero
        if isinstance(ex, SystemExit) and not ex.code:
            raise
        import traceback
        sys.stderr.write("\n[bench.py] rank %s failed:\n%s\n" % (os.environ.get("RANK", "0"), traceback.format_exc()))
        sys.stderr.flush()
        os._exit(1)
