#!/usr/bin/env python
"""bench.py — assignments/sec of the scheduler-tick hot path (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # CUDA path (this repo)
    python bench.py --impl reference --steps K --warmup W    # restated reference tick on the host CPU

One "step" = one scheduler tick over one batch of synthetic input, mode M1 of SURVEY.md §8(d): capacity >= demand, so
every ready task is assigned in that one tick and value = tasks / tick time.

  N = 1   BASELINE.json configs[1] (cfg2): 1 M independent ready tasks x 256 workers x 4 resource kinds (one
          fractional), Q = 16 request classes, Zipf(1.1) class mix, 8 priority levels.
  N > 1   BASELINE.json configs[4] (cfg5) shape: 1024 workers, the task table block-sharded by handle over the ranks,
          1.25 M tasks per GPU (10 M at N = 8), weak scaling.  The only exchange of a tick is the per-group count vector
          (4 B x groups per rank): NVLink peer stores issued by the tick kernel itself (default), or an NCCL all-gather
          between two kernel launches (--nccl-exchange).

  value     device-resident: the ready set already sits in HBM; the timed region holds K ticks on K different contexts
            (K + W distinct 12-15 MB task tables > the 126 MB L2, so no step re-reads a warm table); a tick = ONE
            cooperative kernel (histogram, solve, emit) that reads the worker state from pinned host memory.
  e2e       the same tick through the public C ABI with HOST buffers: hqs_ready_push (H2D of the task, class and
            priority arrays from pinned memory) + hqs_tick (D2H of the 8-byte assignments and the free vectors) inside
            the timed region.
  roofline  the tick kernel (the only kernel of a step) against MEASURED_PEAKS.json: algorithmic bytes of SURVEY.md
            §8(d)'s contract (36 B per assignment + the worker vectors) / the kernel's duration; the same with the
            interned 20 B/task budget, and the kernel's phases, are reported next to it.
  cpu_baseline / --impl reference   the oracle (restated reference tick, HiGHS 1.12.0) on the SAME workload, single-
            threaded like the reference (Rc<RefCell<Core>>), with the reference's solver defaults relaxed to a 1 % MIP gap
            and a 2 s cap (parity.ORACLE_FAST; `solver_hit_cap` says whether the cap was reached).

--dump-outputs DIR writes what the last timed step returned to its caller, so that two builds can be compared output for
output (the inputs are seeded: the same arguments give the same inputs): the assignment records as assignment_task (float64),
assignment_worker, assignment_variant, assignment_kind (float32) and the free vectors after the tick as free_after [W][R]
(float64), one DIR/<name>.npy each; with several GPUs every rank writes its own files (<name>.rank<r>.npy).  Above 64 MB in
all, a fixed seeded sample of the records is written, with their positions in assignment_row.
"""
from __future__ import annotations

import argparse
import ctypes as C
import datetime
import json
import os
import subprocess
import sys
import threading
import time
import traceback

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.dont_write_bytecode = True          # the benchmark leaves the source tree as it found it
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

N_CLASSES = 16
FREE_SCALE = 1024
METRIC = "assignments/sec on 1M ready tasks x 256 workers x 4 resource kinds"
CFG2 = {"name": "cfg2-M1", "tasks_per_gpu": 1_000_000, "workers": 256, "free_scale": 1024,
        "workload": "cfg2-M1: 1M independent tasks, 256 workers, R=4 (gpus fractional), Q=16 Zipf(1.1), 8 priorities, one tick, all assignable"}
# free_scale 4096: mode M1 needs capacity >= demand for the WHOLE job; with 1024 x the per-worker numbers the 10 M tasks of
# 8 GPUs ask for 89 % of the pool's gpus and first-fit leaves tasks behind (measured: all_assigned false, 34 k segments)
CFG5 = {"name": "cfg5-M1", "tasks_per_gpu": 1_250_000, "workers": 1024, "free_scale": 4096,
        "workload": "cfg5-M1: 1.25M independent tasks per GPU (10M at 8 GPUs) block-sharded by handle, 1024 workers, R=4 (gpus fractional), "
                    "Q=16 Zipf(1.1), 8 priorities, one tick, all assignable"}
BYTES_CONTRACT = 36      # SURVEY.md §8(d): V*R*4 amounts + 8 priority + 4 class/flags read, 8 written per assignment (cfg2, cfg5)
BYTES_INTERNED = 20      # what the path moves with interned classes: 4 key read (count) + 4 key read (emit) + 8 assignment + 4 key write-back
DUMP_BYTES = 64 << 20    # --dump-outputs: all files of all ranks together
DUMP_ROW_BYTES = 28      # one dumped record: task (8) + worker, variant, kind (4 each) + its position when sampled (8)


def dump_outputs(out_dir: str, rank: int, world: int, assignments: np.ndarray, free_after: np.ndarray) -> None:
    """Writes one step's result (assignment records, free vectors after the tick) as float .npy files (exact: handles are
    u32, the benchmark's amounts stay below 2^53).  More records than this rank's share of DUMP_BYTES: a fixed seeded
    sample of them, in output order, with their positions."""
    os.makedirs(out_dir, exist_ok=True)
    a = assignments
    arrays = {}
    rows = (DUMP_BYTES - world * (free_after.size * 8 + 1024)) // (world * DUMP_ROW_BYTES)     # 1 KB: the .npy headers
    if a.size > rows:
        idx = np.sort(np.random.default_rng(0).choice(a.size, size=rows, replace=False))
        a = a[idx]
        arrays["assignment_row"] = idx.astype(np.float64)
    arrays["assignment_task"] = a["task"].astype(np.float64)
    for f in ("worker", "variant", "kind"):
        arrays[f"assignment_{f}"] = a[f].astype(np.float32)
    arrays["free_after"] = free_after.astype(np.float64)
    sfx = f".rank{rank}" if world > 1 else ""
    for name, arr in arrays.items():
        np.save(os.path.join(out_dir, f"{name}{sfx}.npy"), arr)


def _peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler(threading.Thread):
    """Samples nvidia-smi clocks and throttle reasons while the timed region runs."""

    def __init__(self, index: int = 0) -> None:
        super().__init__(daemon=True)
        self.index = index
        self.samples = []
        self.reasons = set()
        self.sm_max = None
        self._halt = threading.Event()

    def run(self) -> None:
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        while not self._halt.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}",
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                f = [x.strip() for x in out.strip().split(",")]
                self.samples.append(float(f[0]))
                self.sm_max = float(f[1])
                for n, v in zip(names, f[2:]):
                    if v.lower().startswith("active"):
                        self.reasons.add(n)
            except Exception:
                pass
            self._halt.wait(0.1)

    def stop(self) -> dict:
        self._halt.set()
        self.join(timeout=6)
        return {"sm_mhz": float(np.median(self.samples)) if self.samples else None, "sm_max_mhz": self.sm_max,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


def make_workload(cfg: dict, seed: int, n_classes: int = N_CLASSES, free_scale=None, **kw):
    import workloads as WL          # synthetic inputs only; does not import the oracle
    fs = cfg.get("free_scale", FREE_SCALE) if free_scale is None else free_scale
    return WL.make_independent(cfg["tasks_per_gpu"], cfg["workers"], n_classes, seed=seed, free_scale=fs, **kw)


def config_block(cfg: dict, world: int, **extra) -> dict:
    """The `config` object of the JSON line: identical keys and values in the CUDA arm and in the reference arm."""
    c = {"workload": cfg["workload"], "name": cfg["name"], "tasks_per_gpu": cfg["tasks_per_gpu"], "workers": cfg["workers"],
         "classes": N_CLASSES, "pool_free_scale": cfg.get("free_scale", FREE_SCALE)}
    c.update(extra)
    return c


# ---------------------------------------------------------------------------------------------------
# reference arm / cpu baseline: the oracle on the host CPU, same workload
# ---------------------------------------------------------------------------------------------------
def oracle_step(cfg: dict, seed: int):
    """One M1 tick of the restated reference on the workload.  Returns (assignments, seconds, solver hit its cap) —
    queue construction is outside the timed region, like the HBM-resident ready set of the CUDA arm."""
    import parity as P
    wl = make_workload(cfg, seed)
    core = P.oracle_core(wl)
    core.scheduler_state.config.proactive_filling_max = 0
    # cfg2 (256 workers): the oracle's usual relaxation (1 % gap, 2 s cap).  cfg5 (1024 workers: 16.5 k variables, 1.7 M rows):
    # HiGHS has no incumbent after 2 s, the tick would schedule nothing; 20 s and a 5 % gap give one (37 s per tick)
    opts = P.ORACLE_FAST if cfg["workers"] <= 256 else dict(time_limit=20.0, mip_rel_gap=0.05, accept_incumbent=True)
    from oracle.batches import create_task_batches
    from oracle.mapping import create_task_mapping
    from oracle.solver import run_scheduling_solver
    t0 = time.perf_counter()
    # run_scheduling_inner (main.rs:40-46) stage by stage, like Core.schedule_mapping
    batches = create_task_batches(core, 0.0)
    solution = run_scheduling_solver(core, 0.0, batches, **opts)
    if not getattr(solution, "solved", True) and opts.get("time_limit"):
        # no incumbent inside the cap (the reference would schedule nothing, solver.rs:412-415): one more try with three
        # times the cap, inside the timed region — the time the reference needs to produce a schedule at all
        solution = run_scheduling_solver(core, 0.0, batches, **dict(opts, time_limit=3.0 * opts["time_limit"]))
        oracle_step.retried = getattr(oracle_step, "retried", 0) + 1
    # Mode M1 scales the pool by 1024, so one worker fits more than 1024 tasks of a class.  The reference's batch limit counts
    # at most 1024 per worker (workerload.rs:12, batches.rs:80-91); once a class's count exceeds that limit (`limit_reached`)
    # the MILP gets NO size row for it (solver.rs:245-252) and may hand out more tasks of the class than its queue holds —
    # take_tasks then unwraps an empty queue (taskqueue.rs:326) and the real server panics.  The harness keeps the tick
    # alive instead: such a class's counts are cut back (highest worker ids first) to the length of its queue.
    truncated = 0
    left = {}
    for (rq_id, v_id) in sorted(solution.sn_counts):
        counts = solution.sn_counts[(rq_id, v_id)]
        if rq_id not in left:
            left[rq_id] = sum(n for _, n in core.task_queues.get(rq_id).iter_priority_sizes())
        over = sum(counts.values()) - left[rq_id]
        for w_id in sorted(counts, reverse=True):
            if over <= 0:
                break
            cut = min(over, counts[w_id])
            counts[w_id] -= cut
            over -= cut
            truncated += cut
        for w_id in [w for w, c in counts.items() if c == 0]:
            del counts[w_id]
        left[rq_id] -= sum(counts.values())
    mapping = create_task_mapping(core, solution)
    dt = time.perf_counter() - t0
    info = getattr(core, "last_solver_info", None) or {}
    oracle_step.truncated = getattr(oracle_step, "truncated", 0) + (1 if truncated else 0)
    return mapping.n_assigned(), dt, bool(info.get("hit_time_limit", False))


def run_reference(args) -> None:
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cfg = CFG2 if args.gpus == 1 else CFG5
    # the CPU arm has no caches to warm beyond the first import: one untimed step on cfg2 (6 s), none on cfg5 (40-100 s each)
    for i in range(min(args.warmup, 1) if cfg["workers"] <= 256 else 0):
        oracle_step(cfg, 100 + i)
    # every step is the FULL workload (6-20 s of CPU work each on cfg2, more on cfg5)
    n_tot, t_tot, capped, timed = 0, 0.0, 0, 0
    for i in range(args.steps):
        n, dt, cap = oracle_step(cfg, i)
        n_tot += n
        t_tot += dt
        capped += int(cap)
        timed += 1
    value = n_tot / t_tot if t_tot > 0 else 0.0
    desc = {"value": value, "unit": "assignments/s", "cores": 1, "kind": "port",
            "sample": f"the full workload of one GPU per step ({cfg['tasks_per_gpu']} tasks, {cfg['workers']} workers, one M1 tick; the "
                      f"reference's batch limit counts at most 1024 tasks of a class per worker, workerload.rs:12); oracle = restated "
                      f"reference tick (Python + HiGHS 1.12.0 via scipy, {'1 % MIP gap, 2 s cap' if cfg['workers'] <= 256 else '5 % MIP gap, 20 s cap (no incumbent inside 2 s at 1024 workers)'}, "
                      f"cap reached in {capped} of {timed} timed steps, {getattr(oracle_step, 'retried', 0)} steps found no incumbent inside "
                      f"the cap and were solved again with three times the cap (both attempts timed); in {getattr(oracle_step, 'truncated', 0)} steps (warm-up included) the MILP "
                      f"handed out more tasks of a class than its queue holds — no size row once the 1024-per-worker batch limit is "
                      f"reached, the real server would panic in take_tasks — and the harness cut the counts back to the queue length); "
                      f"host has {os.cpu_count()} cores, 1 used (the reference tick is single-threaded)"}
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": value, "unit": "assignments/s", "n_gpus": args.gpus,
        "steps": args.steps, "steps_timed": timed, "warmup": args.warmup, "ms_per_step": 1000.0 * t_tot / max(timed, 1),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u64", "data": "synthetic",
        "config": config_block(cfg, args.gpus),
        "cpu_baseline": desc,
        "e2e": {"value": value, "unit": "assignments/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


# ---------------------------------------------------------------------------------------------------
# CUDA arm
# ---------------------------------------------------------------------------------------------------
def device_m1(P, L, wl, n_ticks: int, device: int, stream, profile: bool = False):
    """n_ticks M1 ticks of one workload on one context, re-armed in between; returns (per-tick kernel ms list, stats)."""
    import torch
    s = P.gpu_scheduler(wl, device=device)
    s._check(s._lib.hqs_set_profile(s._ctx, 1))
    out = []
    for _ in range(n_ticks + 1):
        s.free = wl.worker_free.copy()
        m = s.run_scheduling()
        ms = (C.c_float * 4)()
        s._check(s._lib.hqs_get_kernel_ms(s._ctx, ms))
        out.append((float(ms[3]), m.n_assigned()))
        s.rearm()
    st = s.stats()
    s.close()
    return out[1:], st


def drain(P, wl, device: int, max_ticks: int = 20000, dag: bool = False):
    """Mode M2: zero-duration drain through the public call (tick, finish everything, return resources)."""
    s = P.gpu_scheduler(wl, device=device)
    t0 = time.perf_counter()
    left, ticks = wl.n_tasks, 0
    while left > 0 and ticks < max_ticks:
        m = s.run_scheduling()
        if m.n_assigned() == 0:
            break
        left -= m.n_assigned()
        ticks += 1
        s.tasks_finished(m.assignments["task"], propagate=dag)
    dt = time.perf_counter() - t0
    s.close()
    return {"value": (wl.n_tasks - left) / dt, "unit": "assignments/s", "ticks": ticks, "seconds": dt,
            "ms_per_tick": 1000.0 * dt / max(ticks, 1), "assigned": wl.n_tasks - left}


def run_cuda(args) -> dict:
    import torch
    import torch.distributed as dist
    import workloads as P           # the CUDA arm never imports oracle/ (only the cpu_baseline leg below does)
    from hyperqueue_b200 import _lib as L, priority_from_user

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback); use --impl reference for the CPU arm")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank), timeout=datetime.timedelta(seconds=180))
    dev = torch.device("cuda", local_rank)
    K, Wm = args.steps, args.warmup
    n_ctx = K + Wm
    cfg = CFG2 if world == 1 else CFG5
    n_tasks, n_workers = cfg["tasks_per_gpu"], cfg["workers"]

    # one stream shared by every context so the ticks serialise and torch events time them
    stream = torch.cuda.Stream(device=dev)
    # one class table / worker pool for every rank; the ranks' task tables differ (rolled class / priority arrays)
    wl = make_workload(cfg, seed=0)
    if rank:
        wl.task_class = np.roll(wl.task_class, rank * 104729)
        wl.task_user_priority = np.roll(wl.task_user_priority, rank * 15485863 % n_tasks)
    prio = priority_from_user(wl.task_user_priority)
    task_handles = np.arange(n_tasks, dtype=np.uint32)
    scheds = []
    for i in range(n_ctx):
        s = P.gpu_scheduler(wl, add_tasks=False, device=local_rank)
        s._sync_classes()
        s._check(s._lib.hqs_set_stream(s._ctx, C.c_void_p(stream.cuda_stream)))
        lv = np.ascontiguousarray(np.unique(prio))
        s._check(s._lib.hqs_levels_add(s._ctx, lv.size, L.ptr(lv)))      # same level numbering on every rank
        # distinct device tables: rotate the class / priority arrays
        s.add_ready_tasks(task_handles, np.roll(wl.task_class, i * 7919), np.roll(prio, i * 7919))
        scheds.append(s)
    torch.cuda.synchronize()

    workers = scheds[0]._worker_structs(0.0)
    free = np.ascontiguousarray(wl.worker_free)
    total = np.ascontiguousarray(wl.worker_total)
    lib = scheds[0]._lib
    p2p = world > 1 and not args.nccl_exchange

    def launch(s):
        s._check(lib.hqs_tick_launch(s._ctx, n_workers, L.ptr(workers), L.ptr(free), L.ptr(total), None, n_tasks))

    def sharded_tick(s, bufs):
        if p2p:
            # fused: histogram -> NVLink peer stores of the count vector + release flags -> the solver acquires the flags
            # and sums the vectors -> local emit, all inside ONE kernel.  No host collective on the data path.
            s._check(lib.hqs_shard_tick_launch(s._ctx, n_workers, L.ptr(workers), L.ptr(free), L.ptr(total), None, n_tasks))
            return
        # SURVEY.md §8(e): count locally, all-gather the count vectors (NCCL), replicated solve, local emit
        cnt, gathered = bufs
        ng = C.c_uint32(0)
        s._check(lib.hqs_shard_count(s._ctx, n_workers, L.ptr(workers), L.ptr(free), L.ptr(total), None,
                                     C.c_void_p(cnt.data_ptr()), cnt.numel(), C.byref(ng)))
        with torch.cuda.stream(stream):
            dist.all_gather_into_tensor(gathered, cnt)
            g2 = gathered.view(world, -1)
            allc = g2.sum(0, dtype=torch.int64).to(torch.int32)
            before = g2[:rank].sum(0, dtype=torch.int64).to(torch.int32) if rank else torch.zeros_like(cnt)
        s._sh = (allc, before)
        s._check(lib.hqs_shard_solve_emit(s._ctx, C.c_void_p(allc.data_ptr()), C.c_void_p(before.data_ptr()), n_tasks))

    if world > 1:
        # one local (unsharded) tick per rank first: module load and first-launch costs differ between processes by
        # hundreds of milliseconds, and a sharded tick waits for its peers on the device
        warm = P.gpu_scheduler(make_workload({"tasks_per_gpu": 4096, "workers": n_workers}, seed=1), device=local_rank)
        warm.run_scheduling()
        warm.close()
        barrier_host = dist.barrier
        barrier_host()
    if p2p:
        from hyperqueue_b200.sharded import gather_peer_handles, open_and_attach
        ok = 1
        pending = [gather_peer_handles(s, rank, world) for s in scheds]          # collective: every rank, every context
        try:
            for s, (own, ipc_handles) in zip(scheds, pending):                   # local: may fail without hanging the others
                open_and_attach(s, rank, world, own, ipc_handles)
                s._check(lib.hqs_tick_reserve(s._ctx, n_workers, n_tasks, 0))
        except Exception as e:          # e.g. CUDA IPC not permitted in this container: every rank falls back together
            print(f"[bench] rank {rank}: peer-to-peer exchange unavailable ({e}); using the NCCL all-gather", file=sys.stderr)
            ok = 0
        flag = torch.tensor([ok], dtype=torch.int32, device=dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        p2p = bool(flag.item())
        dist.barrier()
    bufs = None
    if world > 1:
        with torch.cuda.stream(stream):
            bufs = (torch.zeros(L.HQS_MAX_GROUPS, dtype=torch.int32, device=dev),
                    torch.zeros(L.HQS_MAX_GROUPS * world, dtype=torch.int32, device=dev))

    def step(s):
        if world > 1:
            sharded_tick(s, bufs)
        else:
            launch(s)

    def barrier():
        # the device drains FIRST: a sharded tick is a cooperative kernel that occupies every SM and waits for its peers on
        # the device; an NCCL kernel that slips in between two ticks on one rank (and cannot start on the other, whose SMs
        # are all taken by a tick waiting for exactly that rank) would dead-lock until the tick's peer time-out
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- every context runs one untimed tick first (device buffers are allocated on the first tick),
    #      then its ready set is re-armed on the device
    out_n = C.c_uint32(0)
    tmp_out = np.zeros(n_tasks, dtype=L.assignment_dtype)
    for s in scheds:
        step(s)
        s._check(lib.hqs_tick_fetch(s._ctx, n_tasks, L.ptr(tmp_out), C.byref(out_n), None))
        s._check(lib.hqs_ready_rearm(s._ctx))
    barrier()
    # ---- warm-up, then the timed region: exactly K steps, events on the launching stream -----------
    for i in range(Wm):
        step(scheds[i])
    barrier()
    sampler = ClockSampler(local_rank)
    sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_host0 = time.perf_counter()
    ev0.record(stream)
    for i in range(K):
        step(scheds[Wm + i])
    ev1.record(stream)
    barrier()
    t_host = time.perf_counter() - t_host0
    ms_total = ev0.elapsed_time(ev1)
    launches_timed = K if (world == 1 or p2p) else 2 * K            # tick_k per step (NCCL variant: count_only_k + tick_k)
    for i in range(Wm):                 # the warm-up ticks are fetched too (a context takes one tick at a time)
        scheds[i]._check(lib.hqs_tick_fetch(scheds[i]._ctx, n_tasks, L.ptr(tmp_out), C.byref(out_n), None))
    # every step must have assigned every task of the rank
    n_done_local = 0
    free_last = np.zeros_like(free)
    for i in range(K):
        s = scheds[Wm + i]
        s._check(lib.hqs_tick_fetch(s._ctx, n_tasks, L.ptr(tmp_out), C.byref(out_n), L.ptr(free_last) if i == K - 1 else None))
        n_done_local = int(out_n.value)
        if world == 1:
            assert out_n.value == n_tasks, f"step {i}: {out_n.value} of {n_tasks} tasks assigned"
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, rank, world, tmp_out[:n_done_local], free_last)

    if world > 1:
        t = torch.tensor([ms_total], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_total = float(t.item())
        n_all = torch.tensor([n_done_local], dtype=torch.int64, device=dev)
        dist.all_reduce(n_all)
        n_per_step = int(n_all.item())
    else:
        n_per_step = n_tasks
    ms_per_step = ms_total / K
    value = n_per_step / (ms_per_step / 1000.0)

    # ---- phases of the tick kernel (profiled pass, same workload, re-armed tables) -------------------
    acc = np.zeros(4)
    for i in range(K):
        s = scheds[Wm + i]
        s._check(lib.hqs_ready_rearm(s._ctx))
        s._check(lib.hqs_set_profile(s._ctx, 1))
    barrier()
    for i in range(K):
        s = scheds[Wm + i]
        step(s)
        s._check(lib.hqs_tick_fetch(s._ctx, n_tasks, L.ptr(tmp_out), C.byref(out_n), None))
        ms = (C.c_float * 4)()
        s._check(lib.hqs_get_kernel_ms(s._ctx, ms))
        acc += np.array(list(ms))
    acc /= K
    st = scheds[Wm].stats()
    peak, peak_src = _peaks()
    worker_bytes = 2.0 * n_workers * 4 * 8
    bytes_contract = BYTES_CONTRACT * n_tasks + worker_bytes        # per launch (per GPU)
    bytes_interned = BYTES_INTERNED * n_tasks + worker_bytes
    kernel_ms = ms_per_step if (world == 1 or p2p) else float(acc[3])
    achieved = bytes_contract / kernel_ms / 1e6
    traffic = None          # dram read + write bytes of one tick_k launch from the committed ncu --set full capture
    mp = os.path.join(ROOT, "profiles", "r2_ncu_metrics.json")
    if os.path.exists(mp):
        m = json.load(open(mp)).get("tick_k")
        if m and m.get("dram_bytes_read") is not None:
            traffic = m["dram_bytes_read"] + (m.get("dram_bytes_write") or 0.0)
    roofline = {"bound": "hbm", "kernel": "tick_k (the one kernel of a tick: histogram + solve + emit)", "achieved": achieved,
                "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
                "bytes_per_assignment": BYTES_CONTRACT,
                "algorithmic_bytes_per_launch": bytes_contract,
                "kernel_ms": kernel_ms,
                "interned": {"bytes_per_assignment": BYTES_INTERNED, "achieved": bytes_interned / kernel_ms / 1e6,
                             "frac": bytes_interned / kernel_ms / 1e6 / peak,
                             "note": "classes are interned (ResourceRqId), so the path itself moves 4 B key (histogram) + 4 B key "
                                     "(emit, L2 hit) + 8 B assignment + 4 B key write-back per task"},
                "note": "SURVEY.md §8(d) contract: 36 B per assignment (un-interned amounts 16 + priority 8 + class 4 read, 8 written) "
                        "+ 2*W*R*8 B of worker vectors per tick; duration = CUDA events on the launching stream over the timed region / K"}
    kernels = {"tick_k": {"ms": float(acc[3]), "phases_ms": {"stage+histogram": float(acc[0]), "exchange+compact+solve": float(acc[1]),
                                                             "emit": float(acc[2])},
                          "groups": st["n_groups"], "segments": st["n_segments"],
                          "note": "phases as seen by the solver CTA's clock, scaled to the event-timed kernel duration; the solve is a "
                                  "sequential chain over the non-empty groups (pools of up to 512 workers: every worker a lane, one "
                                  "step per group; larger pools: one warp over tiles of 32 workers), histogram and emit stream the "
                                  "task table"}}

    extra = {}
    # ---- mode M2 (SURVEY.md §8(d)): zero-duration drains with REAL capacities, every tick through the public call;
    #      class-pool sweep and seeds (N = 1 only)
    if rank == 0 and world == 1 and not args.no_extras:
        extra["drain_m2_cfg2"] = dict(drain(P, make_workload(cfg, seed=0, free_scale=1), local_rank),
                                      note="cfg2-M2: 1M tasks, 256 workers x {128 cpus, 8 gpus, 512 GiB, 2048 GiB}; hqs_tick per tick incl. "
                                           "D2H of assignments and host-side resource return")
        extra["drain_m2_cfg3"] = dict(drain(P, make_workload(cfg, seed=0, free_scale=1, variants3=True, blocked_density=0.05), local_rank),
                                      note="cfg3-M2: as cfg2 with 3 variants per class and 5 % blocked (worker, class, variant) triples")
        t0 = time.perf_counter()
        dag = P.make_dag(500_000, 256, N_CLASSES, seed=0)
        extra["drain_m2_cfg4"] = dict(drain(P, dag, local_rank, dag=True),
                                      note=f"cfg4-M2: 500k-node DAG (fan-in <= 8, b-level priorities), one tick per completion wave; ticks = waves "
                                           f"(DAG built on the host in {time.perf_counter() - t0:.1f} s, outside the timed region)")
        sweep = {}
        for q in (1, 16, 256, 4096):
            w2 = make_workload(cfg, seed=0, n_classes=q)
            res, st2 = device_m1(P, L, w2, 3, local_rank, stream)
            ms_med = float(np.median([r[0] for r in res]))
            sweep[f"Q={q}"] = {"kernel_ms": ms_med, "value": res[0][1] / (ms_med / 1e3), "assigned": res[0][1], "classes": len(w2.classes),
                               "groups": st2["n_groups"], "levels": st2["n_levels"], "coarsened": st2["coarsened"]}
        extra["class_pool_sweep_m1"] = dict(sweep, note="one context, kernel time by CUDA events (warm task table); Q > 512 exceeds "
                                                        "HQS_MAX_GROUPS / 8 levels, so the priority levels are coarsened (stat `coarsened`)")
        seeds = {}
        for sd in (0, 1, 2):
            res, _ = device_m1(P, L, make_workload(cfg, seed=sd), 3, local_rank, stream)
            seeds[str(sd)] = float(np.median([r[1] / (r[0] / 1e3) for r in res]))
        extra["seeds_m1"] = {"per_seed_value": seeds, "median": float(np.median(list(seeds.values()))),
                             "note": "cfg2-M1 with seeds 0/1/2, one context each (warm table), assignments/s by kernel time"}

    # ---- e2e: host buffers through the public C ABI -----------------------------------------------
    #      every step: this rank's tasks host -> device (hqs_ready_push), the tick, its assignments device -> host
    s = scheds[0]
    pin = lambda a: torch.from_numpy(np.ascontiguousarray(a)).pin_memory().numpy()
    h_cls, h_prio = pin(wl.task_class), pin(prio)
    out = torch.empty(n_tasks * 8, dtype=torch.uint8).pin_memory().numpy().view(L.assignment_dtype)
    free_after = np.zeros_like(free)
    n_e2e = K

    def e2e_step():
        # the rank's tasks are one task array (consecutive handles): class ids and priorities cross PCIe, the handles do not
        s._check(lib.hqs_ready_push_range(s._ctx, 0, n_tasks, L.ptr(h_cls), L.ptr(h_prio)))
        if world == 1:
            s._check(lib.hqs_tick(s._ctx, n_workers, L.ptr(workers), L.ptr(free), L.ptr(total), None, n_tasks,
                                  L.ptr(out), C.byref(out_n), L.ptr(free_after)))
            assert out_n.value == n_tasks
        else:
            if p2p:
                s._check(lib.hqs_shard_tick_launch(s._ctx, n_workers, L.ptr(workers), L.ptr(free), L.ptr(total), None, n_tasks))
            else:
                sharded_tick(s, bufs)
            s._check(lib.hqs_tick_fetch(s._ctx, n_tasks, L.ptr(out), C.byref(out_n), L.ptr(free_after)))
    for _ in range(3):
        e2e_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(n_e2e):
        e2e_step()
    barrier()
    dt = (time.perf_counter() - t0) / n_e2e
    n_step = n_tasks
    if world > 1:
        tt = torch.tensor([dt], dtype=torch.float64, device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        dt = float(tt.item())
        nn = torch.tensor([int(out_n.value)], dtype=torch.int64, device=dev)
        dist.all_reduce(nn)
        n_step = int(nn.item())
    e2e = {"value": n_step / dt, "unit": "assignments/s", "ms_per_step": dt * 1000.0, "steps": n_e2e,
           "h2d_bytes_per_step": int(world * (n_tasks * 12 + free.nbytes + total.nbytes + workers.nbytes)),
           "d2h_bytes_per_step": int(n_step * 8 + world * (free.nbytes + 16)), "n_gpus": world,
           "note": "per rank: hqs_ready_push_range (4 B class id + 8 B priority per task) + tick + fetch (8 B per assignment) with pinned "
                   "host buffers; host clock between barriers, max over ranks"}
    clocks = sampler.stop()

    # ---- CPU baseline (rank 0, N=1 only): the oracle on the same workload ---------------------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        n, dtc, cap = oracle_step(cfg, 0)
        cpu = {"value": n / dtc, "unit": "assignments/s", "cores": 1, "kind": "port",
               "sample": f"one M1 tick of the restated reference (Python + HiGHS 1.12.0, 1 % MIP gap, 2 s cap{' reached' if cap else ' not reached'}) on the "
                         f"full workload ({n_tasks} tasks, {n_workers} workers): {n} assignments (the reference's batch limit counts at most 1024 "
                         f"tasks of a class per worker) in {dtc:.1f} s; host has {os.cpu_count()} cores, 1 used"}

    result = None
    if rank == 0:
        result = {
            "metric": METRIC, "value": value, "unit": "assignments/s", "n_gpus": world, "steps": K, "warmup": Wm,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u64", "data": "synthetic",
            "config": config_block(cfg, world, all_assigned=bool(n_per_step == world * n_tasks),
                                   exchange=("p2p" if p2p else ("nccl" if world > 1 else "none")),
                                   l2_policy=f"each timed step runs on a different task table (K+W tables x {12 * n_tasks // 1_000_000} MB "
                                             "> 126 MB L2): inputs larger than L2",
                                   host_wall_ms_per_step=1000.0 * t_host / K),
            "gpu_launches": launches_timed, "clocks": clocks, "e2e": e2e, "roofline": roofline, "kernels": kernels,
            "cpu_baseline": cpu, "extra": extra,
        }
    for s in scheds:
        s.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return result


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20, help="timed steps (the e2e figure times as many)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="cuda", choices=["cuda", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the M2 drains, the class-pool sweep and the seed sweep")
    ap.add_argument("--no-drain", action="store_true", help="alias of --no-extras")
    ap.add_argument("--nccl-exchange", action="store_true",
                    help="N > 1: all-gather the count vectors with NCCL instead of the fused peer-to-peer exchange")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the last timed step's assignments and free vectors as DIR/<name>.npy (CUDA arm)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "cuda":
        ap.error("--dump-outputs writes the CUDA arm's outputs")
    args.no_extras = args.no_extras or args.no_drain
    args.warmup = max(args.warmup, 3) if args.impl == "cuda" else args.warmup
    rank = int(os.environ.get("RANK", "0"))
    try:
        if args.impl == "reference":
            run_reference(args)
        else:
            res = run_cuda(args)
            if res is not None:
                print(json.dumps(res))
    except BaseException as e:          # every rank reports its own failure; rank 0 still prints one JSON line
        if isinstance(e, SystemExit) and e.code in (0, None):
            raise
        tb = traceback.format_exc()
        sys.stderr.write(tb)
        msg = f"{type(e).__name__}: {e}"
        if rank == 0:
            print(json.dumps({"metric": METRIC, "impl": args.impl, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
                              "value": None, "error": msg, "traceback_tail": tb.strip().splitlines()[-6:]}))
        sys.stdout.flush()
        sys.stderr.write(f"[bench] rank {rank} failed: {msg}\n")
        sys.stderr.flush()
        os._exit(1)


if __name__ == "__main__":
    main()
