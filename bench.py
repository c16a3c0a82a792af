#!/usr/bin/env python
"""bench.py -- batched BFGS step! throughput (BASELINE.json configs[1]) + n=16384 step! roofline.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

Workload (N=1): 1,000,000 independent extended-Rosenbrock problems, n=16, x0 = 4u-2 with u from
the reference's PCG (legacy/PCG.jl, seed 2024+rank), initial step 1.0.  One "step" = one step!
call on every problem of the batch = ONE launch of bfgs_batched_hybrid_kernel.  For N>1 every rank
holds its own 1M problems (weak scaling, no collective on the data path).

Numbers on the JSON line
  value     active problem-steps/s, state resident in HBM, CUDA events on the launching stream
  e2e       the README loop through the public API with HOST buffers: constructor from pinned
            host x0 (H2D) + K x [step!; read has_converged[] and current_objective_value[] (D2H)];
            e2e.with_point_readback adds the final current_point read (128 MB D2H)
  roofline  the batched kernel against the measured HBM copy bandwidth; achieved = algorithmic bytes
            of the step kinds the kernel itself counted in the timed launches (BFGS-type with /
            without an H read, gradient-descent, terminate, idle) / time -- reproducible from the line
  batched_strong   the SAME 1,000,000 problems split over the N GPUs (BASELINE configs[1] as written)
  large_n   n=16384 single-problem step! (configs[2]): ms per BFGS-type step (>= 50 of them), achieved
            GB/s of the 24 n^2-byte step and of its two n^2 kernels against the same peak
  sharded_large_n  n=65536 (configs[3]): the inverse Hessian row-sharded over the N GPUs (32 GiB on one
            GPU at N=1), both gather modes, with an in-run bitwise check of the sharded result at n=8192
  riesz_gd  config 5 with its FP64-pipe roofline
  cpu_baseline  the CPU oracle (a port of the reference: the reference itself is commented-out
            Julia and no Julia exists here) on all host threads, bounded sample

--dump-outputs DIR writes, after the timed steps, what the last timed step! left in its batch (see dump_outputs) as
DIR/<field>.npy.  The inputs depend only on the arguments, so two builds can be compared output for output.
The benchmark writes nothing into the source tree: the CPU arm's native oracle build goes to a temporary directory.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # no __pycache__ in the tree (it may be read-only)

N_SMALL = 16
BATCH = 1_000_000
LARGE_N = 16384
SHARDED_N = 65536
SHARDED_CHECK_N = 8192
STEPS_PER_BATCH = 25            # timed step! calls per batch (a batch converges within ~100 calls: see device_timed)
METRIC = "batched BFGS problem-steps/s (1M x n=16)"
UNIT = "problem-steps/s"
DUMP_PROBLEMS = 65536           # --dump-outputs: problems of the last timed batch written out (a fixed, seeded sample)
DUMP_SEED = 0


def bytes_by_kind(n, lazy=True):
    """ALGORITHMIC bytes one batched problem-step must move, by what the step does (DESIGN.md section 3).
    Every active problem reads x, g, d (3 x 8n) and f, L, iteration_count, has_terminated (25 B; +1 B for the
    "H is the identity" flag of the lazy layout) and, if it moves, writes x, g, d, dx, dg (5 x 8n) and f, L,
    iteration_count, last_step_type (28 B).  The 8n^2-byte inverse Hessian is read only by a BFGS-type step whose H is
    not the identity and written only by a BFGS-type step; a gradient-descent step leaves H = I implicit (lazy) or
    writes it (round-1 layout).  A step! on a terminated problem reads its flag."""
    vec, H = 8 * n, 8 * n * n
    rd = 3 * vec + 25 + (1 if lazy else 0)
    wr = 5 * vec + 28
    return {"bfgs_read_h": rd + H + wr + H,
            "bfgs_identity_h": rd + wr + H + (1 if lazy else 0),
            "gradient_descent": rd + wr + ((1 if lazy else H)),
            "terminate": rd + 1,
            "idle": 1, "idle_warp": 1}


def batched_bytes(kinds, n, lazy=True):
    table = bytes_by_kind(n, lazy)
    return float(sum(table[k] * kinds.get(k, 0) for k in table))



def load_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_traffic(kernel):
    """The committed ncu capture of `kernel` (profiles/ncu_traffic.json): {"dram_bytes_per_launch", "timed_step_index",
    "source", ...} or None.  timed_step_index = which step! of bench.py's timed region the captured launch was."""
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as f:
            return json.load(f)[kernel]
    except Exception:
        return None


def oracle_mod():
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import oracle
    oracle.build()
    return oracle


def x0_batch(gen, batch, seed):
    """gen: anything with pcg_fill(count, seed) -- the product package in the GPU arm, the oracle in the reference arm"""
    return (4.0 * gen.pcg_fill(batch * N_SMALL, seed) - 2.0).reshape(batch, N_SMALL)


def dump_outputs(opt, out_dir):
    """--dump-outputs DIR: the fields a caller of step! reads, as the last timed step! left them in its batch, for the
    same DUMP_PROBLEMS problems of the batch in every run (their indices in problem_index.npy), one float64 .npy per
    field, 28 MB in all.  Fields with n = 16 values per problem have shape (DUMP_PROBLEMS, 16), the others (DUMP_PROBLEMS,)."""
    rows = np.sort(np.random.default_rng(DUMP_SEED).choice(BATCH, DUMP_PROBLEMS, replace=False))
    fields = {"current_point": opt.current_point, "current_gradient": opt.current_gradient,
              "next_step_direction": opt.next_step_direction, "current_objective_value": opt.current_objective_value,
              "last_step_length": opt.last_step_length, "last_step_type": opt.last_step_type,
              "iteration_count": opt.iteration_count, "has_converged": opt.has_converged}
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "problem_index.npy"), rows.astype(np.float64))
    for name, a in fields.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.asarray(a)[rows].astype(np.float64))


class ClockSampler:
    """SM clock + throttle reasons DURING the timed region (B200_PROFILING.md): NVML polled every
    2 ms from a thread (nvidia-smi's fastest loop is too coarse for a 30 ms region)."""

    def __init__(self, index):
        self.index, self.rows, self.stop = index, [], False
        self.nvml = None
        self.max_mhz = None

    def __enter__(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            # CUDA_VISIBLE_DEVICES may renumber devices; resolve through the PCI bus id of the torch device
            import torch
            bus = torch.cuda.get_device_properties(self.index).pci_bus_id if hasattr(
                torch.cuda.get_device_properties(self.index), "pci_bus_id") else None
            h = None
            if bus is not None:
                for i in range(pynvml.nvmlDeviceGetCount()):
                    hh = pynvml.nvmlDeviceGetHandleByIndex(i)
                    if pynvml.nvmlDeviceGetPciInfo(hh).bus == bus:
                        h = hh
                        break
            if h is None:
                h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.nvml, self.h = pynvml, h
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
            self.t = threading.Thread(target=self._poll, daemon=True)
            self.t.start()
        except Exception:
            self.nvml = None
        return self

    def _poll(self):
        nv = self.nvml
        while not self.stop:
            try:
                self.rows.append((nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM),
                                  nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                                  if hasattr(nv, "nvmlDeviceGetCurrentClocksEventReasons")
                                  else nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)))
            except Exception:
                pass
            time.sleep(0.002)

    def __exit__(self, *a):
        self.stop = True
        if self.nvml:
            self.t.join(timeout=1)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": [], "samples": 0}
        bits = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}
        reasons = set()
        for _, r in self.rows:
            for b, nm in bits.items():
                if r & b:
                    reasons.add(nm)
        return {"sm_mhz": float(np.median([c for c, _ in self.rows])), "sm_max_mhz": self.max_mhz,
                "reasons": sorted(reasons), "samples": len(self.rows)}


# ----------------------------------------------------------------------------- CPU legs
def pin_host_threads():
    """A fair, stable CPU arm (round-1 review): every host core, explicitly.  torchrun exports OMP_NUM_THREADS=1 and the
    launcher may have narrowed the affinity mask; the oracle takes its thread count as an argument (num_threads
    clauses), but libgomp reads its placement policy from the environment when it is first loaded."""
    threads = os.cpu_count() or 1
    try:
        os.sched_setaffinity(0, range(threads))
    except Exception:
        pass
    os.environ["OMP_NUM_THREADS"] = str(threads)
    os.environ.setdefault("OMP_PROC_BIND", "close")
    os.environ.setdefault("OMP_PLACES", "cores")
    os.environ.setdefault("OMP_DYNAMIC", "false")
    return threads


def bind_to_gpu_numa_node(torch, index):
    """Multi-rank runs: keep this rank's host threads -- and with them the first-touch placement of its page-locked x0 and
    field buffers -- on the NUMA node its GPU hangs off (what `numactl --cpunodebind` does for a user).  Round-2 phase
    timers of an 8-rank run: constructors (128 MB of x0 over PCIe each) took 6.5 ms on ranks 0-3 and 4.4 ms on ranks 4-7
    against 2.9 ms alone.  Returns a description for the JSON line, or None when sysfs does not say."""
    try:
        props = torch.cuda.get_device_properties(index)
        bus = "%04x:%02x:%02x.0" % (props.pci_domain_id, props.pci_bus_id, props.pci_device_id)
        with open("/sys/bus/pci/devices/%s/numa_node" % bus) as f:
            node = int(f.read().strip())
        if node < 0:
            return None
        with open("/sys/devices/system/node/node%d/cpulist" % node) as f:
            cpus = set()
            for part in f.read().strip().split(","):
                lo, _, hi = part.partition("-")
                cpus.update(range(int(lo), int(hi or lo) + 1))
        allowed = cpus & os.sched_getaffinity(0)
        if not allowed:
            return None
        os.sched_setaffinity(0, allowed)
        return {"numa_node": node, "cpus": len(allowed)}
    except Exception:
        return None


def cpu_leg(orc, steps, warmup, sample_batch, flags):
    """Oracle (port of the reference path) on every host thread; bounded sample of the workload.  Timed twice, the
    faster pass is reported (the direction that favours the CPU arm)."""
    threads = os.cpu_count() or 1
    nb = -(-steps // STEPS_PER_BATCH)
    x0s = [x0_batch(orc, sample_batch, 2024 + 1000 * b) for b in range(nb)]      # same batches as the GPU arm (rank 0)
    best = None
    for _ in range(2):
        refs = [orc.BFGS(orc.OBJ_ROSENBROCK, x0, 1.0, order=orc.SEQ, nthreads=threads) for x0 in x0s]
        for ref in refs:
            ref.step(warmup)
        active0 = refs[0].count_active()
        t0 = time.perf_counter()
        done = 0
        for i in range(steps):
            ref = refs[i // STEPS_PER_BATCH]
            done += ref.count_active()
            ref.step(1)
        dt = time.perf_counter() - t0
        for ref in refs:
            ref.close()
        if best is None or dt < best[0]:
            best = (dt, done, active0)
    dt, done, active0 = best
    return {"value": done / dt, "unit": UNIT, "cores": threads, "kind": "port",
            "sample": f"{sample_batch} of the {BATCH} problems of each batch (same PCG streams), {steps} step! calls over {nb} batch(es) after {warmup} warm-up each, "
                      f"{active0} active at start, best of 2 passes; oracle/dzo_oracle.c built here with '{flags}' "
                      f"(bit-identical to the -O2 checker build), OpenMP over problems, threads pinned",
            "seconds": dt, "ms_per_step": 1e3 * dt / steps}


def readme_gap(orc):
    """BASELINE configs[0] on this host: the port's time per README n=2 optimisation next to the reference's own
    published figure, so nobody reads `vs_reference` as "vs Julia" (round-1 review)."""
    x0 = np.stack([orc.pcg_fill(2, s) for s in range(1000)])
    best = None
    for _ in range(3):
        t0 = time.perf_counter()
        ref = orc.BFGS(orc.OBJ_ROSENBROCK, x0, 1.0, order=orc.SEQ, nthreads=1)
        while ref.count_active():
            ref.step(16)
        dt = time.perf_counter() - t0
        ref.close()
        best = dt if best is None else min(best, dt)
    us = 1e6 * best / 1000
    return {"port_us_per_optimisation": us, "reference_published_us": {"min": 2.8, "median": 5.563},
            "port_over_published_median": us / 5.563,
            "note": "README.md:62-63 (Julia, unspecified CPU) vs the C port on one core of this host, 1000 PCG starts, "
                    "constructor included; divide vs_reference by this ratio for an estimate against tuned Julia"}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    pin_host_threads()
    orc = oracle_mod()
    flags = orc.use_native_build()
    sample = 100_000
    leg = cpu_leg(orc, args.steps, args.warmup, sample, flags)
    line = {
        "impl": "reference", "metric": METRIC, "value": leg["value"], "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": leg["ms_per_step"], "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": "batched BFGS 1,000,000 x n=16 extended Rosenbrock (BASELINE configs[1])",
                   "sample_batch": sample, "note": "reference = CPU oracle port (Julia reference is dead code; no Julia here)"},
        "cpu_baseline": {k: leg[k] for k in ("value", "unit", "cores", "kind", "sample")},
        "e2e": {"value": leg["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "readme_rosenbrock_n2": readme_gap(orc),
    }
    print(json.dumps(line))


# ----------------------------------------------------------------------------- GPU arm
def run_gpu(args):
    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    distributed = world > 1
    torch.cuda.set_device(local_rank)
    numa = None
    if distributed:
        if not args.no_numa_bind:
            numa = bind_to_gpu_numa_node(torch, local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    import dzopt_b200 as dz
    EF = dz.ExampleFunctions
    for kv in args.tune:
        k, v = kv.split("=")
        dz.set_tuning(k, int(v))
    # the checker: only the cpu_baseline legs and the sharded bitwise check below touch it (inputs come from the
    # product's own dz.pcg_fill)
    want_cpu = (rank == 0 and not args.skip_cpu)
    orc = None
    cpu_flags = None
    if want_cpu:
        if not distributed:
            pin_host_threads()      # (multi-rank runs keep the NUMA binding; their only oracle use is the small sharded check)
        orc = oracle_mod()
        cpu_flags = orc.use_native_build()
    peak, peak_src = load_peaks()
    K, W = args.steps, args.warmup
    launches = 0                      # kernels of this library launched inside timed regions (all legs, this rank)

    def barrier():
        if distributed:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(v):
        if not distributed:
            return v
        t = torch.tensor([v], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(v):
        if not distributed:
            return v
        t = torch.tensor(np.atleast_1d(np.asarray(v, dtype=np.float64)), dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        out = t.cpu().numpy()
        return float(out[0]) if np.ndim(v) == 0 else out

    stream = torch.cuda.Stream()      # a real (non-default) stream: handle 0 would mean "the handle's own stream"
    torch.cuda.set_stream(stream)
    lazy = True
    KINDS = dz.BFGSOptimizer.STEP_KINDS

    def make(x0_host):
        o = dz.BFGSOptimizer(EF.rosenbrock_function, EF.rosenbrock_gradient_, x0_host, 1.0, batched=True, device=local_rank)
        o.set_stream(stream.cuda_stream)
        return o

    def device_timed(x0_list, dump_dir=None):
        """K back-to-back step! launches after W warm-up steps per batch.  A batch of this workload converges within ~100
        step! calls, so K > STEPS_PER_BATCH launches walk through ceil(K / STEPS_PER_BATCH) independent batches of the same
        synthetic workload (each constructed and warmed up before the clock starts): every timed launch is a step! in
        the regime the metric is quoted on, however long the timed region.  Returns (ms max over ranks, kind counts of
        this rank summed over the batches, clock sampler).  With dump_dir, the batch of the last timed launch is written
        there after the clock stops (dump_outputs)."""
        opts = [make(x) for x in x0_list]
        for o in opts:
            o.step(W)
            o.step_kind_counts(reset=True)
        barrier()
        with ClockSampler(local_rank) as clk:
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            barrier()
            ev0.record(stream)
            for i in range(K):
                opts[i // STEPS_PER_BATCH].step_async(1)
            ev1.record(stream)
            barrier()
            ms = ev0.elapsed_time(ev1)
        if dump_dir is not None:
            dump_outputs(opts[(K - 1) // STEPS_PER_BATCH], dump_dir)
        kinds = {}
        for o in opts:
            for k, v in o.step_kind_counts().items():
                kinds[k] = kinds.get(k, 0) + v
            o.close()
        return max_over_ranks(ms), kinds, clk

    def e2e_timed(x0_list, read_point):
        """the README loop through the public API with HOST buffers (constructor H2D + per-step field reads), once per
        batch of the timed region.  Also returns this rank's host-side phase times (ms): constructor, warm-up call,
        step! calls, field reads, final point read."""
        barrier()
        barrier()
        ph = {"constructor": 0.0, "warmup_call": 0.0, "step_calls": 0.0, "field_reads": 0.0, "point_read": 0.0}
        now = time.perf_counter
        t1 = now()
        opts, flags_last, d2h, point_bytes, left = [], [], 0, 0, K
        for x0_host in x0_list:
            ta = now()
            e2 = dz.BFGSOptimizer(EF.rosenbrock_function, EF.rosenbrock_gradient_, x0_host, 1.0, batched=True,
                                  device=local_rank)       # H2D of x0 inside the timed region
            e2.reuse_host_buffers(True)                     # cached page-locked field arrays; has_converged / objective become
                                                            # zero-copy mirrors the step kernel writes over PCIe while it runs
            tb = now()
            e2.step(W)                                      # same starting state as the device-timed arm
            tc = now()
            ph["constructor"] += tb - ta
            ph["warmup_call"] += tc - tb
            flags = obj = None
            for _ in range(min(left, STEPS_PER_BATCH)):
                td = now()
                dz.step_(e2)
                te = now()
                flags = e2.has_converged                    # D2H, what `while !opt.has_converged[]` reads
                obj = e2.current_objective_value            # D2H
                tf = now()
                ph["step_calls"] += te - td
                ph["field_reads"] += tf - te
            left -= STEPS_PER_BATCH
            if read_point:
                tg = now()
                point_bytes += e2.current_point.nbytes      # the answer itself (D2H, n x batch doubles)
                ph["point_read"] += now() - tg
            d2h = flags.nbytes + obj.nbytes
            opts.append(e2)
            flags_last.append(flags)
        torch.cuda.synchronize()
        secs = now() - t1
        # every step! of an active problem either moves it (iteration_count + 1) or terminates it; the
        # warm-up steps of this arm are inside its timed region and count as work too
        steps_total = 0.0
        for e2, flags in zip(opts, flags_last):
            steps_total += float(e2.iteration_count.sum() + flags.sum())
            e2.close()
        ph = {k: 1e3 * v for k, v in ph.items()}
        ph["total"] = 1e3 * secs
        if distributed:
            box = [None] * world
            dist.all_gather_object(box, ph)
            ph = {"per_rank": box}
        return max_over_ranks(secs), sum_over_ranks(steps_total), d2h, point_bytes, ph

    # ================================================================== main metric: weak scaling, 1M problems per GPU
    nbatches = -(-K // STEPS_PER_BATCH)
    x0_hosts = [torch.from_numpy(x0_batch(dz, BATCH, 2024 + rank + 1000 * b)).pin_memory().numpy() for b in range(nbatches)]
    x0_host = x0_hosts[0]
    x0 = x0_host
    ms, kinds, clk = device_timed(x0_hosts, dump_dir=args.dump_outputs if rank == 0 else None)
    launches += K
    active_steps = float(sum(kinds[k] for k in ("bfgs_read_h", "bfgs_identity_h", "gradient_descent", "terminate")))
    total_problem_steps = sum_over_ranks(active_steps)
    value = total_problem_steps / (ms * 1e-3)
    kernel_ms = ms / K
    alg_bytes = batched_bytes(kinds, N_SMALL, lazy)            # this rank's launches
    achieved = alg_bytes / K / (kernel_ms * 1e-3) / 1e9
    active_frac = active_steps / (K * BATCH)

    # per-step kind mix of the same W+K steps (untimed replay, counters read after every step!) -- makes the
    # convergence tail visible and lets the ncu capture of one launch be compared with ITS algorithmic bytes
    per_step = None
    if rank == 0:
        rp = make(x0_host)
        per_step = []
        for i in range(W + min(K, STEPS_PER_BATCH)):
            rp.step_kind_counts(reset=True)
            rp.step(1)
            c = rp.step_kind_counts()
            per_step.append([c[k] for k in KINDS[:4]] + [c["idle"] + c["idle_warp"]])
        rp.close()

    # ---- k step! calls fused into ONE launch (SURVEY 8d: "report also with k fused steps per launch")
    fused = None
    if rank == 0 and not args.skip_large:
        kf = 50
        f_opt = make(x0_host)
        f_opt.step(W)
        f_opt.step_kind_counts(reset=True)
        fe0, fe1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        fe0.record(stream); f_opt.step_async(kf); fe1.record(stream)
        torch.cuda.synchronize()
        f_ms = fe0.elapsed_time(fe1)
        fk = f_opt.step_kind_counts()
        f_steps = float(sum(fk[k] for k in KINDS[:4]))
        fused = {"k": kf, "launches": 1, "ms": f_ms, "problem_steps": f_steps, "problem_steps_per_s": f_steps / (f_ms * 1e-3),
                 "still_active_after": int(f_opt.count_active())}
        f_opt.close()
        launches += 1

    # ---- end to end through the public API with host buffers
    # one untimed pass of the same code path first: fills the device memory pool and the recycled page-locked
    # field buffers (page-locking costs 10-40 ms on this virtualised host), like the W warm-up steps do for kernels
    _, _, _, _, e2e_first_pass = e2e_timed(x0_hosts, read_point=True)
    e2e_s, e2e_steps, d2h, _, e2e_phases = e2e_timed(x0_hosts, read_point=False)
    e2e_value = e2e_steps / e2e_s
    e2p_s, e2p_steps, _, point_bytes, _ = e2e_timed(x0_hosts, read_point=True)
    launches += 2 * (K + nbatches * (W + 1))
    h2d = nbatches * x0.nbytes / (K + nbatches * W)

    # ================================================================== strong scaling: the SAME 1M problems over N GPUs
    strong = None
    if distributed:
        share = BATCH // world
        lo = rank * share
        hi = BATCH if rank == world - 1 else lo + share
        xs_all = x0_batch(dz, BATCH, 2024)                 # the single-GPU problem set (seed 2024), every rank its slice
        xs = torch.from_numpy(np.ascontiguousarray(xs_all[lo:hi])).pin_memory().numpy()
        xs_list = [xs] + [torch.from_numpy(np.ascontiguousarray(x0_batch(dz, BATCH, 2024 + 1000 * b)[lo:hi])).pin_memory().numpy()
                          for b in range(1, nbatches)]
        s_ms, s_kinds, _ = device_timed(xs_list)
        launches += K
        s_active = float(sum(s_kinds[k] for k in KINDS[:4]))
        s_total = sum_over_ranks(s_active)
        s_bytes = batched_bytes(s_kinds, N_SMALL, lazy)
        e2e_timed(xs_list, read_point=False)               # untimed pass of the same code path (see above)
        se_s, se_steps, _, _, _ = e2e_timed(xs_list, read_point=False)
        launches += K + nbatches * (W + 1)
        strong = {"batch_total": BATCH, "batch_per_gpu": hi - lo, "n_gpus": world, "ms_per_step": s_ms / K,
                  "problem_steps_per_s": s_total / (s_ms * 1e-3),
                  "per_gpu_achieved_gbs": s_bytes / K / (s_ms / K * 1e-3) / 1e9,
                  "per_gpu_frac_of_peak": s_bytes / K / (s_ms / K * 1e-3) / 1e9 / peak,
                  "e2e_problem_steps_per_s": se_steps / se_s,
                  "limiter": "per-launch tail: a launch is %d CTAs = %.1f waves of 148 SMs x 4 CTAs, the last partial wave and "
                             "the ~5 us launch latency are a larger share of a %.0f us step than of the 1M-problem one; "
                             "e2e additionally pays N constructors' H2D through one host" % (
                                 -(-(hi - lo) // 128), (hi - lo) / 128 / (148 * 4), 1e3 * s_ms / K)}

    # ---- large-n step! (configs[2]) and its two n^2 kernels, rank 0 only
    large = None
    if rank == 0 and not args.skip_large:
        large = bench_large(dz, orc, torch, stream, peak, local_rank, cpu=want_cpu and world == 1)
        launches += large.pop("_launches", 0)

    # ---- row-sharded n=65536 (configs[3]) at every N: all ranks
    sharded = None
    if not args.skip_large:
        sharded = bench_sharded(dz, orc, torch, dist if distributed else None, stream, peak, rank, world, local_rank)
        launches += sharded.pop("_launches", 0) if sharded else 0

    riesz = None
    if rank == 0 and not args.skip_large:
        riesz = bench_riesz(dz, orc, torch, stream, local_rank, cpu=want_cpu and world == 1)
        launches += 1
    readme = bench_readme(dz, orc) if (want_cpu and world == 1) else None
    lbfgs = bench_lbfgs(dz, orc, torch, stream, cpu=want_cpu and world == 1) if (rank == 0 and not args.skip_large) else None
    pairwise = bench_pairwise(dz, orc, torch, cpu=want_cpu and world == 1) if (rank == 0 and not args.skip_large) else None

    cpu = None
    if want_cpu and world == 1:
        cpu = cpu_leg(orc, K, W, args.cpu_sample, cpu_flags)
        cpu = {k: cpu[k] for k in ("value", "unit", "cores", "kind", "sample")}

    if rank == 0:
        table = bytes_by_kind(N_SMALL, lazy)
        traffic = ncu_traffic("bfgs_batched_hybrid_kernel<16>")
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": kernel_ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": {"workload": "batched BFGS 1,000,000 x n=16 extended Rosenbrock per GPU (BASELINE configs[1])",
                       "batch_per_gpu": BATCH, "n": N_SMALL, "initial_step_length": 1.0,
                       "batches_in_timed_region": nbatches, "steps_per_batch": STEPS_PER_BATCH,
                       "batches_note": "a batch converges within ~100 step! calls; K > %d timed launches walk through "
                                       "independent batches of the same workload (PCG seed 2024 + rank + 1000 b), each "
                                       "constructed and warmed up W steps before the clock starts (e2e: inside it)" % STEPS_PER_BATCH,
                       "l2": "state per GPU = 2.9 GB >> 126 MB L2 (inputs larger than L2, no flush needed)",
                       "active_fraction_in_timed_region": active_frac, "timed_region_ms": ms,
                       "parallelism": f"independent problems, {world} GPU(s), no collective",
                       "host_numa_binding_rank0": numa},
            "clocks": clk.summary(),
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "host_phases_ms": e2e_phases, "untimed_first_pass_host_phases_ms": e2e_first_pass,
                    "with_point_readback": {"value": e2p_steps / e2p_s, "unit": UNIT, "extra_d2h_bytes_total": point_bytes,
                                            "what": "the same loop followed by ONE current_point read (the answer)"},
                    "what": "BFGSOptimizer(host x0) + W+K x [step!; has_converged[]; current_objective_value[]] via the C ABI; the two fields reach the host as zero-copy mirrors (dzo_bfgs_mirror_fields): the step kernel stores them into page-locked host memory, the reads only synchronise"},
            "gpu_launches": K,
            "gpu_launches_what": "one bfgs_batched_hybrid_kernel<16> per step! in the timed region of `value`",
            "gpu_launches_all_timed_legs": launches,
            "roofline": {"bound": "hbm", "kernel": "bfgs_batched_hybrid_kernel<16>", "achieved": achieved, "peak": peak,
                         "unit": "GB/s", "frac": achieved / peak,
                         "how": "achieved = sum_kind(count_kind x bytes_kind) / K launches / ms_per_step; counts come from "
                                "the kernel's own per-launch counters over exactly the timed launches (rank 0)",
                         "step_kinds_in_timed_region": kinds, "bytes_per_problem_step_by_kind": table,
                         "algorithmic_bytes_per_launch": alg_bytes / K,
                         "mean_bytes_per_active_problem_step": alg_bytes / max(active_steps, 1.0),
                         "traffic": traffic["dram_bytes_per_launch"] if traffic else None,
                         "traffic_unit": "bytes per launch (dram__bytes_read.sum + dram__bytes_write.sum, ncu --set full)",
                         "traffic_detail": traffic,
                         "peak_source": peak_src},
            "per_step_kinds": {"columns": list(KINDS[:4]) + ["idle"], "rows": per_step,
                               "note": f"batch 0: rows 0..{W - 1} are the warm-up steps, rows {W}..{W + min(K, STEPS_PER_BATCH) - 1} the timed ones"},
        }
        if traffic and per_step and traffic.get("timed_step_index") is not None:
            row = per_step[W + int(traffic["timed_step_index"])]
            alg = sum(table[k] * c for k, c in zip(list(KINDS[:4]), row[:4])) + row[4]
            line["roofline"]["traffic_over_algorithmic"] = traffic["dram_bytes_per_launch"] / alg
            line["roofline"]["algorithmic_bytes_of_the_captured_launch"] = alg
        if cpu:
            line["cpu_baseline"] = cpu
        if strong:
            line["batched_strong"] = strong
        elif not distributed:
            line["batched_strong"] = {"batch_total": BATCH, "n_gpus": 1, "note": "at N=1 this is `value`/`e2e` above"}
        if fused:
            line["fused_k_steps"] = fused
        if large:
            line["large_n"] = large
        if sharded:
            line["sharded_large_n"] = sharded
            line["sharded_check"] = sharded.get("bitwise_check")
        if riesz:
            line["riesz_gd"] = riesz
        if readme:
            line["readme_rosenbrock_n2"] = readme
        if pairwise:
            line["pairwise_radial"] = pairwise
        if lbfgs:
            line["live_lbfgs"] = lbfgs
        print(json.dumps(line))
    if distributed:
        dist.barrier()
        dist.destroy_process_group()


def bench_large(dz, orc, torch, stream, peak, device, cpu=True):
    import ctypes as C
    EF = dz.ExampleFunctions
    n = LARGE_N
    x0 = 4.0 * dz.pcg_fill(n, 1) - 2.0
    opt = dz.BFGSOptimizer(EF.rosenbrock_function, EF.rosenbrock_gradient_, x0, 1.0, device=device)
    opt.set_stream(stream.cuda_stream)
    opt.step(3)
    # 20 step! calls enqueued back to back (no host sync in between), an event after each; the device-side
    # step log says afterwards which calls were BFGS-type (GEMV + fused update) and which reset H
    nsteps = 60                       # the device-side step log keeps the last 64 kinds
    calls0, _ = opt.step_log()
    evs = [torch.cuda.Event(enable_timing=True) for _ in range(nsteps + 1)]
    evs[0].record(stream)
    for i in range(nsteps):
        opt.step_async(1)
        evs[i + 1].record(stream)
    torch.cuda.synchronize()
    times = [evs[i].elapsed_time(evs[i + 1]) for i in range(nsteps)]
    calls1, kinds = opt.step_log()
    types = [int(kinds[(calls0 + i) % 64]) for i in range(nsteps)]
    opt.close()
    bf = [t for t, ty in zip(times, types) if ty == dz.StepType.BFGSStep]
    gd = [t for t, ty in zip(times, types) if ty == dz.StepType.GradientDescentStep]
    out = {"n": n, "steps_timed": len(times), "bfgs_steps": len(bf), "gd_steps": len(gd),
           "timing": "back-to-back launches, CUDA event after every step!", "_launches": 4 * nsteps}
    if gd:
        out["ms_per_gd_step"] = float(np.mean(gd))
        out["gd_step_algorithmic_bytes"] = 8 * n * n      # identity_matrix! (:981): one write sweep
    if bf:
        ms = float(np.mean(bf))
        gbs = 24.0 * n * n / (ms * 1e-3) / 1e9
        out.update({"ms_per_bfgs_step": ms, "steps_per_s": 1e3 / ms, "achieved_gbs": gbs, "frac_of_peak": gbs / peak,
                    "algorithmic_bytes_per_step": 24 * n * n})
    if cpu:
        # the same step! on the host: oracle, TREE order, every host thread over rows (bit-identical to 1 thread)
        threads = os.cpu_count() or 1
        ref = orc.BFGS(orc.OBJ_ROSENBROCK, x0[None, :], 1.0, order=orc.TREE, nthreads=threads)
        ref.step(3)
        ts = []
        for _ in range(3):
            t0 = time.perf_counter(); ref.step(1); ts.append((time.perf_counter() - t0, int(ref.step_type[0])))
        bfc = [t for t, ty in ts if ty == 2]
        if bfc:
            out["cpu_baseline"] = {"ms_per_bfgs_step": 1e3 * float(np.mean(bfc)), "cores": threads, "kind": "port",
                                   "sample": f"{len(bfc)} BFGS-type step! calls of the same n=16384 problem, oracle with OpenMP over rows"}
    ms = C.c_float()
    for which, name, nbytes in ((1, "gemv_kernel", 8), (2, "update_gemv_kernel", 16), (3, "identity_kernel", 8)):
        rc = dz.lib().dzo_bench_kernel(which, n, 10, 0, C.byref(ms), device)
        if rc == 0:
            g = nbytes * n * n / (ms.value * 1e-3) / 1e9
            out[name] = {"ms": ms.value, "achieved_gbs": g, "frac_of_peak": g / peak}
    return out


def bench_sharded(dz, orc, torch, dist, stream, peak, rank, world, device):
    """BASELINE configs[3]: one extended-Rosenbrock problem of n = 65536 whose 32 GiB inverse Hessian is ROW-SHARDED over
    the `world` GPUs of this run (at N = 1 it fits one B200, so N = 1 -> 8 is a strong-scaling curve).  Every rank runs
    the O(n) stage redundantly; per BFGS-type step two n-vectors are gathered -- fused into the GEMV / update kernels
    over NVLink peer memory, or with ncclAllGather (both measured).  Times are CUDA events per step!, max over ranks,
    BFGS-type steps only (device-side step log).  The sharded result is checked in the run: at n = 8192 every rank
    compares its replicated vectors after every step! and its row slab of H at the end with the UNSHARDED CPU oracle,
    bit for bit (the oracle here is the checker, not the thing timed)."""
    import ctypes as C
    EF = dz.ExampleFunctions

    def make(n, x0):
        if world == 1:
            return dz.BFGSOptimizer(EF.rosenbrock_function, EF.rosenbrock_gradient_, x0, 1.0, device=device)
        idbuf = C.create_string_buffer(128)
        if rank == 0:
            assert dz.lib().dzo_nccl_get_unique_id(idbuf) == 0, dz.lib().dzo_last_error()
        box = [bytes(idbuf.raw)]
        dist.broadcast_object_list(box, src=0)
        return dz.BFGSOptimizer(EF.rosenbrock_function, EF.rosenbrock_gradient_, x0, 1.0, device=device,
                                shard=(rank, world, box[0]))

    def bits(a):
        return np.ascontiguousarray(a, dtype=np.float64).view(np.uint64)

    def check(mode_name):
        n, steps = SHARDED_CHECK_N, 6
        x0 = 4.0 * dz.pcg_fill(n, 2) - 2.0
        have = torch.tensor([1.0 if orc is not None else 0.0], device="cuda")
        if dist is not None:
            dist.broadcast(have, src=0)
        if have.item() == 0.0:
            return "skipped (--skip-cpu: no checker loaded)"
        trace = torch.empty((steps, 3 * n + 2), dtype=torch.float64, device="cuda")
        Href = torch.empty((n, n), dtype=torch.float64, device="cuda")
        if rank == 0:
            ref = orc.BFGS(orc.OBJ_ROSENBROCK, x0[None, :], 1.0, order=orc.TREE, nthreads=os.cpu_count() or 1)
            rows = []
            for _ in range(steps):
                ref.step(1)
                rows.append(np.concatenate([ref.point[0], ref.gradient[0], ref.direction[0], ref.objective, ref.step_length]))
            trace.copy_(torch.from_numpy(np.stack(rows)))
            Href.copy_(torch.from_numpy(np.ascontiguousarray(ref.inverse_hessian(0))))
            ref.close()
        if dist is not None:
            dist.broadcast(trace, src=0)
            dist.broadcast(Href, src=0)
        tr = trace.cpu().numpy()
        opt = make(n, x0)
        ok = True
        for it in range(steps):
            opt.step(1)
            d_now = opt.next_step_direction                        # read right behind step!: must already be complete
            got = np.concatenate([opt.current_point, opt.current_gradient, d_now,
                                  [float(opt.current_objective_value[()])], [float(opt.last_step_length[()])]])
            ok = ok and bool(np.array_equal(bits(got), bits(tr[it])))
        r0, r1 = opt.row_range
        ok = ok and bool(np.array_equal(bits(opt.inverse_hessian()), bits(Href[r0:r1].cpu().numpy())))
        opt.close()
        flag = torch.tensor([1.0 if ok else 0.0], device="cuda")
        if dist is not None:
            dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        return "ok" if flag.item() == 1.0 else "FAILED"

    n = SHARDED_N
    x0 = 4.0 * dz.pcg_fill(n, 2) - 2.0
    out = {"n": n, "n_gpus": world, "rows_per_gpu": n // world, "algorithmic_bytes_per_bfgs_step_per_gpu": 24 * n * n // world,
           "check_n": SHARDED_CHECK_N, "_launches": 0}
    modes = [("fused-peer-memory", 0), ("nccl-allgather", 1)] if world > 1 else [("single-gpu", 0)]
    nsteps = 24
    for name, variant in modes:
        dz.set_tuning("sharded_variant", variant)
        res = {"bitwise_check": check(name)}
        opt = make(n, x0)
        actual = {0: "single-gpu", 1: "fused-peer-memory", 2: "nccl-allgather"}[opt.gather_mode]
        opt.set_stream(stream.cuda_stream)
        opt.step(3)
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()
        calls0, _ = opt.step_log()
        evs = [torch.cuda.Event(enable_timing=True) for _ in range(nsteps + 1)]
        evs[0].record(stream)
        for i in range(nsteps):              # back to back: no host sync between step! calls
            opt.step_async(1)
            evs[i + 1].record(stream)
        torch.cuda.synchronize()
        tt = torch.tensor([evs[i].elapsed_time(evs[i + 1]) for i in range(nsteps)], device="cuda", dtype=torch.float64)
        if dist is not None:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        times = tt.tolist()
        _, kinds = opt.step_log()
        types = [int(kinds[(calls0 + i) % 64]) for i in range(nsteps)]
        opt.close()
        out["_launches"] += (4 + (1 if world > 1 else 0)) * nsteps
        bf = [t for t, ty in zip(times, types) if ty == dz.StepType.BFGSStep]
        res.update({"gather_mode": actual, "bfgs_steps": len(bf), "steps_timed": nsteps})
        if bf:
            ms = float(np.mean(bf))
            gbs = 24.0 * n * n / world / (ms * 1e-3) / 1e9
            res.update({"ms_per_bfgs_step": ms, "steps_per_s": 1e3 / ms, "per_gpu_gbs": gbs, "frac_of_peak": gbs / peak})
        out[name] = res
    dz.set_tuning("sharded_variant", 0)
    first = out[modes[0][0]]
    for k in ("ms_per_bfgs_step", "per_gpu_gbs", "frac_of_peak", "gather_mode", "bitwise_check"):
        if k in first:
            out[k] = first[k]
    if world > 1 and any(out[m[0]].get("bitwise_check") == "FAILED" for m in modes):
        out["bitwise_check"] = "FAILED"
    return out


def bench_riesz(dz, orc, torch, stream, device, cpu=True):
    """BASELINE configs[4]: GradientDescentOptimizer on Riesz-energy points on the sphere, N=4096 (n=12288).
    FP64-pipe bound (one sqrt + one or two divisions per pair), not an HBM roofline: reported as GD steps/s
    and pair terms/s.  Inputs per SURVEY 8d: PCG seed 3 uniform in [-1,1)^3, normalised; initial step 1e-3."""
    EF = dz.ExampleFunctions
    N = 4096
    p = 2.0 * dz.pcg_fill(3 * N, 3).reshape(N, 3) - 1.0
    p = p / np.sqrt((p * p).sum(axis=1, keepdims=True))
    opt = dz.GradientDescentOptimizer(dz.SPHERE_CONSTRAINT, EF.riesz_energy, EF.riesz_gradient_,
                                      dz.QuadraticLineSearch(0), p, 1e-3, device=device)
    opt.set_stream(stream.cuda_stream)
    opt.step(3)
    k = 20
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    it0 = int(opt.iteration_count[()])
    ev0 = opt.evaluation_count()
    e0.record(stream)
    opt.step_async(k)            # k step! calls inside ONE cooperative launch
    e1.record(stream)
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    done = int(opt.iteration_count[()]) - it0
    f = float(opt.current_objective_value[()])
    evals = opt.evaluation_count() - ev0
    opt.close()
    # FP64-pipe roofline (SURVEY 8d): one energy evaluation = N(N-1)/2 pair terms x 22 FP64 instructions (3 sub, 3 mul, 2 add,
    # the IEEE sqrt and reciprocal sequences, accumulate), one gradient = N(N-1) ordered pair terms x 38 (DESIGN.md section 3;
    # counted in the SASS of the pair loops).  Peak: 148 SMs x 64 FP64 lanes per clock (B200: 40 TFLOP/s FP64 FMA) at the
    # maximum SM clock.
    pair_e, pair_g = N * (N - 1) // 2, N * (N - 1)
    fp64_instr = evals * pair_e * 22 + done * pair_g * 38
    fp64_peak = 148 * 64 * 1.965e9
    out = {"N": N, "n": 3 * N, "gd_steps": done, "ms_per_gd_step": ms / max(done, 1), "gd_steps_per_s": 1e3 * done / ms,
           "objective": f, "energy_evaluations": evals, "energy_evaluations_per_step": evals / max(done, 1),
           "pair_terms_per_s": (evals * pair_e + done * pair_g) / (ms * 1e-3),
           "roofline": {"bound": "fp64", "achieved": fp64_instr / (ms * 1e-3), "peak": fp64_peak,
                        "unit": "FP64 thread-instructions/s", "frac": fp64_instr / (ms * 1e-3) / fp64_peak,
                        "how": "(evaluations x N(N-1)/2 x 22 + gradients x N(N-1) x 38) / time; peak = 148 SMs x 64 lanes x 1.965 GHz",
                        "ncu": "profiles/: sm__pipe_fp64_cycles_active of the same kernel"}}
    if cpu:
        ref = orc.GD(orc.OBJ_RIESZ, p.reshape(1, -1), 1e-3, order=orc.TREE, constraint=orc.CONSTRAINT_SPHERE, dim=3)
        ref.step(3)
        t0 = time.perf_counter(); ref.step(3); dt = time.perf_counter() - t0
        out["cpu_baseline"] = {"ms_per_gd_step": 1e3 * dt / 3, "cores": 1, "kind": "port",
                               "sample": "3 GD step! calls of the same N=4096 problem, oracle single thread (the reference is single-threaded)"}
    return out


def bench_pairwise(dz, orc, torch, cpu=True):
    """SURVEY 8f rank 1: the live package's accelerated pairwise radial kernels (Lennard-Jones), device arrays
    in / out as in the reference API.  FP64-pipe bound; reported as pair terms/s (n^2 per launch)."""
    EF = dz.ExampleFunctions
    n = 16384
    L = 1.2 * n ** (1.0 / 3.0)
    p = dz.pcg_fill(3 * n, 21).reshape(3, n) * L
    t = [torch.from_numpy(a.copy()).cuda() for a in p]
    g = [torch.empty(n, dtype=torch.float64, device="cuda") for _ in range(3)]
    out = {"n": n, "potential": "lennard_jones"}
    for name, order in (("sequential", 0), ("tree", 1)):
        for _ in range(3):
            dz.accelerated_pairwise_radial_gradient_(*g, EF.lj_first_derivative, *t, order=order)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        reps = 10
        e0.record()
        for _ in range(reps):
            dz.accelerated_pairwise_radial_gradient_(*g, EF.lj_first_derivative, *t, order=order)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / reps
        out["gradient_" + name] = {"ms": ms, "pair_terms_per_s": n * n / (ms * 1e-3)}
    if cpu:
        t0 = time.perf_counter()
        orc.pairwise_gradient(p[0], p[1], p[2], orc.SEQ)
        dt = time.perf_counter() - t0
        out["cpu_baseline"] = {"ms": 1e3 * dt, "pair_terms_per_s": n * n / dt, "cores": os.cpu_count(), "kind": "port",
                               "sample": "one gradient of the same n=16384 cloud, oracle with OpenMP over particles"}
    return out


def bench_lbfgs(dz, orc, torch, stream, cpu=True):
    """SURVEY 8f rank 2: the live package's LBFGSOptimizer (the package's own answer for large n) on
    extended Rosenbrock n = 2^20, history 10: k step! calls in ONE cooperative launch (eight 512-thread CTAs per block
    of 65536 elements, DZO_ORDER_TREE_BLOCKED, the direction vector in registers).  Algorithmic traffic per step! with
    a full history and one line-search trial: (4m + 12) n-vectors = every s_i and y_i twice (4m), g and x once, the
    direction stored once, accept pass (3 reads, 6 writes).  The step is barrier-bound (2m + 2 grid barriers), so the
    HBM fraction is reported for orientation, not as the bound."""
    EF = dz.ExampleFunctions
    n, m, k = 1 << 20, 10, 50
    x0 = 4.0 * dz.pcg_fill(n, 9) - 2.0
    opt = dz.LBFGSOptimizer(None, EF.rosenbrock_function, EF.rosenbrock_gradient_, x0, 1.0, m)
    opt.set_stream(stream.cuda_stream)
    opt.step(12)
    it0 = int(opt.iteration_count[()])
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream); opt.step_async(k); e1.record(stream)
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    done = int(opt.iteration_count[()]) - it0
    bytes_per_step = 8 * n * (4 * m + 12)
    clusters = C.c_int()
    dz.lib().dzo_lbfgs_info(opt._h, None, None, C.byref(clusters))
    out = {"n": n, "history_length": m, "steps": done, "ms_per_step": ms / max(done, 1), "steps_per_s": 1e3 * done / ms,
           "objective": float(opt.current_objective_value[()]), "ctas": clusters.value,
           "algorithmic_bytes_per_step": bytes_per_step,
           "achieved_gbs": bytes_per_step * done / (ms * 1e-3) / 1e9, "order": "DZO_ORDER_TREE_BLOCKED"}
    opt.close()
    if cpu:
        ref = orc.LBFGS(orc.OBJ_ROSENBROCK, x0, 1.0, m, orc.TREE_BLOCKED)
        ref.step(5)
        t0 = time.perf_counter(); ref.step(5); dt = time.perf_counter() - t0
        out["cpu_baseline"] = {"ms_per_step": 1e3 * dt / 5, "cores": 1, "kind": "port",
                               "sample": "5 step! calls of the same problem, oracle single thread"}
    # SURVEY 8f rank 3: the legacy LBFGSOptimizer (quadratic line search, cyclic history), same grid-wide machinery
    n2 = 1 << 20
    x1 = 4.0 * dz.pcg_fill(n2, 9) - 2.0
    leg = dz.LegacyLBFGSOptimizer(EF.rosenbrock_function, EF.rosenbrock_gradient_, dz.QuadraticLineSearch(0), x1, 1.0, m)
    leg.set_stream(stream.cuda_stream)
    leg.step(12)
    it0 = int(leg.iteration_count[()])
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream); leg.step_async(k); e1.record(stream)
    torch.cuda.synchronize()
    done2 = int(leg.iteration_count[()]) - it0
    out["legacy_lbfgs"] = {"n": n2, "history_length": m, "steps": done2, "ms_per_step": e0.elapsed_time(e1) / max(done2, 1),
                           "objective": float(leg.current_objective_value[()])}
    leg.close()
    return out


def bench_readme(dz, orc):
    """BASELINE configs[0]: README Rosenbrock n=2 from rand(2), step 1.0, run to has_converged -- the
    reference's own CPU-runnable case (README.md:49-66 reports 2.8 us min / 5.6 us median per optimisation
    on an unspecified CPU).  Oracle: 1000 PCG seeds, one thread; GPU: the same 1000 problems as one batch."""
    x0 = np.stack([dz.pcg_fill(2, s) for s in range(1000)])
    t0 = time.perf_counter()
    ref = orc.BFGS(orc.OBJ_ROSENBROCK, x0, 1.0, order=orc.SEQ, nthreads=1)
    while ref.count_active():
        ref.step(16)
    cpu_us = 1e6 * (time.perf_counter() - t0) / 1000
    EF = dz.ExampleFunctions
    t0 = time.perf_counter()
    opt = dz.BFGSOptimizer(EF.rosenbrock_function, EF.rosenbrock_gradient_, x0, 1.0, batched=True)
    while opt.count_active():
        opt.step(16)
    gpu_us = 1e6 * (time.perf_counter() - t0) / 1000
    same = bool(np.array_equal(opt.current_point, ref.point))
    opt.close()
    return {"problems": 1000, "cpu_us_per_optimisation": cpu_us, "cpu_cores": 1, "cpu_kind": "port",
            "gpu_us_per_optimisation_batched": gpu_us, "bitwise_equal_to_oracle": same,
            "reference_published_us": {"min": 2.8, "median": 5.563, "hardware": "unspecified (README.md:62-63)"},
            "port_over_published_median": cpu_us / 5.563,
            "note": "the C port is slower than the published Julia figure by this factor on config 1: read every "
                    "GPU/CPU-port ratio of this line as an upper bound of the ratio against tuned Julia"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=150,
                    help="default: the timed region of the headline is >= 100 ms (about 0.7 ms per step!), six batches")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--skip-large", action="store_true")
    ap.add_argument("--skip-cpu", action="store_true")
    ap.add_argument("--no-numa-bind", action="store_true", help="multi-rank runs: leave the ranks' CPU affinity alone (A/B)")
    ap.add_argument("--cpu-sample", type=int, default=50_000)
    ap.add_argument("--tune", action="append", default=[], help="key=value passed to dzo_set_tuning (A/B runs)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed as DIR/<field>.npy (GPU arm)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs is not None and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the GPU arm (--impl b200)")
    if args.warmup < 3:
        args.warmup = 3
    if args.impl == "reference":
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
