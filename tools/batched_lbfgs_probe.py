"""Time the batched live L-BFGS kernel (dzo_lbfgs_create_batched) on 1 M extended-Rosenbrock problems.

For every n in --n and history length m in --m (and CTA size in --threads): x0 = 4u - 2 from the product's pcg_fill,
W warm-up step! calls, then K timed launches of step(1), each between two CUDA events on the handle's stream.  Before
and after the timed launches a fixed seeded sample of problems is compared bit for bit with one oracle
DZO_ORDER_SEQUENTIAL handle per problem; any difference aborts the run, so the configuration that is timed is the one
that was verified.

Algorithmic bytes of a launch come from the live-problem count and the history counts read back BETWEEN launches
(outside the timed window): a live problem-step with c history entries reads x, g (2n doubles), the two history
vectors of each of its c slots twice (4cn) and their rho (2c), plus 33 bytes of scalars, and writes x, dx, g, dg, d,
one S and one Y slot (7n doubles), one rho and 32 bytes of scalars; a stuck problem reads its flag (1 byte).
There is no CPU fallback: without a GPU the script fails.

    python tools/batched_lbfgs_probe.py [--n 2,8,16,32] [--m 5,10] [--threads 128] [--out DIR]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))
PEAK_GBS = 6456.8           # measured HBM peak the project quotes (DESIGN.md section 3)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def counts(dz, opt):
    cnt = np.zeros(opt._batch, dtype=np.int64)
    rho = np.zeros((opt._batch, 64))
    assert dz.lib().dzo_lbfgs_get_rho_history(opt._h, cnt.ctypes.data_as(dz._capi.c_i64_p),
                                              rho.ctypes.data_as(dz._capi.c_double_p)) == 0
    return cnt, opt.is_stuck


def launch_bytes(n, cnt, stuck):
    c = cnt[~stuck]
    live = 8 * (2 * n + 4 * c * n + 2 * c + 7 * n + 1) + 33 + 32
    return int(live.sum()) + int(stuck.sum())


def follow(opt, refs, idx, active, k):
    """Step the oracle handles of the still active sample problems k times.  A problem the device left stuck with a
    direction on which the reference's backtracking never ends (not finite, or +0.0 at a -0.0 coordinate; the device
    caps that search) is retired first: the oracle, like the reference, would loop forever on it."""
    x, d, stuck = opt.current_point[idx], opt.step_direction[idx], opt.is_stuck[idx]
    endless = ~np.isfinite(d).all(axis=1) | (np.signbit(x) & (x == 0) & ~np.signbit(d) & (d == 0)).any(axis=1)
    active = active & ~(stuck & endless)
    for j in np.flatnonzero(active):
        refs[j].step(k)
    return active


def verify(orc, opt, refs, idx, what):
    fields = (("current_point", "point"), ("delta_point", "delta_point"), ("current_gradient", "gradient"),
              ("delta_gradient", "delta_gradient"), ("step_direction", "direction"))
    for a, k in fields:
        dev = getattr(opt, a)[idx]
        ref = np.array([getattr(r, k) for r in refs])
        if not np.array_equal(dev.view(np.uint64), ref.view(np.uint64)):
            raise SystemExit(f"{what}: {a} differs from the oracle")
    for a, k in (("current_objective_value", "objective"), ("delta_objective_value", "delta_objective")):
        if not np.array_equal(getattr(opt, a)[idx].view(np.uint64), np.array([getattr(r, k) for r in refs]).view(np.uint64)):
            raise SystemExit(f"{what}: {a} differs from the oracle")
    if not (np.array_equal(opt.iteration_count[idx], [r.iteration_count for r in refs]) and
            np.array_equal(opt.is_stuck[idx], [r.stuck for r in refs])):
        raise SystemExit(f"{what}: iteration_count / is_stuck differ from the oracle")
    hist = opt.rho_history
    for j, p in enumerate(idx):
        if not np.array_equal(hist[p].view(np.uint64), refs[j].rho_history.view(np.uint64)):
            raise SystemExit(f"{what}: rho_history of problem {p} differs from the oracle")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", default="2,8,16,32")
    ap.add_argument("--m", default="5,10")
    ap.add_argument("--threads", default="128")
    ap.add_argument("--batch", type=int, default=1_000_000)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--sample", type=int, default=4096)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    import dzopt_b200 as dz
    import oracle as orc
    orc.build()
    if not torch.cuda.is_available():
        raise SystemExit("no CUDA device: the probe measures the GPU and has no fallback")
    EF = dz.ExampleFunctions
    name = card()
    stream = torch.cuda.Stream()
    lines = []
    for threads in [int(t) for t in args.threads.split(",")]:
        dz.set_tuning("lbfgs_batched_threads", threads)
        for n in [int(v) for v in args.n.split(",")]:
            for m in [int(v) for v in args.m.split(",")]:
                x0 = (4.0 * dz.pcg_fill(args.batch * n, 2024) - 2.0).reshape(args.batch, n)
                idx = np.sort(np.random.default_rng(7).choice(args.batch, args.sample, replace=False))
                opt = dz.LBFGSOptimizer(None, EF.rosenbrock_function, EF.rosenbrock_gradient_, x0, 1.0, m, batched=True)
                opt.set_stream(stream.cuda_stream)
                refs = [orc.LBFGS(orc.OBJ_ROSENBROCK, x0[p], 1.0, m, order=orc.SEQ) for p in idx]
                opt.step(args.warmup)
                active = follow(opt, refs, idx, np.ones(idx.size, dtype=bool), args.warmup)
                verify(orc, opt, [refs[j] for j in np.flatnonzero(active)], idx[active], f"n={n} m={m} after the warm-up")
                ms, nbytes, live_steps = [], 0, 0
                for _ in range(args.steps):
                    cnt, stuck = counts(dz, opt)
                    nbytes += launch_bytes(n, cnt, stuck)
                    live_steps += int((~stuck).sum())
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record(stream)
                    opt.step_async(1)
                    e1.record(stream)
                    e1.synchronize()
                    ms.append(e0.elapsed_time(e1))
                active = follow(opt, refs, idx, active, args.steps)
                verify(orc, opt, [refs[j] for j in np.flatnonzero(active)], idx[active], f"n={n} m={m} after the timed steps")
                total_s = sum(ms) / 1e3
                gbs = nbytes / total_s / 1e9
                line = {"n": n, "m": m, "batch": args.batch, "threads": threads, "warmup": args.warmup,
                        "steps": args.steps, "ms_per_step_median": float(np.median(ms)),
                        "ms_per_step_mean": float(np.mean(ms)), "active_problem_steps_per_s": live_steps / total_s,
                        "live_fraction": live_steps / (args.steps * args.batch),
                        "algorithmic_bytes_per_step": nbytes / args.steps, "GB_per_s": gbs,
                        "share_of_measured_peak": gbs / PEAK_GBS, "verified_sample": int(active.sum()), "card": name}
                print(json.dumps(line), flush=True)
                lines.append(line)
                opt.close()
                del refs
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "batched_lbfgs_probe.jsonl"), "w") as f:
            for line in lines:
                f.write(json.dumps(line) + "\n")


if __name__ == "__main__":
    main()
