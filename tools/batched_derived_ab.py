"""A/B of the batched BFGS layouts (Tuning::batched_derived 0 = every field stored, 1 = derived) in ONE process.

    python tools/batched_derived_ab.py [--reps 3] [--steps 25] [--warmup 5] [--ns 2,4,8,12,16,24,32] [--out FILE]

bench.py's workload: 1 M problems of n = 16 from PCG seed 2024, W warm-up steps, then K single-step launches timed with
CUDA events on a side stream.  The layouts alternate `reps` times each, in the order 0, 1 on even repetitions and 1, 0
on odd ones, so that a drift of clocks or temperature within the call favours neither.  Every run prints one JSON line:
ms per launch, problem-steps/s, the device's step-kind counters and the algorithmic bytes of that mix in the layout it
ran (bytes_by_kind below), and the layout the handle reports (dzo_bfgs_batched_layout).  Then the same for the other n,
one batch of 1 M problems each (as profiles/r02_batched_per_n.jsonl), and for n = 16 at a batch the automatic policy
runs with 27 problems per warp (the run-time-tile instantiations of the kernel).
The card name and power limit are read in the same call.  Nothing is compiled at run time."""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True


def bytes_by_kind(n, derived):
    """ALGORITHMIC bytes of one problem-step by kind (DESIGN.md section 3), lazy identities.  The stored layout reads x, g,
    d and writes x, g, d, dx, dg; the derived layout reads x, d and writes x, d, plus the flags byte on every move."""
    vec, H = 8 * n, 8 * n * n
    rd = (2 if derived else 3) * vec + 26
    wr = (2 if derived else 5) * vec + 28 + (1 if derived else 0)
    return {"bfgs_read_h": rd + H + wr + H,
            "bfgs_identity_h": rd + wr + H + (0 if derived else 1),
            "gradient_descent": rd + wr + (0 if derived else 1),
            "terminate": rd + 1,
            "idle": 1, "idle_warp": 1}


def card():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        return r.stdout.strip().splitlines()[0]
    except Exception as e:   # the timing itself does not depend on it
        return f"unavailable ({e})"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=1_000_000)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--steps", type=int, default=25)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--ns", default="2,4,8,12,16,24,32")
    ap.add_argument("--out", default=None, help="also append the JSON lines to this file")
    args = ap.parse_args()
    import torch
    import dzopt_b200 as dz
    EF = dz.ExampleFunctions
    out = open(args.out, "a") if args.out else None

    def emit(rec):
        line = json.dumps(rec)
        print(line, flush=True)
        if out:
            out.write(line + "\n")

    emit({"card": card(), "torch_device": torch.cuda.get_device_name(0)})
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    import ctypes as C
    slots = torch.cuda.get_device_properties(0).multi_processor_count * 16     # resident warps at n <= 16
    cases = [(16, args.batch)] + [(n, args.batch) for n in (int(v) for v in args.ns.split(",")) if n != 16]
    cases.append((16, 26 * slots + slots // 2))                                   # 27 problems per warp
    for n, batch in cases:
        x0 = (4.0 * dz.pcg_fill(batch * n, 2024) - 2.0).reshape(batch, n)
        for rep in range(args.reps):
            for derived in ((0, 1) if rep % 2 == 0 else (1, 0)):
                dz.set_tuning("batched_derived", derived)
                opt = dz.BFGSOptimizer(EF.rosenbrock_function, EF.rosenbrock_gradient_, x0, 1.0, batched=True)
                opt.set_stream(stream.cuda_stream)
                got = C.c_int(-1)
                assert dz.lib().dzo_bfgs_batched_layout(opt._h, None, C.byref(got)) == 0 and got.value == derived
                opt.step(args.warmup)
                opt.step_kind_counts(reset=True)
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                torch.cuda.synchronize()
                e0.record(stream)
                for _ in range(args.steps):
                    opt.step_async(1)
                e1.record(stream)
                torch.cuda.synchronize()
                ms = e0.elapsed_time(e1) / args.steps
                kinds = opt.step_kind_counts()
                active = sum(kinds[k] for k in ("bfgs_read_h", "bfgs_identity_h", "gradient_descent", "terminate"))
                table = bytes_by_kind(n, derived)
                b = sum(table[k] * kinds.get(k, 0) for k in table) / args.steps
                emit({"n": n, "batch": batch, "batched_derived": derived, "rep": rep, "ms_per_launch": ms,
                      "problem_steps_per_s": active / args.steps / (ms * 1e-3), "kinds": kinds,
                      "algorithmic_bytes_per_launch": b, "achieved_gbs": b / (ms * 1e-3) / 1e9})
                opt.close()
    dz.set_tuning("batched_derived", -1)


if __name__ == "__main__":
    main()
