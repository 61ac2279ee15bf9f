"""The two bottom solvers side by side on one GPU, in one process: BiCGStab and CG on `hpgmg-fv 7 8` (a 2^3 bottom) and
`hpgmg-fv 4 27` (a 3^3 bottom).  For each: ms per FMG solve and DOF/s (the library's device timer, as bench.py), bottom-solver
iterations per FMG solve, the stand-alone single-block bottom kernel (CUDA events around --reps calls of zero_vector(E) +
IterativeSolver(E <- R) on the bottom level, R as the last solve left it), and the driver's Richardson pass (F-cycle norms,
error, order).  Prints a table and writes JSON (--out).

  python tools/bench_bottom.py [--steps 20] [--warmup 3] [--reps 100] [--out profiles/bottom_solvers.json]
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tools")):
    if p not in sys.path:
        sys.path.insert(0, p)
import hpgmg_b200.api as api  # noqa: E402
from bench_smoothers import gpu_info  # noqa: E402

SOLVERS = [("bicgstab", api.BOTTOM_BICGSTAB), ("cg", api.BOTTOM_CG)]
CONFIGS = [(7, 8), (4, 27)]


def measure(name, solver, log2, boxes, steps, warmup, reps):
    L = api.lib()
    with api.Hierarchy(log2, boxes, bottom_solver=solver) as H:
        dof = float(H.dof(0))
        bottom = H.level(H.num_levels - 1)
        for _ in range(warmup):
            H.fmg_solve(0)
        L.hpgmg_b200_sync()
        L.hpgmg_b200_bench_mark(0)
        for _ in range(steps):
            norm, _ = H.fmg_solve(0)
        L.hpgmg_b200_bench_mark(1)
        L.hpgmg_b200_sync()
        ms = L.hpgmg_b200_bench_elapsed_ms(0, 1) / steps
        iters_per_solve = bottom.contents.Krylov_iterations / float(warmup + steps)

        def bottom_solve():
            L.zero_vector(bottom, api.VECTOR_E)
            L.IterativeSolver(bottom, api.VECTOR_E, api.VECTOR_R, H.a, H.b, 1e-3)
        for _ in range(4):
            bottom_solve()
        L.hpgmg_b200_bench_mark(2)
        for _ in range(reps):
            bottom_solve()
        L.hpgmg_b200_bench_mark(3)
        L.hpgmg_b200_sync()
        bottom_us = 1e3 * L.hpgmg_b200_bench_elapsed_ms(2, 3) / reps
        bottom_dim = bottom.contents.box_dim
        err, order, norms = H.richardson()
    return {"solver": name, "workload": f"hpgmg-fv {log2} {boxes}", "bottom_cells": f"{bottom_dim}^3", "ms_per_solve": ms,
            "dof_per_s": dof / (1e-3 * ms), "f_cycle_norm": norm, "bottom_iterations_per_fmg_solve": iters_per_solve,
            "bottom_kernel_us": bottom_us, "richardson_norms": [n[0] for n in norms], "error": err, "order": order}


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--reps", type=int, default=100, help="bottom solves timed (at least 50)")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "bottom_solvers.json"))
    args = ap.parse_args()
    if args.reps < 50:
        raise SystemExit("--reps: at least 50 bottom solves")
    api.init(0)
    api.lib().hpgmg_b200_set_verbose(0)
    card = gpu_info()
    rows = [measure(name, sv, log2, boxes, args.steps, args.warmup, args.reps) for log2, boxes in CONFIGS for name, sv in SOLVERS]
    api.lib().hpgmg_b200_set_bottom_solver(api.BOTTOM_BICGSTAB)
    print(f"one GPU: {card}")
    print(f"{'workload':>14} {'bottom':>6} {'solver':>8} {'ms/solve':>9} {'DOF/s':>10} {'its/solve':>9} {'bottom us':>9} {'F-cycle norm':>23} {'error':>22} {'order':>6}")
    for r in rows:
        print(f"{r['workload']:>14} {r['bottom_cells']:>6} {r['solver']:>8} {r['ms_per_solve']:9.3f} {r['dof_per_s']:10.3e} {r['bottom_iterations_per_fmg_solve']:9.1f} "
              f"{r['bottom_kernel_us']:9.1f} {r['f_cycle_norm']!r:>23} {r['error']!r:>22} {r['order']:6.3f}")
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump({"gpu": card, "steps": args.steps, "warmup": args.warmup, "bottom_reps": args.reps,
                   "bottom_kernel_timing": "zero_vector(E) + IterativeSolver(E <- R) on the bottom level, CUDA events around the calls",
                   "rows": rows}, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
