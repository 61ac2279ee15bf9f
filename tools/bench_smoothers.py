"""The four smoothers side by side on one GPU, in one process: `hpgmg-fv 7 8` (with --big: `8 8`) solved with GSRB, Chebyshev,
weighted Jacobi and L1-Jacobi.  For each: ms per FMG solve and DOF/s (the library's device timer, as bench.py), the level-0
sweep kernel alone (hpgmg_b200_smoother_sweep, CUDA events around --reps launches) with its algorithmic GB/s, and the driver's
Richardson pass (F-cycle norm, error, order).  Prints a table and writes JSON (--out).

  python tools/bench_smoothers.py [--big] [--steps 20] [--warmup 3] [--reps 100] [--out profiles/smoothers_7_8.json]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
import hpgmg_b200.api as api  # noqa: E402

SMOOTHERS = [("gsrb", api.SMOOTHER_GSRB), ("cheby", api.SMOOTHER_CHEBY), ("jacobi", api.SMOOTHER_JACOBI), ("l1jacobi", api.SMOOTHER_L1JACOBI)]
# algorithmic HBM bytes per cell of one sweep: x, rhs, the point-wise inverse (Dinv or lambda) and 3 betas read, x written;
# Chebyshev also reads x_{n-1}
SWEEP_BYTES_PER_CELL = {"gsrb": 56.0, "cheby": 64.0, "jacobi": 56.0, "l1jacobi": 56.0}
COPY_PEAK_GBS = 6456.0                   # measured copy peak of a B200 (DESIGN.md section 3)


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"], capture_output=True, text=True, timeout=60).stdout
        return out.strip().splitlines()[1] if len(out.strip().splitlines()) > 1 else out.strip()
    except Exception as e:                # the numbers then stand without the card: say so
        return f"nvidia-smi unavailable ({e})"


def measure(name, smoother, log2, boxes, steps, warmup, reps):
    L = api.lib()
    with api.Hierarchy(log2, boxes, smoother=smoother) as H:
        lvl = H.level(0)
        dof = float(H.dof(0))
        for _ in range(warmup):
            H.fmg_solve(0)
        L.hpgmg_b200_sync()
        L.hpgmg_b200_bench_mark(0)
        for _ in range(steps):
            norm, _ = H.fmg_solve(0)
        L.hpgmg_b200_bench_mark(1)
        L.hpgmg_b200_sync()
        ms = L.hpgmg_b200_bench_elapsed_ms(0, 1) / steps

        def sweep(s):                 # level 0, U <-> TEMP as smooth() does, no ghost fill
            src, dst = (api.VECTOR_U, api.VECTOR_TEMP) if s % 2 == 0 else (api.VECTOR_TEMP, api.VECTOR_U)
            L.hpgmg_b200_smoother_sweep(lvl, src, dst, api.VECTOR_F, H.a, H.b, s % 6)
        for s in range(4):
            sweep(s)
        L.hpgmg_b200_bench_mark(2)
        for s in range(reps):
            sweep(s)
        L.hpgmg_b200_bench_mark(3)
        L.hpgmg_b200_sync()
        sweep_us = 1e3 * L.hpgmg_b200_bench_elapsed_ms(2, 3) / reps
        Lc = lvl.contents
        cells = Lc.num_my_boxes * Lc.box_dim ** 3
        gbs = SWEEP_BYTES_PER_CELL[name] * cells / (1e-6 * sweep_us) / 1e9
        err, order, norms = H.richardson()
    return {"smoother": name, "ms_per_solve": ms, "dof_per_s": dof / (1e-3 * ms), "f_cycle_norm": norm,
            "sweep_us": sweep_us, "sweep_bytes_per_cell": SWEEP_BYTES_PER_CELL[name], "sweep_gbs": gbs, "sweep_frac_of_copy_peak": gbs / COPY_PEAK_GBS,
            "richardson_norms": [n[0] for n in norms], "error": err, "order": order}


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--big", action="store_true", help="hpgmg-fv 8 8 (512^3) instead of 7 8 (256^3)")
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--reps", type=int, default=100, help="sweep launches timed (at least 50)")
    ap.add_argument("--out", default=None, help="JSON file (default profiles/smoothers_<log2>_8.json)")
    args = ap.parse_args()
    if args.reps < 50:
        raise SystemExit("--reps: at least 50 launches")
    log2 = 8 if args.big else 7
    out = args.out or os.path.join(ROOT, "profiles", f"smoothers_{log2}_8.json")
    api.init(0)
    api.lib().hpgmg_b200_set_verbose(0)
    card = gpu_info()
    rows = [measure(name, sm, log2, 8, args.steps, args.warmup, args.reps) for name, sm in SMOOTHERS]
    api.lib().hpgmg_b200_set_smoother(api.SMOOTHER_GSRB)
    print(f"hpgmg-fv {log2} 8 on one GPU: {card}")
    print(f"{'smoother':>9} {'ms/solve':>9} {'DOF/s':>10} {'sweep us':>9} {'GB/s':>7} {'of peak':>7} {'F-cycle norm':>23} {'error':>22} {'order':>6}")
    for r in rows:
        print(f"{r['smoother']:>9} {r['ms_per_solve']:9.3f} {r['dof_per_s']:10.3e} {r['sweep_us']:9.1f} {r['sweep_gbs']:7.0f} {r['sweep_frac_of_copy_peak']:7.3f} "
              f"{r['f_cycle_norm']!r:>23} {r['error']!r:>22} {r['order']:6.3f}")
    os.makedirs(os.path.dirname(os.path.abspath(out)), exist_ok=True)
    with open(out, "w") as f:
        json.dump({"workload": f"hpgmg-fv {log2} 8, one GPU", "gpu": card, "steps": args.steps, "warmup": args.warmup, "sweep_reps": args.reps,
                   "copy_peak_gbs": COPY_PEAK_GBS, "rows": rows}, f, indent=1)
    print("wrote", out)


if __name__ == "__main__":
    main()
