"""Library flavours against each other on one GPU, in one process: `hpgmg-fv 7 8` (256^3) with GSRB, solved alternately by
each flavour of --flavours (default fv2,fv4: the fv2 flavour libhpgmg_b200_fv2.so and the default fv4 library; fv2_helmholtz is
libhpgmg_b200_fv2_helmholtz.so, solving a = b = 1), --rounds times each.  For each run: ms per FMG solve (the library's device
timer, as bench.py), the level-0 sweep kernel alone (hpgmg_b200_smoother_sweep, CUDA events around --reps launches) with its
GB/s against the flavour's algorithmic byte model and that rate's fraction of the measured copy bandwidth, the F-cycle norm,
and the card's name and power limit.  Prints a table and writes JSON (--out, default profiles/fv2.json).

  python tools/bench_fv2.py [--flavours fv2,fv4] [--rounds 2] [--steps 20] [--warmup 3] [--reps 100] [--out profiles/fv2.json]
"""
import argparse
import ctypes as C
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tools")):
    if p not in sys.path:
        sys.path.insert(0, p)
import hpgmg_b200.api as api  # noqa: E402
from bench_smoothers import COPY_PEAK_GBS, gpu_info  # noqa: E402

# flavour -> (library, a, b, reserved vectors, algorithmic HBM bytes per cell of one GSRB sweep): x, rhs, Dinv and 3 betas
# read, x written (56, the same for both operators); the Helmholtz operator also reads alpha (64)
FLAVOURS = {"fv4": (api.LIB_PATH, 0.0, 1.0, api.VECTORS_RESERVED, 56.0),
            "fv2": (api.FV2_LIB_PATH, 0.0, 1.0, api.VECTORS_RESERVED, 56.0),
            "fv2_helmholtz": (api.FV2_HELMHOLTZ_LIB_PATH, 1.0, 1.0, 11, 64.0)}


def measure(L, flavour, steps, warmup, reps):
    _, a, b, nvec, bytes_per_cell = FLAVOURS[flavour]
    L.hpgmg_b200_set_smoother(api.SMOOTHER_GSRB)
    L.hpgmg_b200_set_bottom_solver(api.BOTTOM_BICGSTAB)
    L.hpgmg_b200_use_graphs(1)
    with api.Hierarchy(7, 8, library=L, a=a, b=b, vectors=nvec) as H:
        lvl = H.level(0)
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
            L.hpgmg_b200_smoother_sweep(lvl, src, dst, api.VECTOR_F, H.a, H.b, s % 2)
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
        gbs = bytes_per_cell * cells / (1e-6 * sweep_us) / 1e9
        return {"flavour": flavour, "a": a, "b": b, "sweep_bytes_per_cell": bytes_per_cell, "levels": H.num_levels, "ghosts": Lc.box_ghosts, "ms_per_solve": ms, "f_cycle_norm": norm,
                "sweep_us": sweep_us, "sweep_gbs": gbs, "sweep_frac_of_copy_peak": gbs / COPY_PEAK_GBS}


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--flavours", default="fv2,fv4", help=f"comma-separated, alternated in this order; of {sorted(FLAVOURS)}")
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--reps", type=int, default=100, help="sweep launches timed (at least 50)")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "fv2.json"))
    args = ap.parse_args()
    if args.reps < 50:
        raise SystemExit("--reps: at least 50 launches")
    flavours = args.flavours.split(",")
    unknown = [f for f in flavours if f not in FLAVOURS]
    if unknown:
        raise SystemExit(f"--flavours: unknown {unknown}; known {sorted(FLAVOURS)}")
    libs = {f: api.lib() if f == "fv4" else api.bind(C.CDLL(FLAVOURS[f][0])) for f in flavours}
    for L in libs.values():
        if L.hpgmg_b200_init(0) != 0:
            raise SystemExit("hpgmg_b200_init(0) failed: a B200 is required")
        L.hpgmg_b200_set_verbose(0)
    card = gpu_info()
    rows = []
    for r in range(args.rounds):
        for flavour in flavours:
            rows.append(dict(measure(libs[flavour], flavour, args.steps, args.warmup, args.reps), round=r))
    print(f"hpgmg-fv 7 8, GSRB, one GPU: {card} (name, power limit, max SM clock)")
    print(f"{'flavour':>13} {'round':>5} {'levels':>6} {'ms/solve':>9} {'sweep us':>9} {'GB/s':>7} {'of copy':>7} {'F-cycle norm':>23}")
    for r in rows:
        print(f"{r['flavour']:>13} {r['round']:5d} {r['levels']:6d} {r['ms_per_solve']:9.3f} {r['sweep_us']:9.1f} {r['sweep_gbs']:7.0f} "
              f"{r['sweep_frac_of_copy_peak']:7.3f} {r['f_cycle_norm']!r:>23}")
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump({"workload": f"hpgmg-fv 7 8, GSRB, BiCGStab, graphs on, one GPU; {' and '.join(flavours)} alternated", "gpu": card,
                   "steps": args.steps, "warmup": args.warmup, "sweep_reps": args.reps, "copy_peak_gbs": COPY_PEAK_GBS, "rows": rows},
                  f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
