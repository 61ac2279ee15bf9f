"""What an FMG solve costs when f and u live on the GPU, against the other two ways in, on one GPU in one process:
`hpgmg-fv 7 8` (256^3), GSRB, BiCGStab, recorded graphs.  The three calls are alternated, --rounds times, --steps calls each:

  resident  zero_vector(U) + FMGSolve on the library's own F (Hierarchy.fmg_solve; nothing crosses the API)
  device    Hierarchy.fmg_solve_device on a (256, 256, 256) float64 torch tensor, into a preallocated one
  host      hpgmg_fmg_solve_host with pinned host buffers (upload f, solve, download u)

Each call ends in a synchronisation, so the host clock around --steps calls gives ms per call; the library's CUDA events around
the same calls give the device time.  Then the two kernels the device call adds are timed alone with CUDA events around --reps
launches each: the grid unpack (F <- f, R <- f, max|f|, with the 8-byte reset of the norm slot before it) and the grid pack
(u -> out), with GB/s from the byte model below.  The device call's u and norm are checked against the host call's, bit for bit.
Prints a table, the card's name and power limit, and writes JSON (--out, default profiles/device_solve.json).

  python tools/bench_device_solve.py [--rounds 3] [--steps 20] [--warmup 3] [--reps 100] [--out profiles/device_solve.json]
"""
import argparse
import ctypes as C
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tools")):
    if p not in sys.path:
        sys.path.insert(0, p)
import hpgmg_b200.api as api  # noqa: E402
from bench_smoothers import gpu_info  # noqa: E402

UNPACK_BYTES_PER_CELL = 24.0          # f read, F and R written
PACK_BYTES_PER_CELL = 16.0            # u read, out written
SCRATCH_SLOT = 9                      # a scratch scalar slot of the library (HPGMG_SLOT_SCRATCH + 1, runtime.h)


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--reps", type=int, default=100, help="launches of each grid kernel timed (at least 50)")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "device_solve.json"))
    args = ap.parse_args()
    if args.reps < 50:
        raise SystemExit("--reps: at least 50 launches")
    import torch
    api.init(0)
    L = api.lib()
    # the grid kernels alone: internal entry points of the library (runtime.h), exported like every extern "C" function
    L.hpgmg_grid_unpack_copy_norm_async.restype = None
    L.hpgmg_grid_unpack_copy_norm_async.argtypes = [C.POINTER(api.level_type), C.c_int, C.c_int, C.c_void_p, C.c_int]
    L.hpgmg_grid_pack_async.restype = None
    L.hpgmg_grid_pack_async.argtypes = [C.POINTER(api.level_type), C.c_int, C.c_void_p]
    card = gpu_info()
    dev = torch.device("cuda", L.hpgmg_b200_device())
    with api.Hierarchy(7, 8, smoother=api.SMOOTHER_GSRB, bottom_solver=api.BOTTOM_BICGSTAB, use_graphs=True) as H:
        lvl = H.level(0)
        Lc = lvl.contents
        n, nb = Lc.box_dim, Lc.num_my_boxes
        cells = nb * n ** 3
        shape = (Lc.dim.k, Lc.dim.j, Lc.dim.i)
        lows = [(Lc.my_boxes[b].low.i, Lc.my_boxes[b].low.j, Lc.my_boxes[b].low.k) for b in range(nb)]
        f_boxes = np.concatenate([np.ascontiguousarray(api.interior(lvl, api.download(lvl, b, api.VECTOR_F))).reshape(-1) for b in range(nb)])
        f_grid = np.empty(shape)
        for b, (i, j, k) in enumerate(lows):
            f_grid[k:k + n, j:j + n, i:i + n] = f_boxes[b * n ** 3:(b + 1) * n ** 3].reshape(n, n, n)
        nbytes = f_boxes.nbytes
        f_host, u_host = L.hpgmg_b200_host_alloc_pinned(nbytes), L.hpgmg_b200_host_alloc_pinned(nbytes)
        C.memmove(f_host, f_boxes.ctypes.data, nbytes)
        f_t = torch.from_numpy(f_grid).to(dev)
        u_t = torch.zeros(shape, dtype=torch.float64, device=dev)
        torch.cuda.synchronize(dev)
        host_args = (H.mg, 0, api.VECTOR_U, api.VECTOR_F, H.a, H.b, 1e-10, f_host, u_host)
        calls = {"resident": lambda: H.fmg_solve(0)[0],
                 "device": lambda: H.fmg_solve_device(f_t, out=u_t)[1][0],
                 "host": lambda: L.hpgmg_fmg_solve_host(*host_args)}
        rows = []
        for r in range(args.rounds):
            for name, call in calls.items():
                for _ in range(args.warmup):
                    call()
                L.hpgmg_b200_sync()
                L.hpgmg_b200_bench_mark(0)
                t0 = time.perf_counter()
                for _ in range(args.steps):
                    norm = call()
                wall_ms = 1e3 * (time.perf_counter() - t0) / args.steps
                L.hpgmg_b200_bench_mark(1)
                L.hpgmg_b200_sync()
                rows.append({"call": name, "round": r, "ms_per_call": wall_ms,
                             "device_ms_per_call": L.hpgmg_b200_bench_elapsed_ms(0, 1) / args.steps, "f_cycle_norm": norm})
        # the device call gives the host call's bits
        r_host = L.hpgmg_fmg_solve_host(*host_args)
        u_boxes = np.ctypeslib.as_array((C.c_double * cells).from_address(u_host)).copy()
        u_t.zero_()
        _, (r_dev, _) = H.fmg_solve_device(f_t, out=u_t)
        u_grid = u_t.cpu().numpy()
        same_u = all(np.array_equal(u_grid[k:k + n, j:j + n, i:i + n].reshape(-1), u_boxes[b * n ** 3:(b + 1) * n ** 3])
                     for b, (i, j, k) in enumerate(lows))
        if r_dev != r_host or not same_u:
            raise SystemExit(f"the device call differs from the host call: norm {r_dev!r} vs {r_host!r}, u equal: {same_u}")
        # the two grid kernels alone
        kern = {}
        for name, launch, bpc in (("unpack", lambda: L.hpgmg_grid_unpack_copy_norm_async(lvl, api.VECTOR_F, api.VECTOR_R, f_t.data_ptr(), SCRATCH_SLOT),
                                   UNPACK_BYTES_PER_CELL),
                                  ("pack", lambda: L.hpgmg_grid_pack_async(lvl, api.VECTOR_U, u_t.data_ptr()), PACK_BYTES_PER_CELL)):
            for _ in range(5):
                launch()
            L.hpgmg_b200_bench_mark(2)
            for _ in range(args.reps):
                launch()
            L.hpgmg_b200_bench_mark(3)
            L.hpgmg_b200_sync()
            us = 1e3 * L.hpgmg_b200_bench_elapsed_ms(2, 3) / args.reps
            kern[name] = {"us": us, "bytes": bpc * cells, "bytes_per_cell": bpc, "gbs": bpc * cells / (1e-6 * us) / 1e9}
        L.hpgmg_b200_host_free_pinned(f_host)
        L.hpgmg_b200_host_free_pinned(u_host)

    def best(name, key):
        return min(r[key] for r in rows if r["call"] == name)
    print(f"hpgmg-fv 7 8 ({shape[0]}^3), GSRB, graphs on, one GPU: {card} (name, power limit, max SM clock)")
    print(f"{'call':>9} {'round':>5} {'ms/call':>8} {'device ms':>9} {'F-cycle norm':>23}")
    for r in rows:
        print(f"{r['call']:>9} {r['round']:5d} {r['ms_per_call']:8.3f} {r['device_ms_per_call']:9.3f} {r['f_cycle_norm']!r:>23}")
    for name, k in kern.items():
        print(f"grid {name:>6}: {k['us']:7.1f} us  {k['bytes'] / 1e6:6.0f} MB  {k['gbs']:6.0f} GB/s")
    added = best("device", "ms_per_call") - best("resident", "ms_per_call")
    print(f"device call - resident solve (best of rounds): {added:.3f} ms; grid kernels alone: {(kern['unpack']['us'] + kern['pack']['us']) / 1e3:.3f} ms")
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump({"workload": f"hpgmg-fv 7 8 ({shape[0]}^3 as {nb} boxes of {n}^3), GSRB, BiCGStab, graphs on, one GPU; resident / device / host alternated",
                   "gpu": card, "steps": args.steps, "warmup": args.warmup, "kernel_reps": args.reps,
                   "device_equals_host": True, "rows": rows, "grid_kernels": kern,
                   "device_minus_resident_ms": added}, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
