#!/usr/bin/env python
"""bench.py -- HPGMG-FV fv4 FMG DOF/s on B200 (BASELINE.json metric) + roofline + CPU baseline.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--log2-box-dim 7] [--boxes-per-rank 8]
                  [--smoother gsrb|cheby] [--scaling weak|strong --global-dim 512] [--dump-outputs DIR]

A step is what the reference's bench_hpgmg times (hpgmg-fv.c:78-80): zero_vector(U); FMGSolve(...)
on the finest level.  Workload at N=1: `hpgmg-fv 7 8` = 256^3 as 2^3 boxes of 128^3 (configs[1]);
at N>1 the same `7 8` per rank (weak scaling; the reference only builds cubic domains, so 2 ranks
give 256^3, 4 ranks 384^3, 8 ranks 512^3 -- SURVEY.md appendix B) and value counts the global DOF.
Inputs (1.3 GB of level-0 vectors) are far larger than the 126 MB L2, so no explicit flush is used.

Other BASELINE.json configs: `--log2-box-dim 8` = config 4 (8 boxes of 256^3 per GPU); `--smoother cheby --scaling strong
--global-dim 512` = config 5 (512^3 fixed, 64/N boxes of 128^3 per rank).

`--impl reference` times the UNMODIFIED reference (oracle/_ref, built from /root/reference by
oracle/Makefile) on the host's cores with OpenMP through oracle/_ref/ref_bench.
"""
import argparse
import ctypes as C
import json
import os
import re
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

ALGORITHMIC_BYTES_PER_DOF = 1076.0      # SURVEY.md 8(d): one GSRB F-cycle, per fine-grid DOF
ALGORITHMIC_BYTES_PER_DOF_CHEBY = 1202.0  # the same with 64 B/cell Chebyshev sweeps
GSRB_SWEEP_BYTES_PER_CELL = 56.0        # x, rhs, Dinv, 3 betas read + x written
CHEBY_SWEEP_BYTES_PER_CELL = 64.0       # + x_{n-1} read


def problem_size(log2_box_dim, target_boxes_per_rank, num_ranks):
    """boxes per side exactly as the reference driver picks it (hpgmg-fv.c:184-197); torch-free copy of api.problem_size"""
    box_dim, best = 1 << log2_box_dim, -1
    for bi in range(1, 1000):
        if bi ** 3 <= target_boxes_per_rank * num_ranks:
            odd = box_dim * bi
            while odd % 2 == 0:
                odd //= 2
            if odd <= 11:
                best = bi
    return box_dim, best


def resolve_workload(args, world):
    """(log2_box_dim, boxes_per_rank) of this run and the `config` dict BOTH arms print (byte-identical)."""
    log2, bpr = args.log2_box_dim, args.boxes_per_rank
    if args.scaling == "strong":
        box = 1 << log2
        per_side = args.global_dim // box
        if per_side * box != args.global_dim or per_side ** 3 % world:
            raise SystemExit(f"--global-dim {args.global_dim} is not {world} x whole boxes of {box}^3")
        bpr = per_side ** 3 // world
    box_dim, bi = problem_size(log2, bpr, world)
    dim = box_dim * bi
    cfg = {"workload": f"hpgmg-fv {log2} {bpr} per rank on {world} rank(s): fv4 {args.smoother.upper()} FMG F-cycle on {dim}^3 = {bi}^3 boxes of {box_dim}^3",
           "smoother": args.smoother, "scaling": args.scaling, "global_dim": dim,
           "l2": "level-0 vectors per GPU (>= 1.3 GB) are far larger than the 126 MB L2; no flush between steps"}
    return log2, bpr, dim, bi ** 3, cfg


def golden_norm(log2, total_boxes, smoother):
    """F-cycle residual norm the reference prints for this grid (tests/golden/goldens.json), or None."""
    try:
        with open(os.path.join(ROOT, "tests", "golden", "goldens.json")) as f:
            return json.load(f)["solves"][f"{log2} {total_boxes} {smoother}"]["norms"][0]
    except Exception:
        return None


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        super().__init__(daemon=True)
        self.index, self.samples, self.stop_flag = index, [], False

    def run(self):
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.samples.append([s.strip() for s in out.split(",")])
            except Exception:
                pass
            time.sleep(0.1)

    def summary(self):
        sm = sorted(int(s[0]) for s in self.samples if s and s[0].isdigit())
        mx = [int(s[1]) for s in self.samples if len(s) > 1 and s[1].isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for s in self.samples for n, v in zip(names, s[2:6]) if v.lower().startswith("active")})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


REF_BUILDS = {  # oracle/Makefile: the unmodified reference sources under three sets of flags
    "O2": ("ref_bench{c}", "gcc -O2 -fopenmp (x86-64 baseline ISA, no FMA: the build the goldens come from)"),
    "Ofast-native": ("ref_bench{c}_ofast_native", "gcc -Ofast -march=native -fopenmp (finite-volume/source/README:96; native = the build container's CPU)"),
    "Ofast-v3": ("ref_bench{c}_ofast_v3", "gcc -Ofast -march=x86-64-v3 -fopenmp (AVX2+FMA; used when the -march=native binary cannot run on this host)"),
}


def run_reference(log2_box_dim, boxes, warmup, steps, threads=None, smoother="gsrb", build="O2"):
    """Time the reference's own FMGSolve on the host cores (oracle/_ref/ref_bench*)."""
    exe = os.path.join(ROOT, "oracle", "_ref", REF_BUILDS[build][0].format(c="_cheby" if smoother == "cheby" else ""))
    if not os.path.exists(exe):
        return None
    env = dict(os.environ)
    threads = threads or os.cpu_count() or 1
    env["OMP_NUM_THREADS"] = str(threads)
    try:
        out = subprocess.run([exe, str(log2_box_dim), str(boxes), str(warmup), str(steps)], capture_output=True, text=True, env=env).stdout
    except OSError:
        return None
    m = re.search(r"REF dof=(\d+) seconds_per_solve=([\d.eE+-]+) norm=([\d.eE+-]+) rel=([\d.eE+-]+) threads=(\d+)", out)
    if not m:
        return None          # e.g. SIGILL: a -march=native binary on a different CPU
    return {"dof": float(m.group(1)), "seconds": float(m.group(2)), "norm": float(m.group(3)), "threads": int(m.group(5)),
            "build": build, "flags": REF_BUILDS[build][1]}


def fastest_reference_build(smoother):
    """The reference's README recommends -Ofast -march=native; probe on a tiny problem which optimised binary runs here."""
    for build in ("Ofast-native", "Ofast-v3"):
        if run_reference(4, 1, 0, 1, threads=1, smoother=smoother, build=build) is not None:
            return build
    return "O2"


def reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    world = args.gpus
    log2, bpr, dim, total_boxes, cfg = resolve_workload(args, world)
    # the N-rank problem is the 1-process problem with boxes_per_rank*N boxes (SURVEY.md 8c)
    build = args.ref_build or fastest_reference_build(args.smoother)
    r = run_reference(log2, bpr * world, args.warmup, args.steps, smoother=args.smoother, build=build)
    if r is None:
        emit({"impl": "reference", "unavailable": "oracle/_ref/ref_bench missing (reference not built)"})
        return
    value = r["dof"] / r["seconds"]
    line = {"impl": "reference", "metric": "fmg_dof_per_s", "value": value, "unit": "DOF/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * r["seconds"], "higher_is_better": True,
            "scaling": args.scaling, "vs_baseline": None, "dtype": "f64", "data": "synthetic (analytic problem.fv.c rhs/beta, deterministic)",
            "config": cfg,
            "cpu_baseline": {"value": value, "unit": "DOF/s", "cores": r["threads"], "kind": "reference",
                             "sample": f"{args.steps} FMGSolve after {args.warmup} warm-up, whole workload; reference built {r['flags']}"},
            "e2e": {"value": value, "unit": "DOF/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "f_cycle_norm": r["norm"]}
    emit(line)


def ours(args):
    import hpgmg_b200.api as api
    if os.environ.get("HPGMG_B200_ABLATE"):
        raise SystemExit("bench.py: HPGMG_B200_ABLATE is set -- that switch skips kernels (timing experiments only); refusing to produce a bench line")
    rank, world = api.init_distributed()
    if world != args.gpus and rank == 0:
        print(f"warning: --gpus {args.gpus} but WORLD_SIZE={world}; using WORLD_SIZE", file=sys.stderr)
    L = api.lib()
    dist = None
    if world > 1:
        import torch
        import torch.distributed as dist
    log2, bpr, dim, total_boxes, cfg = resolve_workload(args, world)
    cheby = args.smoother == "cheby"

    H = api.Hierarchy(log2, bpr, my_rank=rank, num_ranks=world, verbose=False, use_graphs=not args.no_graphs,
                      smoother=api.SMOOTHER_CHEBY if cheby else api.SMOOTHER_GSRB)
    lvl = H.level(0)
    dof = float(H.dof(0))
    assert int(round(dof ** (1.0 / 3.0))) == dim

    def barrier():
        L.hpgmg_b200_sync()
        if dist is not None:
            dist.barrier()
            L.hpgmg_b200_sync()

    def allmax(x):
        if dist is None:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def step():
        return H.fmg_solve(0)

    def sweep(s):     # one smoother sweep kernel of level 0, ping-ponging U <-> TEMP like smooth() does
        src, dst = (api.VECTOR_U, api.VECTOR_TEMP) if s % 2 == 0 else (api.VECTOR_TEMP, api.VECTOR_U)
        L.hpgmg_b200_smoother_sweep(lvl, src, dst, api.VECTOR_F, H.a, H.b, s % 6)

    for _ in range(max(args.warmup, 3)):
        norm_r, rel = step()

    if args.ncu:                     # profiling aid: bracket ONE region for `ncu --profile-from-start off` and leave
        L.hpgmg_b200_profiler_start()
        if args.ncu == "solve":
            step()
        elif args.ncu == "sweep":    # two level-0 smoother sweeps (one per colour)
            for s in range(2):
                sweep(s)
        else:                        # one level-0 V-cycle's worth of every operator: residual, restriction, both interpolations
            l1 = H.level(1)
            L.residual(lvl, api.VECTOR_TEMP, api.VECTOR_U, api.VECTOR_F, H.a, H.b)
            L.restriction(l1, api.VECTOR_R, lvl, api.VECTOR_TEMP, api.RESTRICT_CELL)
            L.interpolation_vcycle(lvl, api.VECTOR_U, 1.0, l1, api.VECTOR_U)
            L.interpolation_fcycle(lvl, api.VECTOR_U, 0.0, l1, api.VECTOR_U)
            L.smooth(l1, api.VECTOR_U, api.VECTOR_R, H.a, H.b)          # the second level: 6 x (ghost fill + sweep), L2-resident
            for l in range(2, H.num_levels):                                # one cycle of the coarse end (single-block kernel)
                if H.level(l).contents.dim.i <= 16:
                    L.MGVCycle(H.mg, api.VECTOR_U, api.VECTOR_R, H.a, H.b, l)
                    break
        L.hpgmg_b200_profiler_stop()
        H.close()
        return

    sampler = ClockSampler(int(os.environ.get("LOCAL_RANK", "0")))
    if rank == 0:
        sampler.start()
    launches0 = L.hpgmg_b200_kernel_launches()
    barrier()
    t0 = time.perf_counter()
    L.hpgmg_b200_bench_mark(0)
    for _ in range(args.steps):
        norm_r, rel = step()
    L.hpgmg_b200_bench_mark(1)
    barrier()
    wall = time.perf_counter() - t0
    dev_ms = allmax(L.hpgmg_b200_bench_elapsed_ms(0, 1))
    launches = L.hpgmg_b200_kernel_launches() - launches0
    ms_per_step = dev_ms / args.steps
    value = dof / (1e-3 * ms_per_step)

    if args.dump_outputs:            # before the check below: outputs that differ are the ones worth comparing
        dump_outputs(args.dump_outputs, api, lvl, norm_r, rel, rank, world)
    # the work must be the reference's work: the F-cycle residual norm has to be the one the reference prints for this grid
    gold = golden_norm(log2, total_boxes, args.smoother)
    if gold is not None and norm_r != gold:
        raise SystemExit(f"bench.py: F-cycle residual norm {norm_r!r} differs from the reference's {gold!r} for this grid -- not a valid run")

    # ---- end to end through the C-ABI with HOST buffers (pinned): H2D f, zero u, FMGSolve, D2H u ----
    Lc = lvl.contents
    import numpy as np
    cells = Lc.box_dim ** 3
    nbytes = Lc.num_my_boxes * cells * 8                     # the cells of this rank's boxes, dense
    e2e = None
    if nbytes > 0:
        # two pinned buffer pairs: the solves are submitted as a stream, two in flight, so that the upload of solve n+1 and
        # the download of solve n-1 overlap solve n (hpgmg_fmg_solve_host_submit/_wait).  Every solve uploads its own f
        # from host memory and downloads its own u; nothing is cached between solves.
        f_hosts = [L.hpgmg_b200_host_alloc_pinned(nbytes) for _ in range(2)]
        u_hosts = [L.hpgmg_b200_host_alloc_pinned(nbytes) for _ in range(2)]
        for b in range(Lc.num_my_boxes):
            arr = np.ascontiguousarray(api.interior(lvl, api.download(lvl, b, api.VECTOR_F))).reshape(-1)
            for fh in f_hosts:
                C.memmove(fh + b * cells * 8, arr.ctypes.data, cells * 8)
        solve_args = (H.mg, 0, api.VECTOR_U, api.VECTOR_F, H.a, H.b, 1e-10)

        def stream_of_solves(count):
            tickets, norms = [], []
            for n in range(count):
                if len(tickets) == 2:
                    norms.append(L.hpgmg_fmg_solve_host_wait(H.mg, tickets.pop(0)))
                tickets.append(L.hpgmg_fmg_solve_host_submit(*solve_args, f_hosts[n % 2], u_hosts[n % 2]))
            while tickets:
                norms.append(L.hpgmg_fmg_solve_host_wait(H.mg, tickets.pop(0)))
            return norms

        # (a) one call at a time (latency of a single end-to-end solve)
        for _ in range(2):
            L.hpgmg_fmg_solve_host(*solve_args, f_hosts[0], u_hosts[0])
        barrier()
        te = time.perf_counter()
        for _ in range(args.steps):
            e2e_norm = L.hpgmg_fmg_solve_host(*solve_args, f_hosts[0], u_hosts[0])
        barrier()
        serial_s = allmax((time.perf_counter() - te) / args.steps)
        # (b) the same solves as a stream, two in flight: the throughput figure
        stream_of_solves(3)
        for uh in u_hosts:
            C.memset(uh, 0xFF, nbytes)
        barrier()
        te = time.perf_counter()
        norms = stream_of_solves(args.steps)
        barrier()
        e2e_s = allmax((time.perf_counter() - te) / args.steps)
        moved = int(L.hpgmg_fmg_solve_host_bytes(H.mg, 0))          # f in, u (+ 3 scalars) out, on this rank
        e2e = {"value": dof / e2e_s, "unit": "DOF/s", "h2d_bytes_per_step": moved, "d2h_bytes_per_step": moved + 24,
               "ms_per_step": 1e3 * e2e_s, "f_cycle_norm": e2e_norm,
               "how": "stream of solves through hpgmg_fmg_solve_host_submit/_wait, two in flight: every solve uploads its f from pinned host "
                      "memory and downloads its u; upload of solve n+1 and download of solve n-1 overlap solve n",
               "single_call_ms": 1e3 * serial_s, "single_call_value": dof / serial_s}
        if gold is not None and (e2e_norm != gold or any(x != gold for x in norms)):
            raise SystemExit(f"bench.py: end-to-end F-cycle residual norm {e2e_norm!r} / {norms!r} differs from the reference's {gold!r}")
        u_dev = api.interior(lvl, api.download(lvl, Lc.num_my_boxes - 1, api.VECTOR_U)).reshape(-1)
        for uh in u_hosts:
            u_back = np.ctypeslib.as_array((C.c_double * cells).from_address(uh + (Lc.num_my_boxes - 1) * cells * 8))
            if not np.array_equal(u_back, u_dev):
                raise SystemExit("bench.py: the solution downloaded by the end-to-end call differs from the one on the device")
        for p_ in f_hosts + u_hosts:
            L.hpgmg_b200_host_free_pinned(p_)

    # ---- roofline of the dominant kernel: one level-0 smoother sweep, timed alone with CUDA events ----
    reps = 20
    for s in range(2):
        sweep(s)
    L.hpgmg_b200_bench_mark(2)
    for s in range(reps):
        sweep(s)
    L.hpgmg_b200_bench_mark(3)
    L.hpgmg_b200_sync()
    sweep_ms = L.hpgmg_b200_bench_elapsed_ms(2, 3) / reps
    local_cells = Lc.num_my_boxes * Lc.box_dim ** 3
    peak, peak_src = measured_peaks()
    per_cell = CHEBY_SWEEP_BYTES_PER_CELL if cheby else GSRB_SWEEP_BYTES_PER_CELL
    per_dof = ALGORITHMIC_BYTES_PER_DOF_CHEBY if cheby else ALGORITHMIC_BYTES_PER_DOF
    achieved = per_cell * local_cells / (1e-3 * sweep_ms) / 1e9
    roofline = {"bound": "hbm", "kernel": f"{args.smoother}_sweep(level 0)", "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": None, "peak_source": peak_src, "us_per_launch": 1e3 * sweep_ms,
                "algorithmic_bytes_per_launch": per_cell * local_cells,
                "solve_frac_of_hbm_roofline": (value / max(world, 1)) * per_dof / (peak * 1e9)}
    ncu = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(ncu):          # DRAM bytes of the ncu capture, only for the configuration that was captured
        with open(ncu) as f:
            t = json.load(f)
        if t.get("local_cells") == local_cells and t.get("smoother", "gsrb") == args.smoother:
            roofline["traffic"] = t.get("sweep_dram_bytes_per_launch")

    if rank == 0:
        sampler.stop_flag = True
        sampler.join(timeout=2)
        # ---- CPU baseline: the reference itself on this box's cores, bounded sample ----
        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            build = fastest_reference_build(args.smoother)
            small = local_cells <= 256 ** 3
            r = run_reference(log2, bpr, 1, 3 if small else 1, smoother=args.smoother, build=build)
            if r:
                cpu = {"value": r["dof"] / r["seconds"], "unit": "DOF/s", "cores": r["threads"], "kind": "reference",
                       "sample": f"{3 if small else 1} FMGSolve (after 1 warm-up) of the same {dim}^3 workload; reference built {r['flags']}",
                       "f_cycle_norm": r["norm"]}
                if small and build != "O2":
                    r2 = run_reference(log2, bpr, 1, 2, smoother=args.smoother, build="O2")
                    if r2:
                        cpu["value_O2_build"] = r2["dof"] / r2["seconds"]
                        cpu["f_cycle_norm_O2_build"] = r2["norm"]
        line = {"metric": "fmg_dof_per_s", "value": value, "unit": "DOF/s", "n_gpus": world, "steps": args.steps,
                "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": args.scaling,
                "vs_baseline": None, "dtype": "f64", "data": "synthetic (analytic problem.fv.c rhs/beta, deterministic)",
                "config": cfg,
                "levels": H.num_levels, "boxes_on_rank0": Lc.num_my_boxes, "cuda_graphs": not args.no_graphs,
                "timing": "CUDA events on the library stream, max over ranks",
                "gpu_launches": int(launches), "wall_ms_per_step": 1e3 * wall / args.steps,
                "f_cycle_norm": norm_r, "f_cycle_rel": rel, "f_cycle_norm_reference": gold,
                "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "clocks": sampler.summary()}
        emit(line)
    H.close()
    if dist is not None:
        L.hpgmg_b200_comm_finalize()
        dist.destroy_process_group()


DUMP_SAMPLE_CELLS = 1 << 22             # 32 MB of float64 over all ranks: a fixed sample of u where the grid has more cells


def dump_outputs(out_dir, api, lvl, norm_r, rel, rank, world):
    """What the last timed FMGSolve gave its caller: u on the cells of this rank's level-0 boxes (box by box, [k][j][i],
    a sample at fixed seeded positions when there are more than this rank's share of DUMP_SAMPLE_CELLS) and the F-cycle
    residual norm."""
    import numpy as np
    Lc = lvl.contents
    u = np.concatenate([np.ascontiguousarray(api.interior(lvl, api.download(lvl, b, api.VECTOR_U))).reshape(-1)
                        for b in range(Lc.num_my_boxes)])
    share = DUMP_SAMPLE_CELLS // world
    if u.size > share:
        u = u[np.sort(np.random.default_rng(rank).choice(u.size, share, replace=False))]
    suffix = f"_rank{rank}" if world > 1 else ""
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, f"u{suffix}.npy"), u.astype(np.float64))
    np.save(os.path.join(out_dir, f"f_cycle_norm{suffix}.npy"), np.array([norm_r, rel], dtype=np.float64))


_REAL_STDOUT = None


def emit(line):
    """The ONE JSON line of the contract, on the process's original stdout."""
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def main():
    # libraries (NCCL's version banner, torchrun) may write to fd 1: keep the real stdout for the JSON line only
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--log2-box-dim", type=int, default=7)
    ap.add_argument("--boxes-per-rank", type=int, default=8)
    ap.add_argument("--smoother", default="gsrb", choices=["gsrb", "cheby"])
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"], help="strong: --global-dim^3 split over the ranks (BASELINE config 5)")
    ap.add_argument("--global-dim", type=int, default=512)
    ap.add_argument("--ref-build", default="", choices=["", "O2", "Ofast-native", "Ofast-v3"], help="--impl reference: which build of the reference (default: the fastest that runs here)")
    ap.add_argument("--no-graphs", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="after the timed steps, write u of the last one (a fixed sample on large grids) and its residual norm to DIR/*.npy")
    ap.add_argument("--ncu", default="", choices=["", "solve", "sweep", "ops"], help="bracket one solve / two smoother sweeps / residual+restriction+interpolations of level 0 with cudaProfilerStart/Stop and exit")
    args = ap.parse_args()
    if args.impl == "reference":
        reference_arm(args)
    else:
        ours(args)


if __name__ == "__main__":
    main()
