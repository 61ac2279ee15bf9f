"""Checks of the Jacobi and L1-Jacobi smoothers that need a process of their own (environment switches, torchrun, a fatal
error).  Used by tests/test_gpu_jacobi.py; each mode prints one line starting with OK or FAIL.

  check_jacobi.py compose <log2> <boxes> jacobi|l1jacobi   one smooth() on level 0 against six steps of apply_op + the update
                                                           in numpy (the kernels chosen by the HPGMG_B200_* switches in effect)
  check_jacobi.py ranks <log2> <boxes/rank> jacobi|l1jacobi <dir>   (under torchrun) one FMG solve; u of every box this rank
                                                           owns goes to <dir>/u_<global box id>.npy
  check_jacobi.py late                                     a hierarchy built under GSRB, then switched to L1-Jacobi: smooth()
                                                           must stop the process with a message
"""
import ctypes as C
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
import hpgmg_b200.api as api  # noqa: E402

SMOOTHERS = {"jacobi": api.SMOOTHER_JACOBI, "l1jacobi": api.SMOOTHER_L1JACOBI}
WEIGHT = {api.SMOOTHER_JACOBI: 2.0 / 3.0, api.SMOOTHER_L1JACOBI: 1.0}     # jacobi.c


def l1inv(L, level, box):
    Lc = level.contents
    out = np.empty(Lc.box_volume, dtype=np.float64)
    L.hpgmg_download_l1inv(level, box, out.ctypes.data_as(C.c_void_p))
    return api.box_view(level, out)


def download(L, level, box, vid):
    out = np.empty(level.contents.box_volume, dtype=np.float64)
    L.hpgmg_download_box_vector(level, box, vid, out.ctypes.data_as(C.c_void_p))
    return api.box_view(level, out)


def upload(L, level, box, vid, a):
    L.hpgmg_upload_box_vector(level, box, vid, np.ascontiguousarray(a, dtype=np.float64).ctypes.data_as(C.c_void_p))


def smooth_vs_composition(L, H, smoother, seed, a=0.0, b=1.0):
    """smooth(level 0, U, R) from seeded random U and R (ghosts included) against six steps of: apply_op(E <- source), which
    fills the source's ghosts, then dst = src + (w*lambda)*(R - E) on the cells in numpy, uploaded.  lambda is read back:
    Dinv for Jacobi, the L1 row inverse for L1-Jacobi.  Returns a list of mismatches (empty: every cell of every box equal)."""
    lvl = H.level(0)
    Lc = lvl.contents
    nb, n, g = Lc.num_my_boxes, Lc.box_dim, Lc.box_ghosts
    s = slice(g, g + n)
    U, R, E, T = api.VECTOR_U, api.VECTOR_R, api.VECTOR_E, api.VECTOR_TEMP
    rng = np.random.default_rng(seed)
    shape = (n + 2 * g, n + 2 * g, Lc.box_jStride)
    u0 = [rng.standard_normal(shape) for _ in range(nb)]
    r0 = [rng.standard_normal(shape) for _ in range(nb)]
    lam = [l1inv(L, lvl, box) if smoother == api.SMOOTHER_L1JACOBI else download(L, lvl, box, api.VECTOR_DINV) for box in range(nb)]
    w = WEIGHT[smoother]
    for box in range(nb):
        upload(L, lvl, box, U, u0[box])
        upload(L, lvl, box, R, r0[box])
    L.smooth(lvl, U, R, a, b)
    got = {(box, v): download(L, lvl, box, v)[s, s, s].copy() for box in range(nb) for v in (U, T)}
    for box in range(nb):
        upload(L, lvl, box, U, u0[box])
    for step in range(6):
        src, dst = (U, T) if step % 2 == 0 else (T, U)
        L.apply_op(lvl, E, src, a, b)
        for box in range(nb):
            x = download(L, lvl, box, src)
            ax = download(L, lvl, box, E)
            out = x.copy()
            out[s, s, s] = x[s, s, s] + (w * lam[box][s, s, s]) * (r0[box][s, s, s] - ax[s, s, s])
            upload(L, lvl, box, dst, out)
    bad = []
    for box in range(nb):
        for v in (U, T):
            want = download(L, lvl, box, v)[s, s, s]
            if not np.array_equal(got[(box, v)], want):
                bad.append(f"box {box} vector {v}: {int(np.sum(got[(box, v)] != want))} cells differ, max |diff| {np.max(np.abs(got[(box, v)] - want)):.3e}")
    return bad


def main():
    mode = sys.argv[1]
    if mode == "compose":
        log2, boxes, name = int(sys.argv[2]), int(sys.argv[3]), sys.argv[4]
        api.init(0)
        L = api.lib()
        with api.Hierarchy(log2, boxes, smoother=SMOOTHERS[name], use_graphs=False) as H:
            bad = smooth_vs_composition(L, H, SMOOTHERS[name], seed=log2 * 1000 + boxes)
        print(("OK" if not bad else "FAIL") + f" compose {log2} {boxes} {name}", *bad[:8], sep="\n  ")
    elif mode == "ranks":
        log2, bpr, name, out = int(sys.argv[2]), int(sys.argv[3]), sys.argv[4], sys.argv[5]
        rank, world = api.init_distributed()
        L = api.lib()
        H = api.Hierarchy(log2, bpr, my_rank=rank, num_ranks=world, smoother=SMOOTHERS[name])
        r, _ = H.fmg_solve(0)
        lvl = H.level(0)
        for b in range(lvl.contents.num_my_boxes):
            np.save(os.path.join(out, f"u_{lvl.contents.my_boxes[b].global_box_id}.npy"), api.interior(lvl, api.download(lvl, b, api.VECTOR_U)))
        print(f"OK rank {rank}/{world} boxes {lvl.contents.num_my_boxes} norm {r!r}")
        H.close()
        if world > 1:
            import torch.distributed as dist
            L.hpgmg_b200_comm_finalize()
            dist.destroy_process_group()
    elif mode == "late":
        api.init(0)
        L = api.lib()
        with api.Hierarchy(4, 8, smoother=api.SMOOTHER_GSRB, use_graphs=False) as H:
            L.hpgmg_b200_set_smoother(api.SMOOTHER_L1JACOBI)
            sys.stdout.flush()
            L.smooth(H.level(0), api.VECTOR_U, api.VECTOR_F, 0.0, 1.0)
            L.hpgmg_b200_sync()
        print("FAIL: smooth() ran L1-Jacobi on a level without the L1 row inverse")
    else:
        raise SystemExit(f"unknown mode {mode}")


if __name__ == "__main__":
    main()
