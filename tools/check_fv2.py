"""Runs of the fv2 flavours (hpgmg_b200/lib/libhpgmg_b200_fv2.so, libhpgmg_b200_fv2_helmholtz.so) that need a process of their
own: the kernel-path switches (HPGMG_B200_*) are read once per process, and multi-GPU runs start under torchrun.  Used by
tests/test_gpu_fv2.py and tests/test_gpu_fv2_helmholtz.py; prints one line starting with OK.

  check_fv2.py solve <log2> <boxes/rank> <smoother> <graphs 0|1> <periodic 0|1> <dir> [fv2|fv2_helmholtz]
      two FMG solves; u of every box this rank owns after the second goes to <dir>/u_<global box id>.npy; the line reports the
      residual norms, the kernel launches of each solve and the level-0 must_subtract_mean.  fv2 (the default) solves a = 0,
      b = 1; fv2_helmholtz solves a = b = 1 with the Helmholtz vector map, as the reference driver built with -DUSE_HELMHOLTZ
"""
import ctypes as C
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
import hpgmg_b200.api as api  # noqa: E402

# flavour -> (library, a, b, reserved vectors)
FLAVOURS = {"fv2": (api.FV2_LIB_PATH, 0.0, 1.0, api.VECTORS_RESERVED), "fv2_helmholtz": (api.FV2_HELMHOLTZ_LIB_PATH, 1.0, 1.0, 11)}


def main():
    mode = sys.argv[1]
    if mode != "solve":
        raise SystemExit(f"unknown mode {mode}")
    log2, bpr, smoother, graphs, periodic = (int(a) for a in sys.argv[2:7])
    out = sys.argv[7]
    path, a, b, nvec = FLAVOURS[sys.argv[8] if len(sys.argv) > 8 else "fv2"]
    api._lib = api.bind(C.CDLL(path))                    # api.lib() and init_distributed() then use this flavour
    rank, world = api.init_distributed()
    L = api.lib()
    L.hpgmg_b200_set_smoother(smoother)
    L.hpgmg_b200_use_graphs(graphs)
    L.hpgmg_b200_set_verbose(0)
    H = api.Hierarchy(log2, bpr, my_rank=rank, num_ranks=world, library=L, bc=api.BC_PERIODIC if periodic else api.BC_DIRICHLET,
                      a=a, b=b, vectors=nvec)
    norms, launches = [], []
    for _ in range(2):
        k0 = L.hpgmg_b200_kernel_launches()
        norms.append(H.fmg_solve(0)[0])
        launches.append(L.hpgmg_b200_kernel_launches() - k0)
    lvl = H.level(0)
    for b in range(lvl.contents.num_my_boxes):
        np.save(os.path.join(out, f"u_{lvl.contents.my_boxes[b].global_box_id}.npy"), api.interior(lvl, api.download(lvl, b, api.VECTOR_U)))
    print(f"OK rank {rank}/{world} levels {H.num_levels} norms {norms[0]!r} {norms[1]!r} launches {launches[0]} {launches[1]} "
          f"must_subtract_mean {lvl.contents.must_subtract_mean}")
    H.close()
    if world > 1:
        import torch.distributed as dist
        L.hpgmg_b200_comm_finalize()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
