"""Checks of the CG bottom solver that need a process of their own (torchrun).  Used by tests/test_gpu_cg.py; prints one line
starting with OK or FAIL.

  check_cg.py ranks <log2> <boxes/rank> <dir>   (under torchrun, or alone for one rank) one FMG solve with CG selected; u of
                                                every box this rank owns goes to <dir>/u_<global box id>.npy
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
import hpgmg_b200.api as api  # noqa: E402


def main():
    mode = sys.argv[1]
    if mode != "ranks":
        raise SystemExit(f"unknown mode {mode}")
    log2, bpr, out = int(sys.argv[2]), int(sys.argv[3]), sys.argv[4]
    rank, world = api.init_distributed()
    L = api.lib()
    H = api.Hierarchy(log2, bpr, my_rank=rank, num_ranks=world, bottom_solver=api.BOTTOM_CG)
    r, _ = H.fmg_solve(0)
    lvl = H.level(0)
    for b in range(lvl.contents.num_my_boxes):
        np.save(os.path.join(out, f"u_{lvl.contents.my_boxes[b].global_box_id}.npy"), api.interior(lvl, api.download(lvl, b, api.VECTOR_U)))
    krylov = H.level(H.num_levels - 1).contents.Krylov_iterations
    print(f"OK rank {rank}/{world} boxes {lvl.contents.num_my_boxes} norm {r!r} bottom iterations {krylov}")
    H.close()
    if world > 1:
        import torch.distributed as dist
        L.hpgmg_b200_comm_finalize()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
