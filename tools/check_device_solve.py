"""One FMG solve through Hierarchy.fmg_solve_device in a process of its own (under torchrun, or alone for one rank).  Used by
tests/test_gpu_device_solve.py; prints one line starting with OK.

  check_device_solve.py <log2> <boxes/rank> <dir>

Every rank passes the same seeded whole-domain f and a zero-initialised u, and writes to <dir>: u_<rank>.npy (its u, all cells),
owned_<rank>.npy (True at the cells of its boxes) and norm_<rank>.npy (the F-cycle residual norm).
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
import hpgmg_b200.api as api  # noqa: E402


def main():
    log2, bpr, out = int(sys.argv[1]), int(sys.argv[2]), sys.argv[3]
    rank, world = api.init_distributed()
    import torch
    L = api.lib()
    L.hpgmg_b200_set_verbose(0)
    H = api.Hierarchy(log2, bpr, my_rank=rank, num_ranks=world)
    lvl = H.level(0).contents
    shape = (lvl.dim.k, lvl.dim.j, lvl.dim.i)
    dev = torch.device("cuda", L.hpgmg_b200_device())
    f = torch.from_numpy(np.random.default_rng(20261022).standard_normal(shape)).to(dev)
    u, (r, _) = H.fmg_solve_device(f)
    owned = np.zeros(shape, dtype=bool)
    n = lvl.box_dim
    for b in range(lvl.num_my_boxes):
        lo = lvl.my_boxes[b].low
        owned[lo.k:lo.k + n, lo.j:lo.j + n, lo.i:lo.i + n] = True
    np.save(os.path.join(out, f"u_{rank}.npy"), u.cpu().numpy())
    np.save(os.path.join(out, f"owned_{rank}.npy"), owned)
    np.save(os.path.join(out, f"norm_{rank}.npy"), np.array(r))
    print(f"OK rank {rank}/{world} boxes {lvl.num_my_boxes} norm {r!r}")
    H.close()
    if world > 1:
        import torch.distributed as dist
        L.hpgmg_b200_comm_finalize()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
