"""GPU suite (-m gpu): hpgmg_fmg_solve_device and Hierarchy.fmg_solve_device -- the FMG solve that reads f from and writes u to
CUDA tensors of the level's whole domain ([k][j][i], i fastest).  Every result is compared bit for bit, tolerance 0, with
hpgmg_fmg_solve_host on the same f in the host call's box-major layout: u of every cell, the returned norm and the norms the
library records.  Also: every library flavour, in-place solves, ordering with the caller's torch stream, the bound on recorded
graphs, the refusal of unusable tensors, and two GPUs against one process."""
import ctypes as C
import os
import subprocess
import sys
import zlib

import numpy as np
import pytest
import torch

import hpgmg_b200.api as api

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TOOL = os.path.join(ROOT, "tools", "check_device_solve.py")
U, F = api.VECTOR_U, api.VECTOR_F
HELM_LIB = os.path.join(os.path.dirname(api.LIB_PATH), "libhpgmg_b200_helmholtz.so")


@pytest.fixture
def lib(gpu_lib):
    yield gpu_lib
    gpu_lib.hpgmg_b200_set_smoother(api.SMOOTHER_GSRB)
    gpu_lib.hpgmg_b200_use_graphs(1)


# ---------------------------------------------------------------------------------- box-major <-> whole-domain grid
def box_lows(lvl):
    Lc = lvl.contents
    return [(Lc.my_boxes[b].low.i, Lc.my_boxes[b].low.j, Lc.my_boxes[b].low.k) for b in range(Lc.num_my_boxes)]


def grid_shape(lvl):
    d = lvl.contents.dim
    return (d.k, d.j, d.i)


def box_major_to_grid(lvl, dense, fill=0.0):
    """the host call's layout (this rank's boxes, [box][k][j][i]) -> a (dim.k, dim.j, dim.i) array; cells of no box get `fill`"""
    n = lvl.contents.box_dim
    grid = np.full(grid_shape(lvl), fill)
    for b, (i, j, k) in enumerate(box_lows(lvl)):
        grid[k:k + n, j:j + n, i:i + n] = dense[b * n ** 3:(b + 1) * n ** 3].reshape(n, n, n)
    return grid


def grid_to_box_major(lvl, grid):
    n = lvl.contents.box_dim
    return np.concatenate([np.ascontiguousarray(grid[k:k + n, j:j + n, i:i + n]).reshape(-1) for (i, j, k) in box_lows(lvl)])


def problem_f(lvl):
    """F of the problem as initialize_problem wrote it, box-major"""
    return np.concatenate([np.ascontiguousarray(api.interior(lvl, api.download(lvl, b, F))).reshape(-1)
                           for b in range(lvl.contents.num_my_boxes)])


def random_f(lvl, *key, mean_zero=False):
    f = np.random.default_rng(zlib.crc32(repr(key).encode())).standard_normal(lvl.contents.num_my_boxes * lvl.contents.box_dim ** 3)
    return f - f.mean() if mean_zero else f


def host_solve(L, H, f):
    """hpgmg_fmg_solve_host on box-major f: (u box-major, returned norm, recorded ||r||, recorded ||F||)"""
    u = np.full_like(f, np.nan)
    r = L.hpgmg_fmg_solve_host(H.mg, 0, U, F, H.a, H.b, 1e-10, f.ctypes.data_as(C.c_void_p), u.ctypes.data_as(C.c_void_p))
    return u, r, L.hpgmg_last_norm_of_residual(H.mg), L.hpgmg_last_norm_of_F(H.mg)


def device(L):
    return torch.device("cuda", L.hpgmg_b200_device())


def device_solve_equals_host(L, H, f, in_place=False):
    """the device call on the grid of f gives the host call's u (every cell) and norms, bit for bit"""
    lvl = H.level(0)
    want_u, want_r, want_rec, want_nf = host_solve(L, H, f)
    fg = torch.from_numpy(box_major_to_grid(lvl, f)).to(device(L))
    u, (r, rel) = H.fmg_solve_device(fg, out=fg if in_place else None)
    assert (u is fg) == in_place
    assert r == want_r == want_rec, (r, want_r, want_rec)
    assert L.hpgmg_last_norm_of_residual(H.mg) == want_rec and L.hpgmg_last_norm_of_F(H.mg) == want_nf
    assert rel == r / want_nf
    np.testing.assert_array_equal(grid_to_box_major(lvl, u.cpu().numpy()), want_u)
    return u


# ------------------------------------------------------------------------------------------------------ the same bits
@pytest.mark.parametrize("graphs", [True, False], ids=["graphs", "stream"])
@pytest.mark.parametrize("smoother", [api.SMOOTHER_GSRB, api.SMOOTHER_CHEBY], ids=["gsrb", "cheby"])
@pytest.mark.parametrize("cfg", ["5 8", "6 8"])
def test_same_bits_as_the_host_call(lib, cfg, smoother, graphs):
    log2, boxes = map(int, cfg.split())
    with api.Hierarchy(log2, boxes, smoother=smoother, use_graphs=graphs) as H:
        lvl = H.level(0)
        assert lvl.contents.num_my_boxes == lvl.contents.boxes_in.i ** 3          # one rank: the grid is every cell
        fs = [problem_f(lvl), random_f(lvl, "device solve", cfg, smoother)]
        for f in fs + fs:                                                          # graphs: record, then replay
            device_solve_equals_host(lib, H, f)


# ------------------------------------------------------------------------------------------------------ every flavour
def test_periodic(lib):
    with api.Hierarchy(5, 8, bc=api.BC_PERIODIC) as H:
        lvl = H.level(0)
        assert lvl.contents.must_subtract_mean == 1
        for f in (problem_f(lvl), random_f(lvl, "device solve periodic", mean_zero=True)):
            device_solve_equals_host(lib, H, f)


@pytest.mark.parametrize("flavour", ["helmholtz", "fv2", "fv2_helmholtz"])
def test_every_flavour(gpu_lib, flavour):
    path, a, b, nvec = {"helmholtz": (HELM_LIB, 1.0, 1.0, 11), "fv2": (api.FV2_LIB_PATH, 0.0, 1.0, None),
                        "fv2_helmholtz": (api.FV2_HELMHOLTZ_LIB_PATH, 1.0, 1.0, 11)}[flavour]
    L = api.bind(C.CDLL(path))
    assert L.hpgmg_b200_init(0) == 0
    L.hpgmg_b200_set_verbose(0)
    with api.Hierarchy(5, 8, library=L, a=a, b=b, vectors=nvec) as H:
        lvl = H.level(0)
        for f in (problem_f(lvl), random_f(lvl, "device solve", flavour)):
            device_solve_equals_host(L, H, f)


# ------------------------------------------------------------------------------------------------- in place, ordering
def test_in_place(lib):
    with api.Hierarchy(5, 8) as H:
        device_solve_equals_host(lib, H, random_f(H.level(0), "device solve in place"), in_place=True)


def test_waits_for_the_callers_stream(lib):
    """f is produced on a fresh torch stream by a chain of ops queued behind a long-running kernel, without synchronising; the
    solve is called with that stream current and must read the finished f."""
    with api.Hierarchy(6, 8) as H:
        lvl = H.level(0)
        f = random_f(lvl, "device solve stream order")
        want_u, want_r, _, _ = host_solve(lib, H, f)
        src = torch.from_numpy(box_major_to_grid(lvl, f)).to(device(lib))
        torch.cuda.synchronize()
        s = torch.cuda.Stream(device=device(lib))
        with torch.cuda.stream(s):
            torch.cuda._sleep(100_000_000)                 # tens of milliseconds of one spinning kernel on s
            g = src * 4.0                                  # scalings by powers of two: exact
            g = g + 0.0
            g = g * 0.25
            u, (r, _) = H.fmg_solve_device(g)
        assert r == want_r
        np.testing.assert_array_equal(grid_to_box_major(lvl, u.cpu().numpy()), want_u)


# -------------------------------------------------------------------------------------------------- recorded graphs
def test_recorded_graphs_do_not_grow_with_new_tensors(lib):
    with api.Hierarchy(5, 8) as H:
        lvl = H.level(0)
        f = random_f(lvl, "device solve graphs")
        want_u, want_r, _, _ = host_solve(lib, H, f)
        fg = box_major_to_grid(lvl, f)
        before = lib.hpgmg_b200_recorded_graphs()
        counts = []
        for _ in range(11):
            ft = torch.from_numpy(fg).to(device(lib))
            out = torch.full(grid_shape(lvl), float("nan"), dtype=torch.float64, device=device(lib))
            u, (r, _) = H.fmg_solve_device(ft, out=out)
            assert r == want_r
            np.testing.assert_array_equal(grid_to_box_major(lvl, u.cpu().numpy()), want_u)
            counts.append(lib.hpgmg_b200_recorded_graphs())
            del ft, out, u
        assert counts[0] == before + 1, "the first call records the solve"
        assert counts[1:] == [counts[0]] * 10, counts


# -------------------------------------------------------------------------------------------------------- refusals
def test_unusable_tensors_are_refused(lib):
    with api.Hierarchy(5, 8) as H:
        lvl = H.level(0)
        shape = grid_shape(lvl)
        dev = device(lib)
        good = torch.zeros(shape, dtype=torch.float64, device=dev)
        cells = good.numel()
        bad = [(TypeError, "must be a torch.Tensor", np.zeros(shape)),
               (TypeError, "must be float64", torch.zeros(shape, dtype=torch.float32, device=dev)),
               (ValueError, "is on cpu", torch.zeros(shape, dtype=torch.float64)),
               (ValueError, "has shape", torch.zeros((shape[0], shape[1], shape[2] // 2), dtype=torch.float64, device=dev)),
               (ValueError, "must be contiguous", good.transpose(0, 2)),
               (ValueError, "16-byte boundary", torch.zeros(cells + 1, dtype=torch.float64, device=dev)[1:].view(shape))]
        for exc, msg, t in bad:
            with pytest.raises(exc, match=msg):
                H.fmg_solve_device(t)
            with pytest.raises(exc, match=msg):
                H.fmg_solve_device(good, out=t)
        device_solve_equals_host(lib, H, random_f(lvl, "device solve after refusals"))


def test_the_c_call_refuses_host_memory(gpu_lib):
    """hpgmg_fmg_solve_device itself checks its pointers: host memory ends the process with a message, before any work."""
    code = ("import ctypes as C, numpy as np, hpgmg_b200.api as api\n"
            "api.init(0)\n"
            "L = api.lib()\n"
            "L.hpgmg_b200_set_verbose(0)\n"
            "H = api.Hierarchy(4, 8)\n"
            "n = H.level(0).contents.dim.i\n"
            "f = np.zeros(n ** 3)\n"
            "L.hpgmg_fmg_solve_device(H.mg, 0, api.VECTOR_U, api.VECTOR_F, 0.0, 1.0, 1e-10, f.ctypes.data, f.ctypes.data, None)\n"
            "print('returned')\n")
    r = subprocess.run([sys.executable, "-c", code], cwd=ROOT, capture_output=True, text=True, timeout=300)
    assert r.returncode == 1, (r.returncode, r.stdout[-2000:], r.stderr[-2000:])
    assert "f_dev" in r.stderr and "is not device memory" in r.stderr, r.stderr[-2000:]
    assert "returned" not in r.stdout


# ---------------------------------------------------------------------------------------------------- two GPUs
def _gpu_count():
    try:
        return len([l for l in subprocess.run(["nvidia-smi", "-L"], capture_output=True, text=True).stdout.splitlines() if l.startswith("GPU ")])
    except Exception:
        return 0


def test_two_gpus_equal_one_process(gpu_lib, tmp_path):
    """`6 8` on 2 ranks, every rank passing the whole-domain f: each rank writes exactly the cells of its boxes, with the values of
    the single-process run of the same grid, and leaves the other cells of its zero-initialised u untouched."""
    ranks = 2
    if _gpu_count() < ranks:
        pytest.skip(f"needs {ranks} GPUs")
    one, many = tmp_path / "one", tmp_path / "many"
    one.mkdir()
    many.mkdir()
    e = {k: v for k, v in os.environ.items() if k not in ("RANK", "WORLD_SIZE")}
    r = subprocess.run([sys.executable, TOOL, "6", str(8 * ranks), str(one)], capture_output=True, text=True, timeout=600, env=e)
    assert r.stdout.startswith("OK"), r.stdout[-2000:] + r.stderr[-2000:]
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={ranks}", "--master-addr", "127.0.0.1",
                        "--master-port", "29761", TOOL, "6", "8", str(many)], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    u1 = np.load(one / "u_0.npy")
    norm1 = float(np.load(one / "norm_0.npy"))
    owned = np.zeros(u1.shape, dtype=int)
    for rank in range(ranks):
        u = np.load(many / f"u_{rank}.npy")
        mine = np.load(many / f"owned_{rank}.npy")
        assert mine.any()
        np.testing.assert_array_equal(u[mine], u1[mine], err_msg=f"rank {rank}")
        assert (u[~mine] == 0.0).all(), f"rank {rank} wrote cells of another rank's boxes"
        assert float(np.load(many / f"norm_{rank}.npy")) == norm1
        owned += mine
    assert (owned == 1).all(), "every cell belongs to exactly one rank"
