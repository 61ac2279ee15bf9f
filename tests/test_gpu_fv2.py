"""GPU suite (-m gpu): the fv2 flavour, hpgmg_b200/lib/libhpgmg_b200_fv2.so -- the same sources compiled with -DHPGMG_FV2, the
counterpart of linking the reference with operators.fv2.c (7-point operator, one ghost layer, 4-sweep smoothers, V-cycle
interpolation p0, F-cycle interpolation v2).  Compared cell by cell, tolerance 0, with the plain-C restatement in
tests/oracle_fv2.c; the multi-box grids are compared across the library's own kernel paths."""
import ctypes as C
import os
import subprocess
import sys
import zlib

import numpy as np
import pytest

import hpgmg_b200.api as api
import oracle_fv2 as of

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
TOOL = os.path.join(os.path.dirname(HERE), "tools", "check_fv2.py")
U, F, E, Rr, T, DINV = api.VECTOR_U, api.VECTOR_F, api.VECTOR_E, api.VECTOR_R, api.VECTOR_TEMP, api.VECTOR_DINV
SMOOTHERS = {"gsrb": api.SMOOTHER_GSRB, "cheby": api.SMOOTHER_CHEBY, "jacobi": api.SMOOTHER_JACOBI, "l1jacobi": api.SMOOTHER_L1JACOBI}
BOTTOMS = {"bicgstab": api.BOTTOM_BICGSTAB, "cg": api.BOTTOM_CG}


@pytest.fixture(scope="module")
def fv2():
    L = api.bind(C.CDLL(api.FV2_LIB_PATH))
    assert L.hpgmg_b200_init(0) == 0
    assert L.stencil_get_radius() == 1 and L.stencil_get_shape() == api.STENCIL_SHAPE_STAR
    L.hpgmg_b200_set_verbose(0)
    yield L
    L.hpgmg_b200_set_smoother(api.SMOOTHER_GSRB)
    L.hpgmg_b200_set_bottom_solver(api.BOTTOM_BICGSTAB)
    L.hpgmg_b200_use_graphs(1)


def hierarchy(L, log2, boxes, smoother=api.SMOOTHER_GSRB, bottom=api.BOTTOM_BICGSTAB, graphs=1, **kw):
    L.hpgmg_b200_set_smoother(smoother)
    L.hpgmg_b200_set_bottom_solver(bottom)
    L.hpgmg_b200_use_graphs(graphs)
    return api.Hierarchy(log2, boxes, library=L, **kw)


def download(L, lvl, box, vid):
    out = np.empty(lvl.contents.box_volume, dtype=np.float64)
    L.hpgmg_download_box_vector(lvl, box, vid, out.ctypes.data_as(C.c_void_p))
    return api.interior(lvl, api.box_view(lvl, out)).copy()


def upload(L, lvl, box, vid, interior):
    a = np.zeros(lvl.contents.box_volume, dtype=np.float64)
    api.interior(lvl, api.box_view(lvl, a))[...] = interior
    L.hpgmg_upload_box_vector(lvl, box, vid, a.ctypes.data_as(C.c_void_p))


def rng_for(*key):
    return np.random.default_rng(zlib.crc32(repr(key).encode()))


# ----------------------------------------------------------------------------------------- against the oracle (one box per level)
@pytest.mark.parametrize("bottom", sorted(BOTTOMS))
@pytest.mark.parametrize("smoother", sorted(SMOOTHERS))
@pytest.mark.parametrize("log2", [5, 6])
def test_fmg_solve_equals_oracle(fv2, log2, smoother, bottom):
    """`hpgmg-fv <log2> 1`: the levels' D^-1 and eigenvalue bounds, the F-cycle residual norm and u equal the oracle's."""
    with of.Hier(log2, SMOOTHERS[smoother], BOTTOMS[bottom]) as O, hierarchy(fv2, log2, 1, SMOOTHERS[smoother], BOTTOMS[bottom]) as H:
        assert H.num_levels == O.num_levels() == log2 + 1
        for l in range(H.num_levels):
            assert H.level(l).contents.box_ghosts == 1
            assert H.level(l).contents.dominant_eigenvalue_of_DinvA == O.O.oracle_level_eig(O.H, l)
            np.testing.assert_array_equal(download(fv2, H.level(l), 0, DINV), O.interior(l, DINV), err_msg=f"D^-1 level {l}")
        want, _ = O.fmg_solve(0)
        r, _ = H.fmg_solve(0)
        assert r == want
        np.testing.assert_array_equal(download(fv2, H.level(0), 0, U), O.interior(0, U))


@pytest.mark.parametrize("op,smoother", [("apply_op", "gsrb"), ("residual", "gsrb"), ("interpolation_p0", "gsrb")] +
                         [("smooth", s) for s in sorted(SMOOTHERS)])
@pytest.mark.parametrize("log2", [5, 6])
def test_operator_equals_oracle(fv2, log2, smoother, op):
    """Each operator on its own, on random inputs, on every level it runs on (the smoother only matters to smooth())."""
    rng = rng_for("op", log2, smoother, op)
    with of.Hier(log2, SMOOTHERS[smoother]) as O, hierarchy(fv2, log2, 1, SMOOTHERS[smoother], graphs=0) as H:
        levels = range(H.num_levels - 1) if op == "interpolation_p0" else range(H.num_levels)
        for l in levels:
            n = H.level(l).contents.box_dim
            for vid in (U, F, E, Rr):
                a = rng.standard_normal((n, n, n))
                upload(fv2, H.level(l), 0, vid, a)
                g = of.G
                O.array(l, vid)[g:g + n, g:g + n, g:g + n] = a
            lv = H.level(l)
            if op == "apply_op":
                fv2.apply_op(lv, E, U, 0.0, 1.0); O.O.fv2_level_apply_op(O.F, l, E, U); checks = [(l, E)]
            elif op == "residual":
                fv2.residual(lv, E, U, F, 0.0, 1.0); O.O.fv2_level_residual(O.F, l, E, U, F); checks = [(l, E)]
            elif op == "smooth":
                fv2.smooth(lv, U, F, 0.0, 1.0); O.O.fv2_level_smooth(O.F, l, U, F); checks = [(l, U)]
            else:
                c = rng.standard_normal((n // 2,) * 3)
                upload(fv2, H.level(l + 1), 0, E, c)
                g = of.G
                O.array(l + 1, E)[g:g + n // 2, g:g + n // 2, g:g + n // 2] = c
                fv2.interpolation_p0(lv, U, 1.0, H.level(l + 1), E); O.O.fv2_level_interpolation_p0(O.F, l, U, 1.0, E); checks = [(l, U)]
            for ll, vid in checks:
                np.testing.assert_array_equal(download(fv2, H.level(ll), 0, vid), O.interior(ll, vid), err_msg=f"{op} level {ll}")


def chebyshev_coefficients(eig, degree=4):
    beta = 1.000 * eig
    alpha = 0.125000 * beta
    theta, delta = 0.5 * (beta + alpha), 0.5 * (beta - alpha)
    sigma = theta / delta
    rho = 1 / sigma
    c1, c2 = [0.0], [1 / theta]
    for _ in range(1, degree):
        rho_nm1 = rho
        rho = 1.0 / (2.0 * sigma - rho_nm1)
        c1.append(rho * rho_nm1)
        c2.append(rho * 2.0 / delta)
    return c1, c2


@pytest.mark.parametrize("smoother", ["gsrb", "cheby", "jacobi"])
@pytest.mark.parametrize("cfg", ["6 1", "4 8"])
def test_smooth_is_four_sweeps_of_apply_op(fv2, cfg, smoother):
    """One smooth() equals its 4 sweeps x -> TEMP -> x composed in numpy from the library's apply_op (the k-marching kernel on
    the 64^3 box of `6 1`, the pair kernel on the 16^3 boxes of `4 8`)."""
    log2, boxes = map(int, cfg.split())
    rng = rng_for("sweeps", cfg, smoother)
    with hierarchy(fv2, log2, boxes, SMOOTHERS[smoother], graphs=0) as H:
        lv = H.level(0)
        nb, n = lv.contents.num_my_boxes, lv.contents.box_dim
        x = [rng.standard_normal((n, n, n)) for _ in range(nb)]
        rhs = [rng.standard_normal((n, n, n)) for _ in range(nb)]
        for b in range(nb):
            upload(fv2, lv, b, U, x[b])
            upload(fv2, lv, b, F, rhs[b])
        dinv = [download(fv2, lv, b, DINV) for b in range(nb)]
        c1, c2 = chebyshev_coefficients(lv.contents.dominant_eigenvalue_of_DinvA)
        k, j, i = np.meshgrid(np.arange(n), np.arange(n), np.arange(n), indexing="ij")
        lows = [(lv.contents.my_boxes[b].low.i, lv.contents.my_boxes[b].low.j, lv.contents.my_boxes[b].low.k) for b in range(nb)]
        cur, prev = [a.copy() for a in x], [np.zeros_like(a) for a in x]
        for s in range(4):
            for b in range(nb):
                upload(fv2, lv, b, E, cur[b])
            fv2.apply_op(lv, Rr, E, 0.0, 1.0)
            nxt = []
            for b in range(nb):
                Ax = download(fv2, lv, b, Rr)
                if smoother == "gsrb":
                    par = (lows[b][0] ^ lows[b][1] ^ lows[b][2] ^ s) & 1
                    upd = cur[b] + dinv[b] * (rhs[b] - Ax)
                    nxt.append(np.where(((i ^ j ^ k ^ par) & 1) == 0, upd, cur[b]))
                elif smoother == "cheby":
                    nxt.append(cur[b] + c1[s] * (cur[b] - prev[b]) + c2[s] * dinv[b] * (rhs[b] - Ax))
                else:
                    nxt.append(cur[b] + ((2.0 / 3.0) * dinv[b]) * (rhs[b] - Ax))
            prev, cur = cur, nxt
        fv2.smooth(lv, U, F, 0.0, 1.0)
        for b in range(nb):
            np.testing.assert_array_equal(download(fv2, lv, b, U), cur[b], err_msg=f"box {b}")


def test_layout_and_bottom_solve_is_one_kernel(fv2):
    """`7 8` has one ghost layer on every level, levels 256^3 .. 2^3, 1^3, and its 1^3 bottom is solved by the single-block
    kernel (one launch), so that FMGSolve can be recorded into a graph."""
    with hierarchy(fv2, 7, 8) as H:
        dims = [H.level(l).contents.dim.i for l in range(H.num_levels)]
        assert dims == [256 >> l for l in range(9)]
        assert all(H.level(l).contents.box_ghosts == 1 for l in range(H.num_levels))
        lb = H.level(H.num_levels - 1)
        for bottom in BOTTOMS.values():
            fv2.hpgmg_b200_set_bottom_solver(bottom)
            k0 = fv2.hpgmg_b200_kernel_launches()
            fv2.IterativeSolver(lb, E, Rr, 0.0, 1.0, 1e-3)
            fv2.hpgmg_b200_sync()
            assert fv2.hpgmg_b200_kernel_launches() - k0 == 1
        fv2.hpgmg_b200_set_bottom_solver(api.BOTTOM_BICGSTAB)


# ----------------------------------------------------------------------------------------- kernel paths (processes of their own)
def run(args, env=None, timeout=900):
    e = dict(os.environ)
    for k in list(e):
        if k.startswith("HPGMG_B200_") or k in ("RANK", "WORLD_SIZE", "LOCAL_RANK"):
            e.pop(k)
    e.update(env or {})
    return subprocess.run([sys.executable] + args, capture_output=True, text=True, timeout=timeout, env=e)


def solve(tmp_path, name, cfg, smoother=0, graphs=1, periodic=0, env=None):
    d = tmp_path / name
    d.mkdir()
    log2, boxes = cfg.split()
    r = run([TOOL, "solve", log2, boxes, str(smoother), str(graphs), str(periodic), str(d)], env)
    assert r.stdout.startswith("OK"), r.stdout[-2000:] + r.stderr[-2000:]
    w = r.stdout.split()
    return d, (float(w[w.index("norms") + 1]), float(w[w.index("norms") + 2])), (int(w[w.index("launches") + 1]), int(w[w.index("launches") + 2]))


def same_u(a, b):
    files = sorted(os.listdir(a))
    assert files and files == sorted(os.listdir(b))
    for f in files:
        np.testing.assert_array_equal(np.load(b / f), np.load(a / f), err_msg=f)


VARIANTS = {"default": ({}, 1), "tma-off": ({"HPGMG_B200_TMA": "0"}, 1), "graphs-off": ({}, 0),
            "pair-off": ({"HPGMG_B200_PAIR_KERNEL": "0"}, 1)}


@pytest.mark.parametrize("smoother", ["gsrb", "cheby"])
@pytest.mark.parametrize("cfg", ["6 8", "7 8"])
def test_kernel_paths_give_the_same_bits(tmp_path, cfg, smoother):
    """Every kernel path equals the generic one-thread-per-cell kernel on every level: the k-marching kernel (boxes >= 32^3),
    the pair kernel, graphs on and off."""
    sm = SMOOTHERS[smoother]
    ref, ref_norms, _ = solve(tmp_path, "generic", cfg, sm, env={"HPGMG_B200_GENERIC_STENCIL": "1"})
    for name, (env, graphs) in VARIANTS.items():
        d, norms, _ = solve(tmp_path, name, cfg, sm, graphs=graphs, env=env)
        assert norms == ref_norms, name
        same_u(ref, d)


def test_periodic_problem(tmp_path):
    """A periodic `6 8` (mean subtraction, no boundary conditions, host-driven bottom solve): the k-marching kernel gives the
    generic kernel's bits."""
    ref, ref_norms, _ = solve(tmp_path, "generic", "6 8", periodic=1, env={"HPGMG_B200_GENERIC_STENCIL": "1"})
    d, norms, _ = solve(tmp_path, "default", "6 8", periodic=1)
    assert norms == ref_norms and np.isfinite(norms[0]) and norms[0] > 0
    same_u(ref, d)


def test_second_fmg_solve_is_a_graph_replay(tmp_path):
    """`7 8`: the second FMGSolve replays the recorded graph -- the same kernel launches as the first, the same result."""
    _, norms, launches = solve(tmp_path, "graphs", "7 8")
    assert launches[0] == launches[1] > 0
    assert norms[0] == norms[1]


def _gpu_count():
    try:
        return len([l for l in subprocess.run(["nvidia-smi", "-L"], capture_output=True, text=True).stdout.splitlines() if l.startswith("GPU ")])
    except Exception:
        return 0


def test_two_gpus_equal_one_process(tmp_path):
    """`6 8` on 2 ranks: u of every box equals the single-process run with 16 boxes."""
    if _gpu_count() < 2:
        pytest.skip("needs 2 GPUs")
    one, _, _ = solve(tmp_path, "one", "6 16")
    many = tmp_path / "many"
    many.mkdir()
    e = {k: v for k, v in os.environ.items() if not k.startswith("HPGMG_B200_")}
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
                        "--master-port", "29742", TOOL, "solve", "6", "8", "0", "1", "0", str(many)], capture_output=True, text=True, timeout=900, env=e)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    same_u(one, many)
