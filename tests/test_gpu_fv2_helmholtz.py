"""GPU suite (-m gpu): the fv2 Helmholtz flavour, hpgmg_b200/lib/libhpgmg_b200_fv2_helmholtz.so -- the same sources compiled
with -DHPGMG_FV2 -DUSE_HELMHOLTZ, the counterpart of the reference's operators.fv2.c built with -DUSE_HELMHOLTZ
(a*alpha*u - b*div(beta grad u), the Helmholtz vector map, a = b = 1 as hpgmg-fv.c:286-288).  Compared cell by cell,
tolerance 0, with the plain-C restatement in tests/oracle_fv2_helmholtz.c; the single-block bottom solvers with their
algorithms written over the library's public operators; the multi-box grids across the library's own kernel paths."""
import ctypes as C
import os
import subprocess
import sys
import zlib

import numpy as np
import pytest

import hpgmg_b200.api as api
import oracle_bindings as ob
import oracle_fv2_helmholtz as oh
from test_gpu_cg import solver_vs_restatement
from test_gpu_fv2 import chebyshev_coefficients, download, same_u, upload

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
TOOL = os.path.join(os.path.dirname(HERE), "tools", "check_fv2.py")
U, F, E, Rr, T, DINV = api.VECTOR_U, api.VECTOR_F, api.VECTOR_E, api.VECTOR_R, api.VECTOR_TEMP, api.VECTOR_DINV
ALPHA, L1INV, NVEC = 9, 10, 11                      # the Helmholtz vector map (include/hpgmg_defines.h)
A_, B_ = oh.A, oh.B
SMOOTHERS = {"gsrb": api.SMOOTHER_GSRB, "cheby": api.SMOOTHER_CHEBY, "jacobi": api.SMOOTHER_JACOBI, "l1jacobi": api.SMOOTHER_L1JACOBI}
BOTTOMS = {"bicgstab": api.BOTTOM_BICGSTAB, "cg": api.BOTTOM_CG}


@pytest.fixture(scope="module")
def fvh():
    L = api.bind(C.CDLL(api.FV2_HELMHOLTZ_LIB_PATH))
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
    return api.Hierarchy(log2, boxes, library=L, a=A_, b=B_, vectors=NVEC, **kw)


def rng_for(*key):
    return np.random.default_rng(zlib.crc32(repr(key).encode()))


# ----------------------------------------------------------------------------------------- against the oracle (one box per level)
@pytest.mark.parametrize("bottom", sorted(BOTTOMS))
@pytest.mark.parametrize("smoother", sorted(SMOOTHERS))
@pytest.mark.parametrize("log2", [5, 6])
def test_fmg_solve_equals_oracle(fvh, log2, smoother, bottom):
    """`hpgmg-fv <log2> 1`: every level's alpha, D^-1, L1 row inverse and eigenvalue bound, the F-cycle residual norm and u equal
    the oracle's."""
    with oh.Hier(log2, SMOOTHERS[smoother], BOTTOMS[bottom]) as O, hierarchy(fvh, log2, 1, SMOOTHERS[smoother], BOTTOMS[bottom]) as H:
        assert H.num_levels == O.num_levels() == log2 + 1
        for l in range(H.num_levels):
            assert H.level(l).contents.box_ghosts == 1
            assert H.level(l).contents.dominant_eigenvalue_of_DinvA == O.eig(l)
            for vid, ovid in ((ALPHA, O.ALPHA), (DINV, DINV), (L1INV, O.L1)):
                np.testing.assert_array_equal(download(fvh, H.level(l), 0, vid), O.interior(l, ovid), err_msg=f"vector {vid} level {l}")
        want, _ = O.fmg_solve(0)
        r, _ = H.fmg_solve(0)
        assert r == want
        np.testing.assert_array_equal(download(fvh, H.level(0), 0, U), O.interior(0, U))


@pytest.mark.parametrize("op,smoother", [("apply_op", "gsrb"), ("residual", "gsrb")] + [("smooth", s) for s in sorted(SMOOTHERS)])
@pytest.mark.parametrize("log2", [5, 6])
def test_operator_equals_oracle(fvh, log2, smoother, op):
    """Each operator on its own, on random inputs, on every level (the smoother only matters to smooth())."""
    rng = rng_for("fvh op", log2, smoother, op)
    with oh.Hier(log2, SMOOTHERS[smoother]) as O, hierarchy(fvh, log2, 1, SMOOTHERS[smoother], graphs=0) as H:
        for l in range(H.num_levels):
            n = H.level(l).contents.box_dim
            for vid in (U, F, E, Rr):
                a = rng.standard_normal((n, n, n))
                upload(fvh, H.level(l), 0, vid, a)
                O.array(l, vid)[oh.G:oh.G + n, oh.G:oh.G + n, oh.G:oh.G + n] = a
            lv = H.level(l)
            if op == "apply_op":
                fvh.apply_op(lv, E, U, A_, B_); O.O.fvh_level_apply_op(O.F, l, E, U); vid = E
            elif op == "residual":
                fvh.residual(lv, E, U, F, A_, B_); O.O.fvh_level_residual(O.F, l, E, U, F); vid = E
            else:
                fvh.smooth(lv, U, F, A_, B_); O.O.fvh_level_smooth(O.F, l, U, F); vid = U
            np.testing.assert_array_equal(download(fvh, lv, 0, vid), O.interior(l, vid), err_msg=f"{op} level {l}")


@pytest.mark.parametrize("smoother", sorted(SMOOTHERS))
@pytest.mark.parametrize("cfg", ["6 1", "4 8"])
def test_smooth_is_four_sweeps_of_apply_op(fvh, cfg, smoother):
    """One smooth() equals its 4 sweeps x -> TEMP -> x composed in numpy from the library's apply_op with a = b = 1 (the
    k-marching kernel on the 64^3 box of `6 1`, the pair kernel on the 16^3 boxes of `4 8`)."""
    log2, boxes = map(int, cfg.split())
    rng = rng_for("fvh sweeps", cfg, smoother)
    with hierarchy(fvh, log2, boxes, SMOOTHERS[smoother], graphs=0) as H:
        lv = H.level(0)
        nb, n = lv.contents.num_my_boxes, lv.contents.box_dim
        x = [rng.standard_normal((n, n, n)) for _ in range(nb)]
        rhs = [rng.standard_normal((n, n, n)) for _ in range(nb)]
        for b in range(nb):
            upload(fvh, lv, b, U, x[b])
            upload(fvh, lv, b, F, rhs[b])
        dinv = [download(fvh, lv, b, DINV) for b in range(nb)]
        l1 = [download(fvh, lv, b, L1INV) for b in range(nb)]
        c1, c2 = chebyshev_coefficients(lv.contents.dominant_eigenvalue_of_DinvA)
        k, j, i = np.meshgrid(np.arange(n), np.arange(n), np.arange(n), indexing="ij")
        lows = [(lv.contents.my_boxes[b].low.i, lv.contents.my_boxes[b].low.j, lv.contents.my_boxes[b].low.k) for b in range(nb)]
        cur, prev = [a.copy() for a in x], [np.zeros_like(a) for a in x]
        for s in range(4):
            for b in range(nb):
                upload(fvh, lv, b, E, cur[b])
            fvh.apply_op(lv, Rr, E, A_, B_)
            nxt = []
            for b in range(nb):
                Ax = download(fvh, lv, b, Rr)
                if smoother == "gsrb":
                    par = (lows[b][0] ^ lows[b][1] ^ lows[b][2] ^ s) & 1
                    upd = cur[b] + dinv[b] * (rhs[b] - Ax)
                    nxt.append(np.where(((i ^ j ^ k ^ par) & 1) == 0, upd, cur[b]))
                elif smoother == "cheby":
                    nxt.append(cur[b] + c1[s] * (cur[b] - prev[b]) + c2[s] * dinv[b] * (rhs[b] - Ax))
                elif smoother == "jacobi":
                    nxt.append(cur[b] + ((2.0 / 3.0) * dinv[b]) * (rhs[b] - Ax))
                else:
                    nxt.append(cur[b] + (1.0 * l1[b]) * (rhs[b] - Ax))
            prev, cur = cur, nxt
        fvh.smooth(lv, U, F, A_, B_)
        for b in range(nb):
            np.testing.assert_array_equal(download(fvh, lv, b, U), cur[b], err_msg=f"box {b}")


# ----------------------------------------------------------------------------------------- the single-block bottom solvers
@pytest.mark.parametrize("solver", sorted(BOTTOMS))
def test_device_solver_equals_restatement(fvh, solver):
    """The 3^3 bottom of `4 27` (one box, Dirichlet): the single-block kernel of each solver equals its algorithm written in
    Python over the library's public operators, a = b = 1."""
    with hierarchy(fvh, 4, 27, graphs=0) as H:
        lvl = H.level(H.num_levels - 1)
        assert lvl.contents.num_my_boxes == 1 and lvl.contents.box_dim == 3
        k0 = fvh.hpgmg_b200_kernel_launches()
        fvh.hpgmg_b200_set_bottom_solver(BOTTOMS[solver])
        fvh.IterativeSolver(lvl, E, Rr, A_, B_, 1e-3)
        fvh.hpgmg_b200_sync()
        assert fvh.hpgmg_b200_kernel_launches() - k0 == 1
        its, bad = solver_vs_restatement(fvh, lvl, BOTTOMS[solver], ob.seed("fv2 helmholtz device bottom", solver), a=A_, b=B_, vr=NVEC)
    assert not bad, bad[:8]
    assert 0 < its < 200


def test_layout_and_bottom_solve_is_one_kernel(fvh):
    """`7 8`: one ghost layer on every level, levels 256^3 .. 1^3, and the 1^3 bottom is solved by one single-block launch for
    each solver, so that FMGSolve can be recorded into a graph."""
    with hierarchy(fvh, 7, 8) as H:
        assert [H.level(l).contents.dim.i for l in range(H.num_levels)] == [256 >> l for l in range(9)]
        assert all(H.level(l).contents.box_ghosts == 1 for l in range(H.num_levels))
        lb = H.level(H.num_levels - 1)
        for bottom in BOTTOMS.values():
            fvh.hpgmg_b200_set_bottom_solver(bottom)
            k0 = fvh.hpgmg_b200_kernel_launches()
            fvh.IterativeSolver(lb, E, Rr, A_, B_, 1e-3)
            fvh.hpgmg_b200_sync()
            assert fvh.hpgmg_b200_kernel_launches() - k0 == 1
        fvh.hpgmg_b200_set_bottom_solver(api.BOTTOM_BICGSTAB)


# ----------------------------------------------------------------------------------------- kernel paths (processes of their own)
def run(args, env=None, timeout=900):
    e = dict(os.environ)
    for k in list(e):
        if k.startswith("HPGMG_B200_") or k in ("RANK", "WORLD_SIZE", "LOCAL_RANK"):
            e.pop(k)
    e.update(env or {})
    return subprocess.run([sys.executable] + args, capture_output=True, text=True, timeout=timeout, env=e)


def solve(tmp_path, name, cfg, smoother=0, graphs=1, periodic=0, env=None):
    """check_fv2.py on the fv2 Helmholtz library: (u directory, the two solves' norms, their launches, must_subtract_mean)"""
    d = tmp_path / name
    d.mkdir()
    log2, boxes = cfg.split()
    r = run([TOOL, "solve", log2, boxes, str(smoother), str(graphs), str(periodic), str(d), "fv2_helmholtz"], env)
    assert r.stdout.startswith("OK"), r.stdout[-2000:] + r.stderr[-2000:]
    w = r.stdout.split()
    at = w.index
    return (d, (float(w[at("norms") + 1]), float(w[at("norms") + 2])), (int(w[at("launches") + 1]), int(w[at("launches") + 2])),
            int(w[at("must_subtract_mean") + 1]))


VARIANTS = {"default": ({}, 1), "tma-off": ({"HPGMG_B200_TMA": "0"}, 1), "graphs-off": ({}, 0),
            "pair-off": ({"HPGMG_B200_PAIR_KERNEL": "0"}, 1)}


@pytest.mark.parametrize("smoother", ["gsrb", "cheby"])
@pytest.mark.parametrize("cfg", ["6 8", "7 8"])
def test_kernel_paths_give_the_same_bits(tmp_path, cfg, smoother):
    """Every kernel path equals the generic one-thread-per-cell kernel on every level: the k-marching kernel (boxes >= 32^3),
    the pair kernel, graphs on and off."""
    sm = SMOOTHERS[smoother]
    ref, ref_norms, _, _ = solve(tmp_path, "generic", cfg, sm, env={"HPGMG_B200_GENERIC_STENCIL": "1"})
    for name, (env, graphs) in VARIANTS.items():
        d, norms, _, _ = solve(tmp_path, name, cfg, sm, graphs=graphs, env=env)
        assert norms == ref_norms, name
        same_u(ref, d)


def test_periodic_problem(tmp_path):
    """A periodic `6 8` with a*alpha != 0: the solution is unique, so no mean is subtracted (mg.c); the bottom stays host-driven,
    and the k-marching kernel gives the generic kernel's bits."""
    ref, ref_norms, _, msm_ref = solve(tmp_path, "generic", "6 8", periodic=1, env={"HPGMG_B200_GENERIC_STENCIL": "1"})
    d, norms, _, msm = solve(tmp_path, "default", "6 8", periodic=1)
    assert msm == msm_ref == 0
    assert norms == ref_norms and np.isfinite(norms[0]) and norms[0] > 0
    same_u(ref, d)


def test_second_fmg_solve_is_a_graph_replay(tmp_path):
    """`7 8`: the second FMGSolve replays the recorded graph -- the same kernel launches as the first, the same result."""
    _, norms, launches, _ = solve(tmp_path, "graphs", "7 8")
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
    one, _, _, _ = solve(tmp_path, "one", "6 16")
    many = tmp_path / "many"
    many.mkdir()
    e = {k: v for k, v in os.environ.items() if not k.startswith("HPGMG_B200_")}
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
                        "--master-port", "29743", TOOL, "solve", "6", "8", "0", "1", "0", str(many), "fv2_helmholtz"],
                       capture_output=True, text=True, timeout=900, env=e)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    same_u(one, many)
