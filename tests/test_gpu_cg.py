"""GPU suite (-m gpu): the D^-1-preconditioned CG bottom solver (the reference's solvers/cg.c, -DUSE_CG), bit for bit,
tolerance 0:
  - against the plain-C oracle (norms, error, order, iteration count; U and R of every level), with and without the
    single-block coarse-cycle kernel;
  - the stand-alone single-block kernels (CG and BiCGStab) against the algorithm written in Python over the library's own
    public operators;
  - the host-driven loop (periodic bottom with mean subtraction, multi-box bottom, the Helmholtz library) against the same;
  - switching solvers on one hierarchy, with and without recorded graphs, and the refusal of invalid values;
  - the other solve drivers with CG at the bottom;
  - several GPUs against one process with all the boxes."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

import hpgmg_b200.api as api
import oracle_bindings as ob
import oracle_cg as oc

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TOOL = os.path.join(ROOT, "tools", "check_cg.py")
U, F, R_ = api.VECTOR_U, api.VECTOR_F, api.VECTOR_R
SMOOTHERS = [api.SMOOTHER_GSRB, api.SMOOTHER_CHEBY]
SM_IDS = ["gsrb", "cheby"]
ORACLE_SMOOTHER = {api.SMOOTHER_GSRB: oc.GSRB, api.SMOOTHER_CHEBY: oc.CHEBY}
SOLVERS = [api.BOTTOM_CG, api.BOTTOM_BICGSTAB]
SOLVER_IDS = ["cg", "bicgstab"]


@pytest.fixture
def lib(gpu_lib):
    yield gpu_lib
    gpu_lib.hpgmg_b200_set_bottom_solver(api.BOTTOM_BICGSTAB)
    gpu_lib.hpgmg_b200_set_smoother(api.SMOOTHER_GSRB)
    gpu_lib.hpgmg_b200_use_graphs(1)
    gpu_lib.hpgmg_b200_use_coarse_kernel(1)


def interior(lvl, arr):
    n, g = lvl.contents.box_dim, lvl.contents.box_ghosts
    return arr[g:g + n, g:g + n, g:g + n]


def download(L, lvl, box, vid):
    out = np.empty(lvl.contents.box_volume, dtype=np.float64)
    L.hpgmg_download_box_vector(lvl, box, vid, out.ctypes.data_as(C.c_void_p))
    return api.box_view(lvl, out)


def upload(L, lvl, box, vid, a):
    L.hpgmg_upload_box_vector(lvl, box, vid, np.ascontiguousarray(a, dtype=np.float64).ctypes.data_as(C.c_void_p))


# ------------------------------------------------------------------- the algorithms over the public operators
def cg_restated(L, lvl, x, R, a, b, vr, dinv=api.VECTOR_DINV, rtol=1e-3):
    """solvers/cg.c written out over residual, mean, shift_vector, scale_vector, mul_vectors, dot, norm, apply_op and
    add_vectors: r0, r, p, Ap, z = vr+0..4."""
    r0, r, p, Ap, z = (vr + q for q in range(5))
    mean_shift = lvl.contents.must_subtract_mean == 1

    def subtract_mean(v):
        if mean_shift:
            L.shift_vector(lvl, v, v, -L.mean(lvl, v))
    L.residual(lvl, r0, x, R, a, b)
    subtract_mean(r0)
    L.scale_vector(lvl, r, 1.0, r0)
    L.mul_vectors(lvl, z, 1.0, dinv, r)
    L.scale_vector(lvl, p, 1.0, z)
    r_dot_z, norm_of_r0 = L.dot(lvl, r, z), L.norm(lvl, r)
    j, done = 0, (r_dot_z == 0.0 or norm_of_r0 == 0.0)
    while j < 200 and not done:
        j += 1
        L.apply_op(lvl, Ap, p, a, b)
        Ap_dot_p = L.dot(lvl, Ap, p)
        if Ap_dot_p == 0.0:
            break
        alpha = r_dot_z / Ap_dot_p
        if np.isinf(alpha):
            break
        L.add_vectors(lvl, x, 1.0, x, alpha, p)
        L.add_vectors(lvl, r, 1.0, r, -alpha, Ap)
        subtract_mean(r)
        norm_of_r = L.norm(lvl, r)
        if norm_of_r == 0.0 or norm_of_r < rtol * norm_of_r0:
            break
        L.mul_vectors(lvl, z, 1.0, dinv, r)
        r_dot_z_new = L.dot(lvl, r, z)
        if r_dot_z_new == 0.0:
            break
        beta = r_dot_z_new / r_dot_z
        if np.isinf(beta):
            break
        L.add_vectors(lvl, p, 1.0, z, beta, p)
        r_dot_z = r_dot_z_new
    return j


def bicgstab_restated(L, lvl, x, R, a, b, vr, dinv=api.VECTOR_DINV, rtol=1e-3):
    """solvers/bicgstab.c written out over the same operators: r0, r, p, q, s, t, Ap, As = vr+0..7."""
    r0, r, p, q, s, t, Ap, As = (vr + k for k in range(8))
    assert lvl.contents.must_subtract_mean != 1
    L.residual(lvl, r0, x, R, a, b)
    L.scale_vector(lvl, r, 1.0, r0)
    L.scale_vector(lvl, p, 1.0, r0)
    r_dot_r0, norm_of_r0 = L.dot(lvl, r, r0), L.norm(lvl, r)
    j, done = 0, (r_dot_r0 == 0.0 or norm_of_r0 == 0.0)
    while j < 200 and not done:
        j += 1
        L.mul_vectors(lvl, q, 1.0, dinv, p)
        L.apply_op(lvl, Ap, q, a, b)
        Ap_dot_r0 = L.dot(lvl, Ap, r0)
        if Ap_dot_r0 == 0.0:
            break
        alpha = r_dot_r0 / Ap_dot_r0
        if np.isinf(alpha):
            break
        L.add_vectors(lvl, x, 1.0, x, alpha, q)
        L.add_vectors(lvl, s, 1.0, r, -alpha, Ap)
        norm_of_s = L.norm(lvl, s)
        if norm_of_s == 0.0 or norm_of_s < rtol * norm_of_r0:
            break
        L.mul_vectors(lvl, t, 1.0, dinv, s)
        L.apply_op(lvl, As, t, a, b)
        As_dot_As, As_dot_s = L.dot(lvl, As, As), L.dot(lvl, As, s)
        if As_dot_As == 0.0:
            break
        omega = As_dot_s / As_dot_As
        if omega == 0.0 or np.isinf(omega):
            break
        L.add_vectors(lvl, x, 1.0, x, omega, t)
        L.add_vectors(lvl, r, 1.0, s, -omega, As)
        norm_of_r = L.norm(lvl, r)
        if norm_of_r == 0.0 or norm_of_r < rtol * norm_of_r0:
            break
        r_dot_r0_new = L.dot(lvl, r, r0)
        if r_dot_r0_new == 0.0:
            break
        beta = (r_dot_r0_new / r_dot_r0) * (alpha / omega)
        if np.isinf(beta):
            break
        L.add_vectors(lvl, api.VECTOR_TEMP, 1.0, p, -omega, Ap)
        L.add_vectors(lvl, p, 1.0, r, beta, api.VECTOR_TEMP)
        r_dot_r0 = r_dot_r0_new
    return j


def solver_vs_restatement(L, lvl, solver, seed, a=0.0, b=1.0, vr=api.VECTORS_RESERVED):
    """IterativeSolver on `lvl` from seeded random x (U) and R (ghosts included) against the restatement from the same start.
    Returns (iterations of the restatement, list of mismatches: empty if x and every solver vector are equal on every cell)."""
    nb = lvl.contents.num_my_boxes
    rng = np.random.default_rng(seed)
    shape = (lvl.contents.box_dim + 2 * lvl.contents.box_ghosts,) * 2 + (lvl.contents.box_jStride,)
    x0 = [rng.standard_normal(shape) for _ in range(nb)]
    f0 = [rng.standard_normal(shape) for _ in range(nb)]

    def start():
        for box in range(nb):
            upload(L, lvl, box, U, x0[box])
            upload(L, lvl, box, R_, f0[box])
    start()
    L.hpgmg_b200_set_bottom_solver(solver)
    L.IterativeSolver(lvl, U, R_, a, b, 1e-3)
    L.hpgmg_b200_sync()
    restate = cg_restated if solver == api.BOTTOM_CG else bicgstab_restated
    ids = [U] + list(range(vr, vr + (5 if solver == api.BOTTOM_CG else 8)))
    got = {(box, v): interior(lvl, download(L, lvl, box, v)).copy() for box in range(nb) for v in ids}
    start()
    its = restate(L, lvl, U, R_, a, b, vr)
    bad = []
    for (box, v), g in got.items():
        want = interior(lvl, download(L, lvl, box, v))
        if not np.array_equal(g, want):
            bad.append(f"box {box} vector {v}: {int(np.sum(g != want))} cells differ, max |diff| {np.max(np.abs(g - want)):.3e}")
    return its, bad


# ------------------------------------------------------------------------------------------- the oracle
@pytest.mark.parametrize("coarse", [1, 0], ids=["coarse_kernel", "multilaunch"])
@pytest.mark.parametrize("smoother", SMOOTHERS, ids=SM_IDS)
@pytest.mark.parametrize("log2", [4, 5, 6])
def test_richardson_and_fcycle_equal_oracle(lib, log2, smoother, coarse):
    O = oc.lib()
    lib.hpgmg_b200_use_coarse_kernel(coarse)
    norms_o, err_o, order_o, krylov_o = oc.richardson(log2, ORACLE_SMOOTHER[smoother])
    with api.Hierarchy(log2, 1, smoother=smoother, bottom_solver=api.BOTTOM_CG) as H:
        err, order, norms = H.richardson()
        assert [n[0] for n in norms] == norms_o
        assert err == err_o and order == order_o
        assert H.level(H.num_levels - 1).contents.Krylov_iterations == krylov_o
    # one F-cycle: every level cell by cell
    Ho = O.oracle_build(log2, ORACLE_SMOOTHER[smoother])
    r_o = O.oracle_cg_fmg_solve(Ho, 0, None)
    with api.Hierarchy(log2, 1, smoother=smoother, bottom_solver=api.BOTTOM_CG) as H:
        r, _ = H.fmg_solve(0)
        assert r == r_o
        for l in range(H.num_levels):
            n = H.level(l).contents.box_dim
            s = slice(2, 2 + n)
            for vid in (U, R_):
                np.testing.assert_array_equal(api.download(H.level(l), 0, vid)[s, s, s], oc.array(Ho, l, vid)[s, s, s], err_msg=f"level {l} vector {vid}")
    O.oracle_destroy(Ho)


# ------------------------------------------------------------- the single-block kernels against the operators
@pytest.mark.parametrize("solver", SOLVERS, ids=SOLVER_IDS)
@pytest.mark.parametrize("cfg", ["5 8", "4 27"])
def test_device_solver_equals_restatement(lib, cfg, solver):
    """`5 8`: a 2^3 bottom, `4 27`: 3^3; one box, Dirichlet: IterativeSolver runs the single-block kernel."""
    log2, boxes = map(int, cfg.split())
    with api.Hierarchy(log2, boxes, use_graphs=False) as H:
        lvl = H.level(H.num_levels - 1)
        assert lvl.contents.num_my_boxes == 1 and lvl.contents.box_dim == {"5 8": 2, "4 27": 3}[cfg]
        its, bad = solver_vs_restatement(lib, lvl, solver, ob.seed("device bottom", cfg, solver))
    assert not bad, bad[:8]
    assert 0 < its < 200


# ------------------------------------------------------------------------------------- the host-driven loop
def test_host_driven_cg_on_a_periodic_bottom(lib):
    """`4 8` periodic: the bottom subtracts the mean of r0 and r, so it runs the host-driven loop."""
    with api.Hierarchy(4, 8, bc=api.BC_PERIODIC, use_graphs=False) as H:
        lvl = H.level(H.num_levels - 1)
        its, bad = solver_vs_restatement(lib, lvl, api.BOTTOM_CG, ob.seed("periodic cg bottom"))
        assert lvl.contents.must_subtract_mean == 1
    assert not bad, bad[:8]
    assert 0 < its < 200


def test_host_driven_cg_on_a_multibox_bottom(lib):
    """MGBuild(minCoarseGridDim=16) on `4 8` stops at a 16^3 bottom level of 8 boxes."""
    H = api.Hierarchy(4, 8, build_operator=False, use_graphs=False)
    try:
        lib.initialize_problem(H.level_h, H.h, 0.0, 1.0)
        lib.rebuild_operator(H.level_h, None, 0.0, 1.0)
        lib.MGBuild(H.mg, H.level_h, 0.0, 1.0, 16)
        H.built = True
        lvl = H.level(H.num_levels - 1)
        assert lvl.contents.num_my_boxes == 8
        its, bad = solver_vs_restatement(lib, lvl, api.BOTTOM_CG, ob.seed("multibox cg bottom"))
    finally:
        H.close()
    assert not bad, bad[:8]
    assert 0 < its < 200


def test_host_driven_cg_in_the_helmholtz_library(lib):
    """libhpgmg_b200_helmholtz.so (VECTORS_RESERVED 11), a = b = 1: always the host-driven loop."""
    helm = api.bind(C.CDLL(os.path.join(os.path.dirname(api.LIB_PATH), "libhpgmg_b200_helmholtz.so")))
    assert helm.hpgmg_b200_init(0) == 0
    helm.hpgmg_b200_set_verbose(0)
    helm.hpgmg_b200_use_graphs(0)
    try:
        with api.Hierarchy(4, 8, library=helm, a=1.0, b=1.0, vectors=11) as H:
            lvl = H.level(H.num_levels - 1)
            its, bad = solver_vs_restatement(helm, lvl, api.BOTTOM_CG, ob.seed("helmholtz cg bottom"), a=1.0, b=1.0, vr=11)
        assert not bad, bad[:8]
        assert 0 < its < 200
    finally:
        helm.hpgmg_b200_set_bottom_solver(api.BOTTOM_BICGSTAB)
        helm.hpgmg_b200_use_graphs(1)


# ------------------------------------------------------------------------------- switching and selection
def level0_u(H):
    lvl = H.level(0)
    return [api.interior(lvl, api.download(lvl, b, U)).copy() for b in range(lvl.contents.num_my_boxes)]


def solve_snapshot(H):
    r, _ = H.fmg_solve(0)
    return r, level0_u(H)


@pytest.mark.parametrize("graphs", [False, True], ids=["stream", "graphs"])
def test_switching_bottom_solvers_on_one_hierarchy(lib, graphs):
    """BiCGStab -> CG -> BiCGStab on one built hierarchy, twice each (graphs: record, then replay): every solve equals the same
    solve on a hierarchy built with that solver selected, so a recording is never replayed for the other solver."""
    order = [api.BOTTOM_BICGSTAB, api.BOTTOM_CG, api.BOTTOM_BICGSTAB]
    fresh = {}
    for sv in SOLVERS:
        with api.Hierarchy(5, 8, bottom_solver=sv, use_graphs=graphs) as H:
            fresh[sv] = solve_snapshot(H)
    assert fresh[api.BOTTOM_CG][0] != fresh[api.BOTTOM_BICGSTAB][0], "the two solvers give different solves"
    with api.Hierarchy(5, 8, use_graphs=graphs) as H:
        for sv in order:
            lib.hpgmg_b200_set_bottom_solver(sv)
            for _ in range(2):
                r, u = solve_snapshot(H)
                assert r == fresh[sv][0], sv
                for a, b in zip(u, fresh[sv][1]):
                    np.testing.assert_array_equal(a, b)


def test_invalid_bottom_solver_is_refused(lib, capfd):
    for sv in SOLVERS:
        lib.hpgmg_b200_set_bottom_solver(sv)
        for bad in (-1, 2, 99):
            lib.hpgmg_b200_set_bottom_solver(bad)
            assert lib.hpgmg_b200_get_bottom_solver() == sv
    C.CDLL(None).fflush(None)
    assert "is not a bottom solver" in capfd.readouterr().err


# ----------------------------------------------------------------------------------------- other drivers
@pytest.mark.parametrize("driver", ["MGSolve", "FMGSolve2", "MGPCG"])
def test_other_drivers_with_cg(lib, driver):
    """MGSolve, FMGSolve2 and MGPCG on `5 8` with CG at the bottom reach rtol, and graphs on or off give the same bits."""
    rtol = 1e-10
    snaps = []
    for graphs in (True, False):
        with api.Hierarchy(5, 8, bottom_solver=api.BOTTOM_CG, use_graphs=graphs) as H:
            lib.zero_vector(H.level(0), U)
            getattr(lib, driver)(H.mg, 0, U, F, 0.0, 1.0, rtol)
            r, f = lib.hpgmg_last_norm_of_residual(H.mg), lib.hpgmg_last_norm_of_F(H.mg)
            assert r / f < rtol, (driver, graphs, r, f)
            assert H.level(H.num_levels - 1).contents.Krylov_iterations > 0
            snaps.append((r, level0_u(H)))
    assert snaps[0][0] == snaps[1][0]
    for a, b in zip(snaps[0][1], snaps[1][1]):
        np.testing.assert_array_equal(a, b)


# ----------------------------------------------------------------------------------------- several GPUs
def _gpu_count():
    try:
        return len([l for l in subprocess.run(["nvidia-smi", "-L"], capture_output=True, text=True).stdout.splitlines() if l.startswith("GPU ")])
    except Exception:
        return 0


def run(args, timeout=600):
    e = dict(os.environ)
    e.pop("RANK", None)
    e.pop("WORLD_SIZE", None)
    return subprocess.run([sys.executable] + args, capture_output=True, text=True, timeout=timeout, env=e)


@pytest.mark.parametrize("ranks", [2, 4])
def test_multi_gpu_cg_equals_single_process(lib, ranks, tmp_path):
    """CG `6 8` on N ranks: u of every box on every rank equals the single-process run with N x the boxes."""
    if _gpu_count() < ranks:
        pytest.skip(f"needs {ranks} GPUs")
    one, many = tmp_path / "one", tmp_path / "many"
    one.mkdir()
    many.mkdir()
    r = run([TOOL, "ranks", "6", str(8 * ranks), str(one)])
    assert r.stdout.startswith("OK"), r.stdout[-2000:] + r.stderr[-2000:]
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={ranks}", "--master-addr", "127.0.0.1",
                        "--master-port", str(29710 + ranks), TOOL, "ranks", "6", "8", str(many)], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    files = sorted(os.listdir(one))
    assert files and files == sorted(os.listdir(many))
    for f in files:
        np.testing.assert_array_equal(np.load(many / f), np.load(one / f), err_msg=f)
