"""GPU suite (-m gpu): the weighted Jacobi and L1-Jacobi smoothers (the reference's operators/jacobi.c, -DUSE_JACOBI /
-DUSE_L1JACOBI), bit for bit, tolerance 0:
  - against the plain-C oracle (norms, error, order, Krylov count; U, R, Dinv and the L1 row inverse of every level);
  - one smooth() against six sweeps composed from apply_op (already verified) and the update in numpy, on every kernel path:
    the k-marching TMA kernel (32^3 .. 128^3 boxes), the fill-fused box kernel (4^3 .. 16^3) and, with the switches, the pair
    and generic kernels;
  - the single-block coarse-cycle kernel against one launch per operator;
  - the Helmholtz library (lambda from VECTOR_L1INV);
  - switching smoothers on one hierarchy, with and without recorded graphs, and the errors of a late or invalid selection;
  - several GPUs against one process with all the boxes."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

import hpgmg_b200.api as api
import oracle_bindings as ob
import oracle_jacobi as oj

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TOOL = os.path.join(ROOT, "tools", "check_jacobi.py")
sys.path.insert(0, os.path.join(ROOT, "tools"))
import check_jacobi as cj  # noqa: E402

NEW = [api.SMOOTHER_JACOBI, api.SMOOTHER_L1JACOBI]
IDS = ["jacobi", "l1jacobi"]
NAME = {api.SMOOTHER_JACOBI: "jacobi", api.SMOOTHER_L1JACOBI: "l1jacobi"}
ORACLE_INDEX = {api.SMOOTHER_JACOBI: oj.JACOBI, api.SMOOTHER_L1JACOBI: oj.L1JACOBI}      # oracle_jacobi_build's smoother index


@pytest.fixture
def lib(gpu_lib):
    yield gpu_lib
    gpu_lib.hpgmg_b200_set_smoother(api.SMOOTHER_GSRB)
    gpu_lib.hpgmg_b200_use_graphs(1)
    gpu_lib.hpgmg_b200_use_coarse_kernel(1)


def run(args, env=None, timeout=600):
    e = dict(os.environ)
    e.update(env or {})
    e.pop("RANK", None)
    e.pop("WORLD_SIZE", None)
    return subprocess.run([sys.executable] + args, capture_output=True, text=True, timeout=timeout, env=e)


# ------------------------------------------------------------------------------------------- the oracle
@pytest.mark.parametrize("smoother", NEW, ids=IDS)
@pytest.mark.parametrize("log2", [4, 5, 6])
def test_richardson_and_fcycle_equal_oracle(lib, log2, smoother):
    O = oj.lib()
    norms_o, err_o, order_o, krylov_o = oj.richardson(log2, ORACLE_INDEX[smoother])
    with api.Hierarchy(log2, 1, smoother=smoother) as H:
        err, order, norms = H.richardson()
        assert [n[0] for n in norms] == norms_o
        assert err == err_o and order == order_o
        assert H.level(H.num_levels - 1).contents.Krylov_iterations == krylov_o
    # one F-cycle: every level cell by cell
    Ho = O.oracle_jacobi_build(log2, ORACLE_INDEX[smoother])
    r_o = O.oracle_jacobi_fmg_solve(Ho, 0, None)
    with api.Hierarchy(log2, 1, smoother=smoother) as H:
        r, _ = H.fmg_solve(0)
        assert r == r_o
        for l in range(H.num_levels):
            n = H.level(l).contents.box_dim
            s = slice(2, 2 + n)
            for vid in (api.VECTOR_U, api.VECTOR_R, api.VECTOR_DINV):
                np.testing.assert_array_equal(api.download(H.level(l), 0, vid)[s, s, s], oj.array(Ho, l, vid)[s, s, s], err_msg=f"level {l} vector {vid}")
            if smoother == api.SMOOTHER_L1JACOBI:
                np.testing.assert_array_equal(cj.l1inv(lib, H.level(l), 0)[s, s, s], oj.l1inv(Ho, l)[s, s, s], err_msg=f"level {l} L1 inverse")
    O.oracle_destroy(Ho)


# --------------------------------------------------------------- one smooth() against composed operators
@pytest.mark.parametrize("smoother", NEW, ids=IDS)
@pytest.mark.parametrize("cfg", ["4 8", "4 27", "5 8", "6 8", "7 8"])
def test_smooth_equals_composed_sweeps(lib, cfg, smoother):
    """4 8 / 4 27: 16^3 boxes (fill-fused box kernel); 5 8, 6 8, 7 8: 32^3 .. 128^3 boxes (TMA kernel) and the coarser levels."""
    log2, boxes = map(int, cfg.split())
    with api.Hierarchy(log2, boxes, smoother=smoother, use_graphs=False) as H:
        bad = cj.smooth_vs_composition(lib, H, smoother, seed=ob.seed("jacobi compose", cfg, smoother))
    assert not bad, bad[:8]


FALLBACKS = {"HPGMG_B200_GENERIC_STENCIL": "1", "HPGMG_B200_TMA": "0", "HPGMG_B200_PAIR_KERNEL": "0", "HPGMG_B200_BOX_FUSED_MAX": "0"}


@pytest.mark.parametrize("smoother", NEW, ids=IDS)
@pytest.mark.parametrize("switch", sorted(FALLBACKS))
def test_smooth_on_fallback_kernels(lib, switch, smoother):
    """The same check through the generic, pair and separate-fill paths (each switch in a process of its own)."""
    for cfg in ("4 8", "6 8"):
        r = run([TOOL, "compose", *cfg.split(), NAME[smoother]], env={switch: FALLBACKS[switch]})
        assert r.stdout.startswith("OK"), r.stdout[-2000:] + r.stderr[-2000:]


# ---------------------------------------------------------------------------------- coarse-cycle kernel
@pytest.mark.parametrize("smoother", NEW, ids=IDS)
@pytest.mark.parametrize("cfg", ["5 8", "4 27"])
def test_coarse_kernel_equals_multilaunch_path(lib, cfg, smoother):
    log2, boxes = map(int, cfg.split())
    snap = {}
    for coarse in (0, 1):
        lib.hpgmg_b200_use_coarse_kernel(coarse)
        with api.Hierarchy(log2, boxes, smoother=smoother, use_graphs=False) as H:
            launches0 = lib.hpgmg_b200_kernel_launches()
            r = H.fmg_solve(0)
            launches = lib.hpgmg_b200_kernel_launches() - launches0
            arrays = [api.download(H.level(l), b, v).copy() for l in range(H.num_levels)
                      for b in range(H.level(l).contents.num_my_boxes) for v in (api.VECTOR_U, api.VECTOR_R)]
            snap[coarse] = (r, arrays, H.level(H.num_levels - 1).contents.Krylov_iterations, launches)
    assert snap[0][0] == snap[1][0] and snap[0][2] == snap[1][2]
    for a, b in zip(snap[0][1], snap[1][1]):
        n = a.shape[0] - 4
        s = slice(2, 2 + n)
        np.testing.assert_array_equal(a[s, s, s], b[s, s, s])
    assert snap[1][3] < snap[0][3], "the coarse kernel must remove launches"


# ------------------------------------------------------------------------------------- Helmholtz library
@pytest.mark.parametrize("smoother", NEW, ids=IDS)
def test_helmholtz_smooth_equals_composed_sweeps(lib, smoother):
    helm = api.bind(C.CDLL(os.path.join(os.path.dirname(api.LIB_PATH), "libhpgmg_b200_helmholtz.so")))
    assert helm.hpgmg_b200_init(0) == 0
    helm.hpgmg_b200_set_verbose(0)
    helm.hpgmg_b200_use_graphs(0)
    helm.hpgmg_b200_set_smoother(smoother)
    try:
        with api.Hierarchy(4, 8, library=helm, a=1.0, b=1.0, vectors=11) as H:
            lvl = H.level(0)
            for b in range(lvl.contents.num_my_boxes):              # in this build the L1 inverse is VECTOR_L1INV (id 10)
                np.testing.assert_array_equal(cj.l1inv(helm, lvl, b), cj.download(helm, lvl, b, 10))
            bad = cj.smooth_vs_composition(helm, H, smoother, seed=ob.seed("jacobi helmholtz", smoother), a=1.0, b=1.0)
        assert not bad, bad[:8]
    finally:
        helm.hpgmg_b200_set_smoother(api.SMOOTHER_GSRB)
        helm.hpgmg_b200_use_graphs(1)


# ------------------------------------------------------------------------------- switching and selection
def solve_snapshot(H):
    r, _ = H.fmg_solve(0)
    lvl = H.level(0)
    return r, [api.interior(lvl, api.download(lvl, b, api.VECTOR_U)).copy() for b in range(lvl.contents.num_my_boxes)]


@pytest.mark.parametrize("graphs", [False, True], ids=["stream", "graphs"])
def test_switching_smoothers_on_one_hierarchy(lib, graphs):
    """A hierarchy built with L1-Jacobi selected (its levels have the L1 inverse) solves with GSRB, Jacobi, L1-Jacobi and GSRB
    again; every solve equals the same solve on a hierarchy built for that smoother, so a recording is never replayed for
    another smoother."""
    order = [api.SMOOTHER_GSRB, api.SMOOTHER_JACOBI, api.SMOOTHER_L1JACOBI, api.SMOOTHER_GSRB]
    fresh = {}
    for sm in set(order):
        with api.Hierarchy(5, 8, smoother=sm, use_graphs=graphs) as H:
            fresh[sm] = solve_snapshot(H)
    assert len({fresh[sm][0] for sm in fresh}) == 3, "the three smoothers give three different solves"
    with api.Hierarchy(5, 8, smoother=api.SMOOTHER_L1JACOBI, use_graphs=graphs) as H:
        for sm in order:
            lib.hpgmg_b200_set_smoother(sm)
            for _ in range(2):                                   # graphs: record, then replay
                r, u = solve_snapshot(H)
                assert r == fresh[sm][0], NAME.get(sm, sm)
                for a, b in zip(u, fresh[sm][1]):
                    np.testing.assert_array_equal(a, b)


def test_l1jacobi_selected_after_the_build_stops(lib):
    r = run([TOOL, "late"], timeout=300)
    assert r.returncode != 0, r.stdout[-2000:]
    assert "no L1 row inverse" in r.stderr and "before rebuild_operator / MGBuild" in r.stderr, r.stderr[-2000:]
    assert "FAIL" not in r.stdout


def test_invalid_smoother_is_refused(lib, capfd):
    for sm in (api.SMOOTHER_CHEBY, api.SMOOTHER_L1JACOBI):
        lib.hpgmg_b200_set_smoother(sm)
        for bad in (-1, 4, 99):
            lib.hpgmg_b200_set_smoother(bad)
            assert lib.hpgmg_b200_get_smoother() == sm
    C.CDLL(None).fflush(None)
    assert "is not a smoother" in capfd.readouterr().err


# ----------------------------------------------------------------------------------------- several GPUs
def _gpu_count():
    try:
        return len([l for l in subprocess.run(["nvidia-smi", "-L"], capture_output=True, text=True).stdout.splitlines() if l.startswith("GPU ")])
    except Exception:
        return 0


@pytest.mark.parametrize("ranks", [2, 4])
def test_multi_gpu_jacobi_equals_single_process(lib, ranks, tmp_path):
    """Jacobi `6 8` on N ranks: u of every box on every rank equals the single-process run with N x the boxes."""
    if _gpu_count() < ranks:
        pytest.skip(f"needs {ranks} GPUs")
    one, many = tmp_path / "one", tmp_path / "many"
    one.mkdir()
    many.mkdir()
    r = run([TOOL, "ranks", "6", str(8 * ranks), "jacobi", str(one)])
    assert r.stdout.startswith("OK"), r.stdout[-2000:] + r.stderr[-2000:]
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={ranks}", "--master-addr", "127.0.0.1",
                        "--master-port", str(29700 + ranks), TOOL, "ranks", "6", "8", "jacobi", str(many)], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    files = sorted(os.listdir(one))
    assert files and files == sorted(os.listdir(many))
    for f in files:
        np.testing.assert_array_equal(np.load(many / f), np.load(one / f), err_msg=f)
