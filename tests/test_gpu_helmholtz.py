"""GPU suite (-m gpu), SURVEY.md section 8 row f1: the Helmholtz build.  The reference selects it at compile time
(-DUSE_HELMHOLTZ: defines.h:12-26 adds VECTOR_ALPHA / VECTOR_L1INV, operators.fv4.c:56-85 adds a*alpha*x to the operator,
hpgmg-fv.c:286-288 solves a = b = 1), and so does this library: hpgmg_b200/lib/libhpgmg_b200_helmholtz.so is the same
sources compiled with -DUSE_HELMHOLTZ.  Compared cell by cell, tolerance 0, with oracle/_ref/libhpgmg_ref_helmholtz.so
(the unmodified reference compiled the same way), Dirichlet and periodic."""
import ctypes as C
import os

import numpy as np
import pytest

import hpgmg_b200.api as api
import oracle_bindings as ob

HELM_LIB = os.path.join(os.path.dirname(api.LIB_PATH), "libhpgmg_b200_helmholtz.so")
HELM_REF = os.path.join(ob.REF_DIR, "libhpgmg_ref_helmholtz.so")
pytestmark = pytest.mark.gpu
needs_ref = pytest.mark.skipif(not os.path.exists(HELM_REF), reason="the reference's Helmholtz build (oracle/_ref) is not built")

NVEC = 11                      # VECTORS_RESERVED of the Helmholtz map
U, F, E, Rr, T, DINV, ALPHA, L1INV = 1, 2, 3, 4, 0, 5, 9, 10
A_, B_ = 1.0, 1.0              # hpgmg-fv.c:287


@pytest.fixture(scope="module")
def helm():
    L = api.bind(C.CDLL(HELM_LIB))
    assert L.hpgmg_b200_init(0) == 0
    L.hpgmg_b200_set_verbose(0)
    L.hpgmg_b200_set_smoother(api.SMOOTHER_GSRB)
    yield L


@pytest.fixture(scope="module")
def helm_ref():
    return api.bind(C.CDLL(HELM_REF), {k: api.SIGNATURES[k] for k in ob._REF_SYMBOLS})


def download(L, level, box, vid):
    Lc = level.contents
    out = np.empty(Lc.box_volume, dtype=np.float64)
    L.hpgmg_download_box_vector(level, box, vid, out.ctypes.data_as(C.c_void_p))
    return api.box_view(level, out)


def assert_equal(L, H, R, l, vid, what, interior=True):
    Lc = R.level(l).contents
    n = Lc.box_dim
    s = slice(2, 2 + n) if interior else slice(0, n + 4)
    for b in range(Lc.num_my_boxes):
        np.testing.assert_array_equal(download(L, H.level(l), b, vid)[s, s, s], R.array(l, b, vid)[s, s, s], err_msg=f"{what}: level {l} box {b} vector {vid}")


@needs_ref
@pytest.mark.parametrize("cfg", ["4 1", "4 8", "5 8", "4 27"])
@pytest.mark.parametrize("bc", [api.BC_DIRICHLET, api.BC_PERIODIC])
def test_helmholtz_fmg_equals_reference(helm, helm_ref, cfg, bc):
    log2, boxes = map(int, cfg.split())
    with ob.ref_threads(1):
        R = ob.RefHierarchy(log2, boxes, bc=bc, library=helm_ref, a=A_, b=B_, vectors=NVEC)
        with ob.quiet():
            helm_ref.zero_vector(R.level(0), U)
            helm_ref.FMGSolve(R.mg, 0, U, F, A_, B_, 1e-10)
            helm_ref.residual(R.level(0), T, U, F, A_, B_)
            want = helm_ref.norm(R.level(0), T)
    helm.hpgmg_b200_use_graphs(1)
    with api.Hierarchy(log2, boxes, bc=bc, library=helm, a=A_, b=B_, vectors=NVEC) as H:
        assert H.num_levels == R.num_levels
        for l in range(H.num_levels):
            assert H.level(l).contents.dominant_eigenvalue_of_DinvA == R.level(l).contents.dominant_eigenvalue_of_DinvA
            assert H.level(l).contents.must_subtract_mean == R.level(l).contents.must_subtract_mean == 0      # a*alpha != 0: not singular
            assert_equal(helm, H, R, l, DINV, "D^-1 with the a*alpha term")
            assert_equal(helm, H, R, l, ALPHA, "alpha restricted to the level")
            assert_equal(helm, H, R, l, L1INV, "L1^-1")
        r, _ = H.fmg_solve(0)
        assert r == want
        assert_equal(helm, H, R, 0, U, "Helmholtz FMGSolve: u")


@needs_ref
@pytest.mark.parametrize("op", ["apply_op", "residual", "smooth", "vcycle", "iterative_solver"])
def test_helmholtz_operator_equals_reference(helm, helm_ref, op):
    log2, boxes = 4, 8
    helm.hpgmg_b200_use_graphs(0)
    with ob.ref_threads(1):
        R = ob.RefHierarchy(log2, boxes, library=helm_ref, a=A_, b=B_, vectors=NVEC)
    with api.Hierarchy(log2, boxes, library=helm, a=A_, b=B_, vectors=NVEC) as H:
        rng = np.random.default_rng(hash(op) % (2 ** 32))
        levels = range(H.num_levels) if op == "vcycle" else (0, H.num_levels - 1)
        for l in levels:
            for b in range(R.level(l).contents.num_my_boxes):
                for vid in (U, E, Rr, T):
                    a = rng.standard_normal(R.array(l, b, vid).shape)
                    R.array(l, b, vid)[...] = a
                    helm.hpgmg_upload_box_vector(H.level(l), b, vid, np.ascontiguousarray(a).ctypes.data_as(C.c_void_p))
        l0, r0 = H.level(0), R.level(0)
        with ob.ref_threads(1), ob.quiet():
            if op == "apply_op":
                helm.apply_op(l0, T, U, A_, B_); helm_ref.apply_op(r0, T, U, A_, B_); checks = [(0, T)]
            elif op == "residual":
                helm.residual(l0, T, U, Rr, A_, B_); helm_ref.residual(r0, T, U, Rr, A_, B_); checks = [(0, T)]
            elif op == "smooth":
                helm.smooth(l0, U, Rr, A_, B_); helm_ref.smooth(r0, U, Rr, A_, B_); checks = [(0, U), (0, T)]
            elif op == "vcycle":
                helm.MGVCycle(H.mg, E, Rr, A_, B_, 0); helm_ref.MGVCycle(R.mg, E, Rr, A_, B_, 0); checks = [(l, E) for l in range(H.num_levels)]
            else:
                lb, rb = H.level(H.num_levels - 1), R.level(R.num_levels - 1)
                helm.IterativeSolver(lb, U, Rr, A_, B_, 1e-3); helm_ref.IterativeSolver(rb, U, Rr, A_, B_, 1e-3); checks = [(H.num_levels - 1, U)]
        for l, vid in checks:
            assert_equal(helm, H, R, l, vid, "Helmholtz " + op)


@pytest.mark.parametrize("key", ["4 8 dirichlet helmholtz", "5 8 dirichlet helmholtz", "4 8 periodic helmholtz", "4 27 dirichlet helmholtz"])
def test_helmholtz_goldens(helm, key):
    """The driver's three Richardson solves against tests/golden/goldens.json["variants"] (recorded from the reference built
    -DUSE_HELMHOLTZ, make_goldens.py: variant_record)."""
    log2, boxes, bc, _ = key.split()
    gold = ob.goldens()["variants"][key]
    helm.hpgmg_b200_use_graphs(1)
    with api.Hierarchy(int(log2), int(boxes), bc=api.BC_PERIODIC if bc == "periodic" else api.BC_DIRICHLET, library=helm, a=A_, b=B_, vectors=NVEC) as H:
        assert [H.level(l).contents.dominant_eigenvalue_of_DinvA for l in range(H.num_levels)] == gold["eigs"]
        norms = []
        for l in range(3):
            if l > 0:
                helm.restriction(H.level(l), F, H.level(l - 1), F, api.RESTRICT_CELL)
            norms.append(H.fmg_solve(l)[0])
        helm.richardson_error(H.mg, 0, U)
        assert norms == gold["norms"]
        assert helm.hpgmg_last_richardson_error() == gold["error"] and helm.hpgmg_last_richardson_order() == gold["order"]
