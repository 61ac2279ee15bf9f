"""CPU suite: the plain-C restatement of the fv2 Helmholtz flavour (tests/oracle_fv2_helmholtz.c) that
tests/test_gpu_fv2_helmholtz.py compares the library with, and the fv2 Helmholtz library's exports and level layout
(layout-only mode, no device).

The pinned numbers were produced by the oracle itself: they guard it against unintended change.  Two checks tie it to
something else: with a = 0 it gives the fv2 oracle's F-cycles bit for bit, and its operator on the cell averages of a
quadratic with alpha = beta = 1 equals the exact a*u - b*Laplacian(u)."""
import ctypes as C

import numpy as np
import pytest

import hpgmg_b200.api as api
import oracle_fv2 as of
import oracle_fv2_helmholtz as oh
from test_abi import declared_functions

# hpgmg-fv <log2> 1, a = b = 1, BiCGStab bottom: (F-cycle residual norms of the level-0/1/2 solves, Richardson error, order,
# Krylov iterations)
PINS = {
    (5, oh.GSRB): ([0.008975889947651416, 0.010425276508076009, 0.0028418765088511766], 0.00010883303512492382, -0.43199535400463174, 15),
    (5, oh.CHEBY): ([0.006664965671278833, 0.002208924598034491, 0.0006955240450238836], 0.0001137604512812156, -0.4549591313633487, 15),
    (6, oh.GSRB): ([0.005107004798749815, 0.008983964137508571, 0.010428774787027084], 3.486805647334463e-05, 1.6426940610716003, 15),
    (6, oh.CHEBY): ([0.007764479544982716, 0.0066675923106913615, 0.002208678395115394], 4.9153146071811895e-05, 1.211152282619722, 15),
    (7, oh.GSRB): ([0.002020619747297947, 0.0051072771245120885, 0.008984446864565676], 8.992114103129056e-06, 1.955228405317078, 21),
    (7, oh.CHEBY): ([0.004599247060993572, 0.007764820915136195, 0.00666775072068565], 1.6605989579845416e-05, 1.565622332975314, 21),
}
SMOOTHERS = [oh.GSRB, oh.CHEBY, oh.JACOBI, oh.L1JACOBI]


@pytest.mark.parametrize("log2,smoother", sorted(PINS))
def test_oracle_fcycle_is_pinned(log2, smoother):
    assert oh.richardson(log2, smoother, oh.BICGSTAB) == PINS[(log2, smoother)]


def test_gsrb_richardson_order_is_two():
    """hpgmg-fv 7 1 with a = b = 1: the error between the 2h and 4h solutions over the one between h and 2h."""
    _, _, order, _ = oh.richardson(7, oh.GSRB, oh.BICGSTAB)
    assert 1.9 <= order <= 2.1


@pytest.mark.parametrize("bottom", [oh.BICGSTAB, oh.CG])
@pytest.mark.parametrize("smoother", SMOOTHERS)
def test_a_zero_is_the_fv2_oracle(smoother, bottom):
    """a = 0 drops the term: 0*alpha*x - q and the fv2 oracle's (-b*h2inv)*S are the same number, so the Richardson passes
    and the solution of one F-cycle are equal bit for bit."""
    assert oh.richardson(5, smoother, bottom, a=0.0) == of.richardson(5, smoother, bottom)
    with oh.Hier(5, smoother, bottom, a=0.0) as H, of.Hier(5, smoother, bottom) as F:
        assert H.fmg_solve(0) == F.fmg_solve(0)
        np.testing.assert_array_equal(H.interior(0, 1), F.interior(0, 1))


def test_operator_on_quadratics_is_exact():
    """beta = 1, alpha = 1: the operator on the cell averages of u = x^2 + 2y^2 - z^2 + xy equals a*u - b*Laplacian(u) =
    a*u - 4b at the cells whose stencil stays inside the box (a second difference of cell averages of a quadratic is exact)."""
    a, b = 2.0, 1.5
    with oh.Hier(3, a=a, b=b) as H:
        n = H.O.oracle_level_dim(H.H, 0)
        h = 1.0 / n
        lo, hi = np.arange(n) * h, np.arange(1, n + 1) * h
        m1 = (hi ** 2 - lo ** 2) / (2 * h)
        m2 = (hi ** 3 - lo ** 3) / (3 * h)
        X1, Y1, _ = np.meshgrid(m1, m1, m1, indexing="ij")
        X2, Y2, Z2 = np.meshgrid(m2, m2, m2, indexing="ij")
        u = (X2 + 2 * Y2 - Z2 + X1 * Y1).transpose(2, 1, 0)             # [k][j][i]
        for vid in (6, 7, 8, H.ALPHA):                                 # V_BI, V_BJ, V_BK, alpha
            H.array(0, vid)[...] = 1.0
        g = oh.G
        H.array(0, 1)[g:g + n, g:g + n, g:g + n] = u                   # U
        H.O.fvh_level_apply_op(H.F, 0, 3, 1)                           # E = A U
        Au = H.interior(0, 3)
    s = slice(1, n - 1)
    np.testing.assert_allclose(Au[s, s, s], a * u[s, s, s] - 4 * b, rtol=1e-10, atol=1e-9)


@pytest.fixture(scope="module")
def fv2h_layout():
    L = api.bind(C.CDLL(api.FV2_HELMHOLTZ_LIB_PATH))
    L.hpgmg_b200_set_layout_only(1)
    L.hpgmg_b200_set_verbose(0)
    return L


def test_fv2_helmholtz_library_exports_every_declared_symbol():
    lib = C.CDLL(api.FV2_HELMHOLTZ_LIB_PATH)
    missing = [n for n in sorted(declared_functions()) if not hasattr(lib, n)]
    assert not missing, missing


def test_fv2_helmholtz_layout(fv2h_layout):
    """`7 8` with the Helmholtz vector map: radius 1, STAR shape, one ghost layer and the 11 reserved vectors on every level (the
    1^3 bottom also has the bottom solver's 8), levels 256^3 .. 1^3."""
    L = fv2h_layout
    assert L.stencil_get_radius() == 1 and L.stencil_get_shape() == api.STENCIL_SHAPE_STAR
    H = api.Hierarchy(7, 8, build_operator=False, library=L, a=oh.A, b=oh.B, vectors=11)
    L.MGBuild(H.mg, H.level_h, oh.A, oh.B, 1)
    H.built = True
    try:
        assert [H.level(l).contents.dim.i for l in range(H.num_levels)] == [256 >> l for l in range(9)]
        assert [H.level(l).contents.box_ghosts for l in range(H.num_levels)] == [1] * 9
        assert [H.level(l).contents.numVectors for l in range(H.num_levels)] == [11] * 8 + [11 + 8]
        lv = H.level(0).contents
        assert lv.box_dim == 128 and lv.box_jStride == 132 and lv.box_kStride == 132 * 130
    finally:
        H.close()
