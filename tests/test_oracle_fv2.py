"""CPU suite: the plain-C restatement of the fv2 flavour (tests/oracle_fv2.c) that tests/test_gpu_fv2.py compares the library
with, and the fv2 library's level layout (layout-only mode, no device).

The pinned numbers were produced by the oracle itself: they guard it against unintended change.  The discretisation's own
check does not depend on the oracle: the Richardson order of a second-order operator is close to 2, and the operator with
beta = 1 is exact (-b times the Laplacian) on the cell averages of a quadratic."""
import ctypes as C
import os

import numpy as np
import pytest

import hpgmg_b200.api as api
import oracle_fv2 as of

# hpgmg-fv <log2> 1, BiCGStab bottom: (F-cycle residual norms of the level-0/1/2 solves, Richardson error, order, Krylov iterations)
PINS = {
    (5, of.GSRB): ([0.008996533942771445, 0.010470229445863177, 0.0028902393179073838], 0.00010951570917572002, -0.4280655580936165, 15),
    (5, of.CHEBY): ([0.006712274084555492, 0.002231494786226529, 0.000713389333514937], 0.00011479017701587508, -0.44738215638831497, 15),
    (6, of.GSRB): ([0.005124050340248654, 0.009004624506215309, 0.010473742265296293], 3.50623121792926e-05, 1.6436979248570451, 15),
    (6, of.CHEBY): ([0.007796541597861584, 0.006714908396011465, 0.002231245112297279], 4.951142670377639e-05, 1.2136717625326336, 15),
    (7, of.GSRB): ([0.002026794038565316, 0.005124323173229639, 0.009005108214197088], 9.040178890466766e-06, 1.955552413506433, 21),
    (7, of.CHEBY): ([0.004614961596605349, 0.007796883712259617, 0.0067150672747571805], 1.6704097104294855e-05, 1.5676016004438489, 21),
}


@pytest.mark.parametrize("log2,smoother", sorted(PINS))
def test_oracle_fcycle_is_pinned(log2, smoother):
    assert of.richardson(log2, smoother, of.BICGSTAB) == PINS[(log2, smoother)]


@pytest.mark.parametrize("smoother", [of.GSRB, of.CHEBY, of.JACOBI, of.L1JACOBI])
def test_cg_bottom_matches_bicgstab_on_one_cell(smoother):
    """The fv2 hierarchy ends at 1^3, where both Krylov solvers reach the answer of the single equation in one iteration with the
    same arithmetic: the two bottom solvers give the same F-cycles."""
    assert of.richardson(5, smoother, of.CG) == of.richardson(5, smoother, of.BICGSTAB)


def test_gsrb_richardson_order_is_two():
    """hpgmg-fv 7 1: the error between the 2h and 4h solutions over the one between h and 2h, a second-order operator."""
    _, _, order, _ = of.richardson(7, of.GSRB, of.BICGSTAB)
    assert 1.9 <= order <= 2.1


def test_operator_is_exact_on_quadratics():
    """beta = 1: -b h^-2 (x[i+1] - 2x + x[i-1] + ...) on the cell averages of u = x^2 + 2y^2 - z^2 + xy equals -b * Laplacian u = -4b
    at interior cells (a second difference of cell averages of a quadratic is exact)."""
    n, h, b = 8, 1.0 / 8, 1.5
    e = np.arange(n + 3) * h - h                 # cell low edges, one ghost cell on each side
    lo, hi = e[:-1], e[1:]

    def avg(f1, f2):                             # average over [lo, hi] of the 1-D monomials x^2 (f2) and x (f1)
        return f1(lo, hi), f2(lo, hi)
    m1 = (hi ** 2 - lo ** 2) / (2 * h)
    m2 = (hi ** 3 - lo ** 3) / (3 * h)
    X1, Y1, Z1 = np.meshgrid(m1, m1, m1, indexing="ij")
    X2, Y2, Z2 = np.meshgrid(m2, m2, m2, indexing="ij")
    u = X2 + 2 * Y2 - Z2 + X1 * Y1
    c = u[1:-1, 1:-1, 1:-1]
    Au = -b * (1.0 / h ** 2) * ((u[2:, 1:-1, 1:-1] - c) + (u[:-2, 1:-1, 1:-1] - c) + (u[1:-1, 2:, 1:-1] - c) + (u[1:-1, :-2, 1:-1] - c)
                                + (u[1:-1, 1:-1, 2:] - c) + (u[1:-1, 1:-1, :-2] - c))
    np.testing.assert_allclose(Au, -b * (2 + 4 - 2), rtol=1e-10)


@pytest.fixture(scope="module")
def fv2_layout():
    L = api.bind(C.CDLL(api.FV2_LIB_PATH))
    L.hpgmg_b200_set_layout_only(1)
    L.hpgmg_b200_set_verbose(0)
    return L


def test_fv2_layout_has_one_ghost_layer(fv2_layout):
    """The fv2 library's `7 8` hierarchy: radius 1, STAR shape, ghosts 1 on every level, levels 256^3 .. 2^3, 1^3."""
    L = fv2_layout
    assert L.stencil_get_radius() == 1 and L.stencil_get_shape() == api.STENCIL_SHAPE_STAR
    H = api.Hierarchy(7, 8, build_operator=False, library=L)
    L.MGBuild(H.mg, H.level_h, 0.0, 1.0, 1)
    H.built = True
    try:
        assert [H.level(l).contents.dim.i for l in range(H.num_levels)] == [256, 128, 64, 32, 16, 8, 4, 2, 1]
        assert [H.level(l).contents.box_ghosts for l in range(H.num_levels)] == [1] * 9
        lv = H.level(0).contents
        assert lv.box_dim == 128 and lv.box_jStride == 132 and lv.box_kStride == 132 * 130
    finally:
        H.close()
