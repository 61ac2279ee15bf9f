"""CPU suite: the oracle's weighted Jacobi and L1-Jacobi smoothers (operators/jacobi.c of the reference, selected there with
-DUSE_JACOBI / -DUSE_L1JACOBI; tests/oracle_jacobi.c on top of the unchanged oracle).  One smooth() equals six sweeps
composed from oracle_apply_op and the update in numpy, the kept L1 row inverse is consistent with D^-1, and the F-cycles are
deterministic with the numbers below -- the numbers the CUDA library must reproduce bit for bit (tests/test_gpu_jacobi.py)."""
import ctypes as C

import numpy as np
import pytest

import hpgmg_b200.api as api
import oracle_bindings as ob
import oracle_jacobi as oj

SMOOTHERS = [oj.JACOBI, oj.L1JACOBI]
IDS = ["jacobi", "l1jacobi"]

# the driver's three solves (hpgmg-fv.c:351-366) with the oracle: F-cycle residual norms on levels 0, 1, 2, the Richardson
# error and order, BiCGStab iterations over the three solves
ORACLE = {
    (5, oj.JACOBI): ([0.0038945510405298256, 0.00830936382781311, 0.0016275684757855735], 1.815899360754856e-05, 2.3566080620849745, 21),
    (6, oj.JACOBI): ([0.0005057833951003232, 0.0038991837941014795, 0.008312169381617274], 1.1811926828196248e-06, 3.9433203056881494, 27),
    (5, oj.L1JACOBI): ([0.00474912086726631, 0.009795422674409582, 0.0023943539922050283], 1.7805123921598755e-05, 2.307879927421052, 18),
    (6, oj.L1JACOBI): ([0.0006581325928306514, 0.0047547118667843336, 0.009798784422943907], 1.604705580368973e-06, 3.4727843817009445, 24),
}


def lambda_id(O, H, smoother):
    return O.oracle_jacobi_l1inv_id(H, 0) if smoother == oj.L1JACOBI else api.VECTOR_DINV


@pytest.mark.parametrize("smoother", SMOOTHERS, ids=IDS)
@pytest.mark.parametrize("log2", [4, 5])
def test_smooth_equals_six_composed_sweeps(log2, smoother):
    """oracle_smooth_jacobi on level 0 from seeded random x and rhs (ghosts included) against six steps of
    oracle_apply_op(source) -- which fills the source's ghosts -- and x + (w*lambda)*(rhs - Ax) in numpy."""
    O = oj.lib()
    H1, H2 = O.oracle_jacobi_build(log2, smoother), O.oracle_jacobi_build(log2, smoother)
    rng = np.random.default_rng(ob.seed("oracle jacobi", log2, smoother))
    U, R, E, T = api.VECTOR_U, api.VECTOR_R, api.VECTOR_E, api.VECTOR_TEMP
    for vid in (U, R):
        a = rng.standard_normal(oj.array(H1, 0, vid).shape)
        oj.array(H1, 0, vid)[...] = a
        oj.array(H2, 0, vid)[...] = a
    n = O.oracle_level_dim(H1, 0)
    s = slice(2, 2 + n)
    w = oj.WEIGHT[smoother]
    O.oracle_smooth_jacobi(O.oracle_level(H1, 0), U, R, 1.0, w, lambda_id(O, H1, smoother))
    L2 = O.oracle_level(H2, 0)
    lam = oj.array(H2, 0, lambda_id(O, H2, smoother))[s, s, s].copy()
    rhs = oj.array(H2, 0, R)[s, s, s]
    for step in range(6):
        src, dst = (U, T) if step % 2 == 0 else (T, U)
        O.oracle_apply_op(L2, E, src, 1.0)
        x, ax = oj.array(H2, 0, src)[s, s, s], oj.array(H2, 0, E)[s, s, s]
        oj.array(H2, 0, dst)[s, s, s] = x + (w * lam) * (rhs - ax)
    for vid in (U, T):
        np.testing.assert_array_equal(oj.array(H1, 0, vid)[s, s, s], oj.array(H2, 0, vid)[s, s, s])
    O.oracle_destroy(H1)
    O.oracle_destroy(H2)


def test_l1_inverse_is_consistent_with_dinv():
    """rebuild.c: L1^-1 = 1/Aii where Aii >= 1.5 sum|Aij|, else 1/(Aii + sum|Aij|/2) -- never above D^-1 = 1/Aii, positive."""
    O = oj.lib()
    H = O.oracle_jacobi_build(5, oj.L1JACOBI)
    for l in range(O.oracle_num_levels(H)):
        n = O.oracle_level_dim(H, l)
        s = slice(2, 2 + n)
        l1, dinv = oj.l1inv(H, l)[s, s, s], oj.array(H, l, api.VECTOR_DINV)[s, s, s]
        assert np.all(l1 > 0.0) and np.all(l1 <= dinv), l
        if l == 0:
            assert np.any(l1 < dinv), "the off-diagonal sum never enters"
    O.oracle_destroy(H)


@pytest.mark.parametrize("smoother", SMOOTHERS, ids=IDS)
@pytest.mark.parametrize("log2", [5, 6])
def test_fcycles_are_deterministic_and_pinned(log2, smoother):
    a, b = oj.richardson(log2, smoother), oj.richardson(log2, smoother)
    assert a == b
    norms, err, order, krylov = ORACLE[(log2, smoother)]
    assert a[0] == norms and a[1] == err and a[2] == order and a[3] == krylov


def test_included_oracle_is_the_oracle():
    """The oracle compiled into tests/oracle_jacobi.c is the oracle: its own GSRB F-cycle gives the reference's goldens."""
    O = oj.lib()
    O.oracle_build.restype, O.oracle_build.argtypes = C.c_void_p, [C.c_int, C.c_int]
    O.oracle_richardson.restype, O.oracle_richardson.argtypes = None, [C.c_void_p] + [C.POINTER(C.c_double)] * 3
    H = O.oracle_build(5, 0)
    norms = (C.c_double * 3)()
    err, order = C.c_double(), C.c_double()
    O.oracle_richardson(H, norms, C.byref(err), C.byref(order))
    O.oracle_destroy(H)
    assert list(norms) == ob.goldens()["solves"]["5 1 gsrb"]["norms"]
