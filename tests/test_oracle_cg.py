"""CPU suite: the oracle's D^-1-preconditioned CG bottom solver (solvers/cg.c of the reference, selected there with -DUSE_CG;
tests/oracle_cg.c on top of the unchanged oracle).  cg() equals the algorithm written out in numpy over oracle_apply_op, and the
F-cycles with CG at the bottom are deterministic with the numbers below -- the numbers the CUDA library must reproduce bit for
bit (tests/test_gpu_cg.py).  No bottom solve of a pinned configuration reaches the 200-iteration cap: the totals over all
bottom solves of the three F-cycles are 21 and 27."""
import numpy as np
import pytest

import hpgmg_b200.api as api
import oracle_bindings as ob
import oracle_cg as oc

SMOOTHERS = [oc.GSRB, oc.CHEBY]
IDS = ["gsrb", "cheby"]
R0, R, P, AP, Z, SCRATCH = (api.VECTORS_RESERVED + q for q in range(6))

# the driver's three solves (hpgmg-fv.c:351-366) with the oracle and CG at the bottom: F-cycle residual norms on levels 0, 1, 2,
# the Richardson error and order, CG iterations over the three solves
ORACLE = {
    (5, oc.GSRB): ([0.0008412952115809391, 0.002463322558838287, 0.0007615331127701587], 2.7415249350612892e-05, 1.966129157787269, 21),
    (5, oc.CHEBY): ([0.0002755795533693206, 0.00035998258120206186, 0.0003416886726139175], 2.6404139047325574e-05, 2.043734151000503, 21),
    (6, oc.GSRB): ([6.934040614714476e-05, 0.0008424295375509816, 0.002464277273031978], 2.889814672876311e-06, 3.2468424887986607, 27),
    (6, oc.CHEBY): ([0.00019277220790148153, 0.00027566209930174335, 0.00036014183781592473], 2.865766864619014e-06, 3.2046084145862688, 27),
}


def ordered_dot(a, b):
    """dot() on one tile: the products summed by one accumulator in k, j, i order (misc.c; oracle dot_vec)."""
    s = 0.0
    for v in (a * b).ravel():
        s += v
    return s


def cg_restated(apply_op, get, put, rtol, dinv, rhs):
    """The CG of solvers/cg.c, step by step: `apply_op(out_id, in_id)` fills the ghosts of `in` and writes A in; get / put move
    the cells of one vector.  Returns the iteration count and whether it stopped on convergence."""
    apply_op(SCRATCH, api.VECTOR_U)
    r0 = rhs - get(SCRATCH)
    r = 1.0 * r0
    z = 1.0 * dinv * r
    p = 1.0 * z
    r_dot_z, norm_of_r0 = ordered_dot(r, z), np.max(np.abs(r))
    x = get(api.VECTOR_U)
    j, converged = 0, (r_dot_z == 0.0 or norm_of_r0 == 0.0)
    while j < 200 and not converged:
        j += 1
        put(P, p)
        apply_op(AP, P)
        Ap = get(AP)
        Ap_dot_p = ordered_dot(Ap, p)
        if Ap_dot_p == 0.0:
            break
        alpha = r_dot_z / Ap_dot_p
        if np.isinf(alpha):
            break
        x = 1.0 * x + alpha * p
        r = 1.0 * r + (-alpha) * Ap
        norm_of_r = np.max(np.abs(r))
        if norm_of_r == 0.0 or norm_of_r < rtol * norm_of_r0:
            converged = True
            break
        z = 1.0 * dinv * r
        r_dot_z_new = ordered_dot(r, z)
        if r_dot_z_new == 0.0:
            break
        beta = r_dot_z_new / r_dot_z
        if np.isinf(beta):
            break
        p = 1.0 * z + beta * p
        r_dot_z = r_dot_z_new
    put(api.VECTOR_U, x)
    return j, converged, {R: r, P: p, Z: z}


@pytest.mark.parametrize("log2", [4, 5])
def test_cg_equals_numpy_restatement(log2):
    """oracle cg() on the bottom level (2^3) from seeded random x and R (ghosts included) against the algorithm in numpy over
    oracle_apply_op; tolerance 0 for x, r, p, z and the iteration count."""
    O = oc.lib()
    H1, H2 = O.oracle_build(log2, oc.GSRB), O.oracle_build(log2, oc.GSRB)
    bottom = O.oracle_num_levels(H1) - 1
    rng = np.random.default_rng(ob.seed("oracle cg", log2))
    U, F = api.VECTOR_U, api.VECTOR_R
    for vid in (U, F):
        a = rng.standard_normal(oc.array(H1, bottom, vid).shape)
        oc.array(H1, bottom, vid)[...] = a
        oc.array(H2, bottom, vid)[...] = a
    n = O.oracle_level_dim(H1, bottom)
    s = slice(2, 2 + n)
    its = O.oracle_cg(H1, bottom, U, F, 1e-3)

    L2 = O.oracle_level(H2, bottom)

    def get(vid):
        return oc.array(H2, bottom, vid)[s, s, s].copy()

    def put(vid, v):
        oc.array(H2, bottom, vid)[s, s, s] = v

    its2, converged, vecs = cg_restated(lambda out, inp: O.oracle_apply_op(L2, out, inp, 1.0), get, put, 1e-3,
                                        get(api.VECTOR_DINV), get(F))
    assert converged and its == its2 and 0 < its < 200
    np.testing.assert_array_equal(oc.array(H1, bottom, U)[s, s, s], get(U))
    for vid, want in vecs.items():
        np.testing.assert_array_equal(oc.array(H1, bottom, vid)[s, s, s], want, err_msg=f"vector {vid}")
    O.oracle_destroy(H1)
    O.oracle_destroy(H2)


@pytest.mark.parametrize("smoother", SMOOTHERS, ids=IDS)
@pytest.mark.parametrize("log2", [5, 6])
def test_fcycles_are_deterministic_and_pinned(log2, smoother):
    a, b = oc.richardson(log2, smoother), oc.richardson(log2, smoother)
    assert a == b
    norms, err, order, krylov = ORACLE[(log2, smoother)]
    assert a[0] == norms and a[1] == err and a[2] == order and a[3] == krylov


def test_included_oracle_is_the_oracle():
    """The oracle compiled into tests/oracle_cg.c is the oracle: its own BiCGStab F-cycle gives the reference's goldens."""
    import ctypes as C
    O = oc.lib()
    H = O.oracle_build(5, 0)
    norms = (C.c_double * 3)()
    err, order = C.c_double(), C.c_double()
    O.oracle_richardson(H, norms, C.byref(err), C.byref(order))
    O.oracle_destroy(H)
    assert list(norms) == ob.goldens()["solves"]["5 1 gsrb"]["norms"]
