"""GPU suite (-m gpu), SURVEY.md section 8 row f1: the same path with PERIODIC boundaries (the reference's -DUSE_PERIODIC_BC
driver: hpgmg-fv.c:276-302, level.c:559-563 / 757-761 wrap-around neighbours, mg.c:1016-1017 and 1317-1320 mean
subtraction of the singular Poisson problem, solvers.c:30-38).  Compared cell by cell, tolerance 0, with the unmodified
reference library (oracle/_ref) driven through the same call sequence where the reference is built, and with the pins of
tests/golden/pins.json everywhere."""
import numpy as np
import pytest

import hpgmg_b200.api as api
import oracle_bindings as ob
from test_gpu_parity import assert_level_equal, mirror_random, reference

pytestmark = pytest.mark.gpu

U, E, Rr, T, F = api.VECTOR_U, api.VECTOR_E, api.VECTOR_R, api.VECTOR_TEMP, api.VECTOR_F


@pytest.mark.parametrize("cfg", ["4 1", "4 8", "5 8", "4 27", "6 1"])
@pytest.mark.parametrize("graphs", [True, False])
def test_periodic_fmg_equals_reference(gpu_lib, cfg, graphs):
    """setup (problem, black-box diagonal, mean(f) removal), FMGSolve and the final residual norm"""
    log2, boxes = map(int, cfg.split())
    if not graphs and cfg not in ("4 8", "5 8"):
        pytest.skip("stream-launched variant on two configurations only")
    key = f"periodic FMGSolve {cfg}"                        # the same pins with and without graphs
    with ob.ref_threads(1):                                  # the reference's mean()/dot() are order-defined on one thread only
        R = reference(log2, boxes, bc=api.BC_PERIODIC)
        want = R.fmg_solve(0) if R else None
    with api.Hierarchy(log2, boxes, bc=api.BC_PERIODIC, use_graphs=graphs) as H:
        assert R is None or H.num_levels == R.num_levels
        for l in range(H.num_levels):
            assert H.level(l).contents.must_subtract_mean == 1
            eig = H.level(l).contents.dominant_eigenvalue_of_DinvA
            ref_eig = R.level(l).contents.dominant_eigenvalue_of_DinvA if R else None
            if R is not None:
                assert R.level(l).contents.must_subtract_mean == 1
                assert eig == ref_eig
            ob.pin(f"{key}: eig level {l}", eig, ref_eig)
        r, _ = H.fmg_solve(0)
        assert R is None or r == want
        ob.pin(f"{key}: norm", r, want)
        assert_level_equal(H, R, 0, U, "in", f"{key}: u")
        assert_level_equal(H, R, 0, F, "in", f"{key}: f with its mean removed")
        r2, _ = H.fmg_solve(0)                               # and again (replayed recording where one exists)
        assert r2 == r
        err, order, norms = H.richardson()
    if R is not None:
        with ob.ref_threads(1):
            norms_ref = []
            for l in range(3):
                if l > 0:
                    R.call("restriction", R.level(l), F, R.level(l - 1), F, api.RESTRICT_CELL)
                with ob.quiet():
                    R.L.zero_vector(R.level(l), U)
                    R.L.FMGSolve(R.mg, l, U, F, 0.0, 1.0, 1e-10)
                    R.L.residual(R.level(l), T, U, F, 0.0, 1.0)
                    norms_ref.append(R.L.norm(R.level(l), T))
        assert [n[0] for n in norms] == norms_ref
    for l in range(3):
        ob.pin(f"{key}: richardson norm level {l}", norms[l][0], norms_ref[l] if R else None)


OPS = ["exchange_box", "exchange_star", "exchange_nocorners", "apply_op", "residual", "smooth_gsrb", "interp_v2", "interp_v4",
       "restrict_cell", "mean_shift", "rebuild_blackbox", "iterative_solver", "vcycle"]


@pytest.mark.parametrize("cfg", ["4 8", "4 1", "5 8", "4 27"])
@pytest.mark.parametrize("op", OPS)
def test_periodic_operator_equals_reference(gpu_lib, cfg, op):
    log2, boxes = map(int, cfg.split())
    L = gpu_lib
    with api.Hierarchy(log2, boxes, bc=api.BC_PERIODIC, use_graphs=False) as H:
        with ob.ref_threads(1):
            R = reference(log2, boxes, bc=api.BC_PERIODIC)
        rng = np.random.default_rng(ob.seed(cfg, op, "periodic"))
        mirror_random(H, R, rng, (0, 1), (U, E, Rr, T))
        key = f"periodic operator {cfg} {op}"
        Rc = R or ob.NoReference()
        l0, l1, r0, r1 = H.level(0), H.level(1), Rc.level(0), Rc.level(1)
        a, b = 0.0, 1.0
        checks = []
        with ob.ref_threads(1):
            if op.startswith("exchange_"):
                shape = {"box": 0, "star": 1, "nocorners": 2}[op.split("_")[1]]
                L.exchange_boundary(l0, U, shape); Rc.call("exchange_boundary", r0, U, shape)
                L.apply_BCs(l0, U, shape); Rc.call("apply_BCs", r0, U, shape)           # no-ops on a periodic level
                checks = [(0, U, "all")]
            elif op == "apply_op":
                L.apply_op(l0, T, U, a, b); Rc.call("apply_op", r0, T, U, a, b); checks = [(0, T, "in"), (0, U, "all")]
            elif op == "residual":
                L.residual(l0, T, U, Rr, a, b); Rc.call("residual", r0, T, U, Rr, a, b); checks = [(0, T, "in"), (0, U, "all")]
            elif op == "smooth_gsrb":
                L.smooth(l0, U, Rr, a, b); Rc.call("smooth", r0, U, Rr, a, b); checks = [(0, U, "in"), (0, T, "in")]
            elif op == "restrict_cell":
                L.restriction(l1, Rr, l0, T, 0); Rc.call("restriction", r1, Rr, r0, T, 0); checks = [(1, Rr, "all")]
            elif op == "interp_v2":
                L.interpolation_v2(l0, U, 1.0, l1, E); Rc.call("interpolation_v2", r0, U, 1.0, r1, E); checks = [(0, U, "in"), (1, E, "all")]
            elif op == "interp_v4":
                L.interpolation_v4(l0, U, 0.0, l1, E); Rc.call("interpolation_v4", r0, U, 0.0, r1, E); checks = [(0, U, "in"), (1, E, "all")]
            elif op == "mean_shift":
                m, mr = L.mean(l0, U), Rc.call("mean", r0, U)
                assert R is None or m == mr
                ob.pin(f"{key}: mean", m, mr)
                L.shift_vector(l0, U, U, -m); Rc.call("shift_vector", r0, U, U, -m); checks = [(0, U, "all")]
            elif op == "rebuild_blackbox":
                L.rebuild_operator_blackbox(l0, a, b, 4); Rc.call("rebuild_operator_blackbox", r0, a, b, 4)
                ref_eig = r0.contents.dominant_eigenvalue_of_DinvA if R else None
                assert R is None or l0.contents.dominant_eigenvalue_of_DinvA == ref_eig
                ob.pin(f"{key}: eig", l0.contents.dominant_eigenvalue_of_DinvA, ref_eig)
                checks = [(0, api.VECTOR_DINV, "in"), (0, E, "in")]
            elif op == "iterative_solver":
                lb, rb = H.level(H.num_levels - 1), R.level(R.num_levels - 1) if R else None
                mirror_random(H, R, rng, (H.num_levels - 1,), (U, Rr))
                L.IterativeSolver(lb, U, Rr, a, b, 1e-3); Rc.call("IterativeSolver", rb, U, Rr, a, b, 1e-3)
                checks = [(H.num_levels - 1, U, "in")]
            elif op == "vcycle":
                L.MGVCycle(H.mg, E, Rr, a, b, 0); Rc.call("MGVCycle", Rc.mg, E, Rr, a, b, 0)
                checks = [(l, E, "in") for l in range(H.num_levels)]
            else:
                raise AssertionError(op)
        for l, vid, where in checks:
            assert_level_equal(H, R, l, vid, where, key)


@pytest.mark.parametrize("cfg", ["4 1", "4 8", "5 8", "4 27"])
def test_periodic_goldens(gpu_lib, cfg):
    """The driver's three Richardson solves (hpgmg-fv.c:351-366) against tests/golden/goldens.json["variants"], recorded from the
    reference built -DUSE_PERIODIC_BC semantics (make_goldens.py: variant_record)."""
    log2, boxes = map(int, cfg.split())
    gold = ob.goldens()["variants"][f"{log2} {boxes} periodic poisson"]
    with api.Hierarchy(log2, boxes, bc=api.BC_PERIODIC) as H:
        assert [H.level(l).contents.dim.i for l in range(H.num_levels)] == gold["dims"]
        assert [H.level(l).contents.dominant_eigenvalue_of_DinvA for l in range(H.num_levels)] == gold["eigs"]
        err, order, norms = H.richardson()
        assert [n[0] for n in norms] == gold["norms"]
        assert err == gold["error"] and order == gold["order"]
