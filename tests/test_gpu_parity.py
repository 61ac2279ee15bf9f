"""GPU suite (-m gpu): the CUDA path, called through the C-ABI, against
  (1) goldens produced by the unmodified reference (tests/golden/goldens.json),
  (2) the reference library itself on identical inputs, operator by operator (oracle/_ref, prebuilt), and
  (3) the plain-C oracle restatement.
Contract (BASELINE.json north_star): per-cycle residual norms within 1e-10 relative, error norm and
order within 1e-6, index mapping bit-exact.  The kernels are built -fmad=false with the reference's
association order, so the tests demand MORE: bit-for-bit equality (rel tolerance 0)."""
import ctypes as C

import numpy as np
import pytest

import hpgmg_b200.api as api
import oracle_bindings as ob

pytestmark = pytest.mark.gpu

RTOL_NORM = 0.0        # contract: 1e-10; achieved and enforced: exact
RTOL_ERROR = 0.0       # contract: 1e-6


def close(a, b, rtol):
    return a == b if rtol == 0.0 else abs(a - b) <= rtol * abs(b)


# ------------------------------------------------------------------------------------------------ FMG
GSRB = ["4 1", "5 1", "6 1", "4 8", "5 8", "6 8", "4 27", "5 27", "5 64", "7 8",
        "8 8"]                          # BASELINE config 4 on one GPU: 512^3 as 2^3 boxes of 256^3
CHEBY = ["5 1", "5 8", "6 8", "5 27", "7 8",
         "7 64"]                        # BASELINE config 5: 512^3 as 4^3 boxes of 128^3


@pytest.mark.parametrize("cfg,smoother", [(c, "gsrb") for c in GSRB] + [(c, "cheby") for c in CHEBY])
def test_fmg_matches_reference_goldens(gpu_lib, cfg, smoother):
    log2, boxes = map(int, cfg.split())
    g = ob.goldens()["solves"][f"{cfg} {smoother}"]
    with api.Hierarchy(log2, boxes, smoother=api.SMOOTHER_CHEBY if smoother == "cheby" else api.SMOOTHER_GSRB) as H:
        assert [H.level(l).contents.dim.i for l in range(H.num_levels)] == g["dims"]
        assert [H.level(l).contents.box_dim for l in range(H.num_levels)] == g["box_dims"]
        eigs = [H.level(l).contents.dominant_eigenvalue_of_DinvA for l in range(H.num_levels)]
        assert eigs == g["eigs"], "Gershgorin bound per level (rebuild.c:204)"
        gpu_lib.MGResetTimers(H.mg)
        err, order, norms = H.richardson()
        for l in range(3):
            assert close(norms[l][0], g["norms"][l], RTOL_NORM), f"F-cycle residual norm on level {l}: {norms[l][0]!r} vs {g['norms'][l]!r}"
        assert norms[0][1] == pytest.approx(g["norms"][0] / g["norm_of_F"], rel=1e-15)
        assert close(err, g["error"], RTOL_ERROR), (err, g["error"])
        assert order == pytest.approx(g["order"], rel=1e-12)
        bottom = H.level(H.num_levels - 1).contents
        assert bottom.Krylov_iterations == g["krylov_iterations_3_solves"]
    gpu_lib.hpgmg_b200_set_smoother(api.SMOOTHER_GSRB)


def test_graph_replay_equals_stream_launch(gpu_lib):
    """The captured CUDA graph and plain stream launches run the same kernels: identical bits, and the
    replay of a recorded graph is deterministic."""
    out = {}
    for graphs in (False, True):
        with api.Hierarchy(5, 8, use_graphs=graphs) as H:
            a = H.fmg_solve(0)
            b = H.fmg_solve(0)
            c = H.fmg_solve(0)
            assert a == b == c
            out[graphs] = (a, api.download(H.level(0), 3, api.VECTOR_U).copy())
    assert out[False][0] == out[True][0]
    np.testing.assert_array_equal(out[False][1], out[True][1])
    gpu_lib.hpgmg_b200_use_graphs(1)


@pytest.mark.parametrize("cfg,smoother", [("5 8", api.SMOOTHER_GSRB), ("4 27", api.SMOOTHER_GSRB), ("5 1", api.SMOOTHER_CHEBY)])
def test_coarse_kernel_equals_multilaunch_path(gpu_lib, cfg, smoother):
    """The single-block coarse-cycle kernel (coarse.cu) and the one-launch-per-operator path give the same bits
    on every level (U, R, TEMP of all boxes)."""
    log2, boxes = map(int, cfg.split())
    snap = {}
    for coarse in (0, 1):
        gpu_lib.hpgmg_b200_use_coarse_kernel(coarse)
        with api.Hierarchy(log2, boxes, smoother=smoother, use_graphs=False) as H:
            launches0 = gpu_lib.hpgmg_b200_kernel_launches()
            r = H.fmg_solve(0)
            launches = gpu_lib.hpgmg_b200_kernel_launches() - launches0
            arrays = [api.download(H.level(l), b, v).copy() for l in range(H.num_levels)
                      for b in range(H.level(l).contents.num_my_boxes) for v in (api.VECTOR_U, api.VECTOR_R)]
            its = H.level(H.num_levels - 1).contents.Krylov_iterations
            snap[coarse] = (r, arrays, its, launches)
    gpu_lib.hpgmg_b200_use_coarse_kernel(1)
    gpu_lib.hpgmg_b200_set_smoother(api.SMOOTHER_GSRB)
    assert snap[0][0] == snap[1][0] and snap[0][2] == snap[1][2]
    for a, b in zip(snap[0][1], snap[1][1]):
        n = a.shape[0] - 4
        s = slice(2, 2 + n)
        np.testing.assert_array_equal(a[s, s, s], b[s, s, s])
    assert snap[1][3] < snap[0][3], "the coarse kernel must remove launches"


def test_fmg_solve_host_buffers(gpu_lib):
    """The end-to-end entry point with HOST buffers (what bench.py's e2e times): dense cells in, dense cells out; the
    download of u overlaps the final residual, and a replayed recording must give the same answer as the first call."""
    with api.Hierarchy(5, 8) as H:
        r, _ = H.fmg_solve(0)
        lvl = H.level(0)
        Lc = lvl.contents
        n, nb = Lc.box_dim, Lc.num_my_boxes
        f = np.concatenate([np.ascontiguousarray(api.interior(lvl, api.download(lvl, b, api.VECTOR_F))).reshape(-1) for b in range(nb)])
        u_ref = np.concatenate([np.ascontiguousarray(api.interior(lvl, api.download(lvl, b, api.VECTOR_U))).reshape(-1) for b in range(nb)])
        assert gpu_lib.hpgmg_fmg_solve_host_bytes(H.mg, 0) == nb * n ** 3 * 8
        for b in range(nb):                                  # the call must bring F itself: wipe the device copy
            api.upload(lvl, b, api.VECTOR_F, np.zeros(Lc.box_volume))
        for attempt in range(3):                             # first call records, later calls replay
            u = np.full(nb * n ** 3, np.nan)
            r2 = gpu_lib.hpgmg_fmg_solve_host(H.mg, 0, api.VECTOR_U, api.VECTOR_F, 0.0, 1.0, 1e-10, f.ctypes.data_as(C.c_void_p), u.ctypes.data_as(C.c_void_p))
            assert r2 == r, attempt
            np.testing.assert_array_equal(u, u_ref)
        assert gpu_lib.hpgmg_last_norm_of_residual(H.mg) == r
    gpu_lib.hpgmg_b200_use_graphs(0)
    try:                                                     # the same without recording (plain stream launches on two streams)
        with api.Hierarchy(4, 8, use_graphs=False) as H:
            r, _ = H.fmg_solve(0)
            lvl = H.level(0)
            nb, n = lvl.contents.num_my_boxes, lvl.contents.box_dim
            f = np.concatenate([np.ascontiguousarray(api.interior(lvl, api.download(lvl, b, api.VECTOR_F))).reshape(-1) for b in range(nb)])
            u_ref = np.concatenate([np.ascontiguousarray(api.interior(lvl, api.download(lvl, b, api.VECTOR_U))).reshape(-1) for b in range(nb)])
            u = np.zeros(nb * n ** 3)
            assert gpu_lib.hpgmg_fmg_solve_host(H.mg, 0, api.VECTOR_U, api.VECTOR_F, 0.0, 1.0, 1e-10, f.ctypes.data_as(C.c_void_p), u.ctypes.data_as(C.c_void_p)) == r
            np.testing.assert_array_equal(u, u_ref)
    finally:
        gpu_lib.hpgmg_b200_use_graphs(1)


@pytest.mark.gpu
def test_pipelined_host_solves_equal_the_serial_call(gpu_lib):
    """hpgmg_fmg_solve_host_submit / _wait: a stream of solves with two in flight (upload of the next and download of the
    previous one overlap the running solve).  Alternating right-hand sides f and 2f: every ticket must return exactly
    what the serial call returns for ITS input, in pinned and in pageable host memory."""
    with api.Hierarchy(5, 8) as H:
        lvl = H.level(0)
        Lc = lvl.contents
        n, nb = Lc.box_dim, Lc.num_my_boxes
        f1 = np.concatenate([np.ascontiguousarray(api.interior(lvl, api.download(lvl, b, api.VECTOR_F))).reshape(-1) for b in range(nb)])
        fs = [f1, 2.0 * f1]
        want = []
        for f in fs:
            u = np.zeros_like(f)
            r = gpu_lib.hpgmg_fmg_solve_host(H.mg, 0, api.VECTOR_U, api.VECTOR_F, 0.0, 1.0, 1e-10, f.ctypes.data_as(C.c_void_p), u.ctypes.data_as(C.c_void_p))
            want.append((r, u))
        assert want[0][0] == ob.goldens()["solves"]["5 8 gsrb"]["norms"][0]
        assert want[1][0] != want[0][0]
        nbytes = f1.nbytes
        pinned = [gpu_lib.hpgmg_b200_host_alloc_pinned(nbytes) for _ in range(4)]
        try:
            for use_pinned in (True, False):
                us = [np.full_like(f1, np.nan) for _ in range(2)]
                if use_pinned:
                    for q in range(2):
                        C.memmove(pinned[q], fs[q].ctypes.data, nbytes)
                    fin = [pinned[0], pinned[1]]
                    uout = [pinned[2], pinned[3]]
                else:
                    fin = [f.ctypes.data_as(C.c_void_p) for f in fs]
                    uout = [u.ctypes.data_as(C.c_void_p) for u in us]
                tickets = []
                got = []

                def finish():
                    q, t = tickets.pop(0)
                    r = gpu_lib.hpgmg_fmg_solve_host_wait(H.mg, t)
                    if use_pinned:
                        C.memmove(us[q].ctypes.data, pinned[2 + q], nbytes)
                    got.append((q, r, us[q].copy()))
                    us[q][:] = np.nan
                for step in range(7):
                    q = step % 2
                    if len(tickets) == 2:
                        finish()
                    tickets.append((q, gpu_lib.hpgmg_fmg_solve_host_submit(H.mg, 0, api.VECTOR_U, api.VECTOR_F, 0.0, 1.0, 1e-10, fin[q], uout[q])))
                while tickets:
                    finish()
                assert len(got) == 7
                for q, r, u in got:
                    assert r == want[q][0]
                    np.testing.assert_array_equal(u, want[q][1])
        finally:
            for p_ in pinned:
                gpu_lib.hpgmg_b200_host_free_pinned(p_)


# ------------------------------------------------------------------------------ operator by operator
def mirror_random(H, R, rng, levels, ids):
    """Identical seeded data (ghost zones included) in our device level and, when R is not None, the reference's host level."""
    for l in levels:
        Lc = H.level(l).contents
        n = Lc.box_dim + 2 * Lc.box_ghosts
        for b in range(Lc.num_my_boxes):
            for vid in ids:
                a = rng.standard_normal((n, n, Lc.box_jStride))
                if R is not None:
                    R.array(l, b, vid)[...] = a
                api.upload(H.level(l), b, vid, a)


def assert_level_equal(H, R, l, vid, where, what):
    """Our vector vid on level l, cell by cell: against the reference's when R is not None, and against the reference's
    recorded under `what` (ob.pin)."""
    Lc = H.level(l).contents
    n = Lc.box_dim
    s = slice(2, 2 + n) if where == "in" else slice(0, n + 4)
    ours = [api.download(H.level(l), b, vid)[s, s, s] for b in range(Lc.num_my_boxes)]
    theirs = None if R is None else [R.array(l, b, vid)[s, s, s] for b in range(Lc.num_my_boxes)]
    if R is not None:
        for b in range(Lc.num_my_boxes):
            np.testing.assert_array_equal(ours[b], theirs[b], err_msg=f"{what}: level {l} box {b} vec {vid} ({where})")
    ob.pin(f"{what}: level {l} vec {vid} ({where})", ours, theirs)


def reference(*args, **kw):
    """The reference library's hierarchy, or None where the reference is not built (the pins stand in for it)."""
    return ob.RefHierarchy(*args, **kw) if ob.have_ref(kw.get("cheby", False)) else None


OPS = ["exchange_box", "exchange_star", "exchange_nocorners", "bc_v4_box", "bc_v4_nocorners", "bc_v2_box", "bc_v1_box",
       "apply_op", "residual", "smooth_gsrb", "restrict_cell", "restrict_face_i", "restrict_face_j", "restrict_face_k",
       "interp_v2", "interp_v4_prescale0", "interp_v4_prescale1", "zero", "init", "scale", "add", "mul", "invert", "shift",
       "color", "random", "dot_norm_mean", "extrapolate_betas", "rebuild_blackbox", "iterative_solver", "vcycle"]


@pytest.mark.parametrize("cfg", ["4 8", "4 27", "4 1", "5 8", "6 1"])
@pytest.mark.parametrize("op", OPS)
def test_operator_equals_reference(gpu_lib, cfg, op):
    log2, boxes = map(int, cfg.split())
    L = gpu_lib
    U, E, Rr, T, F, DINV = api.VECTOR_U, api.VECTOR_E, api.VECTOR_R, api.VECTOR_TEMP, api.VECTOR_F, api.VECTOR_DINV
    BI, BJ, BK = api.VECTOR_BETA_I, api.VECTOR_BETA_J, api.VECTOR_BETA_K
    with api.Hierarchy(log2, boxes, use_graphs=False) as H:
        R = reference(log2, boxes)
        rng = np.random.default_rng(ob.seed(cfg, op))
        mirror_random(H, R, rng, (0, 1), (U, E, Rr, T))
        Rc = R or ob.NoReference()
        l0, l1, r0, r1 = H.level(0), H.level(1), Rc.level(0), Rc.level(1)
        a, b = 0.0, 1.0
        checks = []
        key = f"operator {cfg} {op}"

        def same(what, ours, theirs):
            if R is not None:
                assert ours == theirs, (what, ours, theirs)
            ob.pin(f"{key}: {what}", ours, theirs)

        if op.startswith("exchange_"):
            shape = {"box": 0, "star": 1, "nocorners": 2}[op.split("_")[1]]
            L.exchange_boundary(l0, U, shape); Rc.call("exchange_boundary", r0, U, shape); checks = [(0, U, "all")]
        elif op.startswith("bc_"):
            v, shp = op.split("_")[1], {"box": 0, "nocorners": 2}[op.split("_")[2]]
            L.exchange_boundary(l0, U, shp); Rc.call("exchange_boundary", r0, U, shp)
            getattr(L, f"apply_BCs_{v}")(l0, U, shp)
            with ob.ref_threads(1):
                Rc.call(f"apply_BCs_{v}", r0, U, shp)
            checks = [(0, U, "all")]
        elif op == "apply_op":
            L.apply_op(l0, T, U, a, b); Rc.call("apply_op", r0, T, U, a, b); checks = [(0, T, "in"), (0, U, "all")]
        elif op == "residual":
            L.residual(l0, T, U, Rr, a, b); Rc.call("residual", r0, T, U, Rr, a, b); checks = [(0, T, "in"), (0, U, "all")]
        elif op == "smooth_gsrb":
            L.smooth(l0, U, Rr, a, b); Rc.call("smooth", r0, U, Rr, a, b); checks = [(0, U, "in"), (0, T, "in")]
        elif op.startswith("restrict_"):
            t = {"cell": 0, "face_i": 1, "face_j": 2, "face_k": 3}[op[len("restrict_"):]]
            L.restriction(l1, Rr, l0, T, t); Rc.call("restriction", r1, Rr, r0, T, t); checks = [(1, Rr, "all")]
        elif op == "interp_v2":
            L.interpolation_v2(l0, U, 1.0, l1, E); Rc.call("interpolation_v2", r0, U, 1.0, r1, E); checks = [(0, U, "in"), (1, E, "all")]
        elif op.startswith("interp_v4"):
            ps = float(op[-1])
            L.interpolation_v4(l0, U, ps, l1, E); Rc.call("interpolation_v4", r0, U, ps, r1, E); checks = [(0, U, "in"), (1, E, "all")]
        elif op == "zero":
            L.zero_vector(l0, U); Rc.call("zero_vector", r0, U); checks = [(0, U, "all")]
        elif op == "init":
            L.init_vector(l0, U, 3.25); Rc.call("init_vector", r0, U, 3.25); checks = [(0, U, "all")]
        elif op == "scale":
            L.scale_vector(l0, T, -1.7, U); Rc.call("scale_vector", r0, T, -1.7, U); checks = [(0, T, "all")]
        elif op == "add":
            L.add_vectors(l0, T, 0.3, U, -2.1, E); Rc.call("add_vectors", r0, T, 0.3, U, -2.1, E); checks = [(0, T, "all")]
        elif op == "mul":
            L.mul_vectors(l0, T, 1.3, U, E); Rc.call("mul_vectors", r0, T, 1.3, U, E); checks = [(0, T, "all")]
        elif op == "invert":
            L.invert_vector(l0, T, 2.0, U); Rc.call("invert_vector", r0, T, 2.0, U); checks = [(0, T, "all")]
        elif op == "shift":
            L.shift_vector(l0, T, U, 0.125); Rc.call("shift_vector", r0, T, U, 0.125); checks = [(0, T, "all")]
        elif op == "color":
            L.color_vector(l0, T, 4, 1, 2, 3); Rc.call("color_vector", r0, T, 4, 1, 2, 3); checks = [(0, T, "all")]
        elif op == "random":
            L.random_vector(l0, T); Rc.call("random_vector", r0, T); checks = [(0, T, "all")]
        elif op == "dot_norm_mean":
            # the reference's OpenMP reduction order over tiles is only defined for one thread; norm is order-free
            same("norm", L.norm(l0, U), Rc.call("norm", r0, U))
            with ob.ref_threads(1):
                same("dot", L.dot(l0, U, E), Rc.call("dot", r0, U, E))
                same("mean", L.mean(l0, U), Rc.call("mean", r0, U))
            same("error", L.error(l0, U, E), Rc.call("error", r0, U, E))
        elif op == "extrapolate_betas":
            mirror_random(H, R, rng, (0,), (BI, BJ, BK))
            L.extrapolate_betas(l0); Rc.call("extrapolate_betas", r0)
            Lc = l0.contents
            n = Lc.box_dim
            ring = slice(1, n + 3)       # only the first ghost layer is ever read (and is order-independent)
            for vid in (BI, BJ, BK):
                ours = [api.download(l0, bx, vid)[ring, ring, ring] for bx in range(Lc.num_my_boxes)]
                if R is not None:
                    for bx in range(Lc.num_my_boxes):
                        np.testing.assert_array_equal(ours[bx], R.array(0, bx, vid)[ring, ring, ring])
                ob.pin(f"{key}: vec {vid} (ring)", ours, [R.array(0, bx, vid)[ring, ring, ring] for bx in range(Lc.num_my_boxes)] if R else None)
        elif op == "rebuild_blackbox":
            L.rebuild_operator_blackbox(l0, a, b, 4); Rc.call("rebuild_operator_blackbox", r0, a, b, 4)
            same("eig", l0.contents.dominant_eigenvalue_of_DinvA, r0.contents.dominant_eigenvalue_of_DinvA if R else None)
            checks = [(0, DINV, "in"), (0, E, "in")]
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


@pytest.mark.parametrize("log2", [7, 8])
def test_large_single_box_operators_equal_reference(gpu_lib, log2):
    """One 128^3 box (`7 1`: the box size behind the headline number) and one 256^3 box (`8 1`: BASELINE config 4):
    smooth, residual, restriction and both interpolations cell by cell against the reference library -- the
    TMA-staged kernels, their k-chunking and the k-marching interpolation at full box size."""
    L = gpu_lib
    U, E, Rr, T = api.VECTOR_U, api.VECTOR_E, api.VECTOR_R, api.VECTOR_TEMP
    with api.Hierarchy(log2, 1, use_graphs=False) as H:
        R = reference(log2, 1)
        Rc = R or ob.NoReference()
        rng = np.random.default_rng(log2)
        mirror_random(H, R, rng, (0,), (U, Rr, T))
        mirror_random(H, R, rng, (1,), (E,))
        l0, l1, r0, r1 = H.level(0), H.level(1), Rc.level(0), Rc.level(1)
        key = f"large box {log2} 1"
        L.smooth(l0, U, Rr, 0.0, 1.0); Rc.call("smooth", r0, U, Rr, 0.0, 1.0)
        assert_level_equal(H, R, 0, U, "in", f"{key} smooth")
        assert_level_equal(H, R, 0, T, "in", f"{key} smooth (TEMP)")
        L.residual(l0, T, U, Rr, 0.0, 1.0); Rc.call("residual", r0, T, U, Rr, 0.0, 1.0)
        assert_level_equal(H, R, 0, T, "in", f"{key} residual")
        norm, ref_norm = L.norm(l0, T), Rc.call("norm", r0, T)
        assert R is None or norm == ref_norm
        ob.pin(f"{key} norm", norm, ref_norm)
        L.restriction(l1, Rr, l0, T, api.RESTRICT_CELL); Rc.call("restriction", r1, Rr, r0, T, api.RESTRICT_CELL)
        assert_level_equal(H, R, 1, Rr, "in", f"{key} restriction")
        L.interpolation_v2(l0, U, 1.0, l1, E); Rc.call("interpolation_v2", r0, U, 1.0, r1, E)
        assert_level_equal(H, R, 0, U, "in", f"{key} interpolation_v2")
        L.interpolation_v4(l0, T, 0.0, l1, E); Rc.call("interpolation_v4", r0, T, 0.0, r1, E)
        assert_level_equal(H, R, 0, T, "in", f"{key} interpolation_v4")


def test_overwritten_diagonal_is_read_not_recomputed(gpu_lib):
    """The TMA GSRB kernel forms Dinv = 1/Aii in registers only while VECTOR_DINV is known to come from
    rebuild_operator_blackbox: once ANY operator of the API writes vector 5 the kernel must read it again."""
    L = gpu_lib
    U, Rr, DINV, E = api.VECTOR_U, api.VECTOR_R, api.VECTOR_DINV, api.VECTOR_E
    for writer in ("scale", "mul", "add", "restriction"):
        with api.Hierarchy(6, 1, use_graphs=False) as H:             # one 64^3 box: the TMA kernel, tiles away from the boundary
            R = reference(6, 1)
            rng = np.random.default_rng(11)
            mirror_random(H, R, rng, (0, 1), (U, Rr, E))
            lv, rl = (1, 1) if writer == "restriction" else (0, 0)
            Rc = R or ob.NoReference()
            l, r = H.level(lv), Rc.level(rl)
            if writer == "scale":
                L.scale_vector(l, DINV, 0.5, DINV); Rc.call("scale_vector", r, DINV, 0.5, DINV)
            elif writer == "mul":
                L.mul_vectors(l, DINV, 1.25, DINV, DINV); Rc.call("mul_vectors", r, DINV, 1.25, DINV, DINV)
            elif writer == "add":
                L.add_vectors(l, DINV, 0.75, DINV, 0.0, E); Rc.call("add_vectors", r, DINV, 0.75, DINV, 0.0, E)
            else:                                                    # level 1 (32^3): Dinv <- restriction of the fine Dinv
                L.restriction(l, DINV, H.level(0), DINV, api.RESTRICT_CELL); Rc.call("restriction", r, DINV, Rc.level(0), DINV, api.RESTRICT_CELL)
            L.smooth(l, U, Rr, 0.0, 1.0); Rc.call("smooth", r, U, Rr, 0.0, 1.0)
            assert_level_equal(H, R, lv, U, "in", f"smooth after {writer} wrote Dinv")


def test_recorded_solves_survive_reallocation_and_rebuild(gpu_lib):
    """FMGSolve -> MGPCG (create_vectors on every level moves the slabs) -> FMGSolve -> rebuild_operator -> MGSolve ->
    FMGSolve on ONE hierarchy: recorded graphs must not outlive what they captured."""
    g = ob.goldens()["solves"]["5 8 gsrb"]
    U, F = api.VECTOR_U, api.VECTOR_F
    with api.Hierarchy(5, 8) as H:
        assert H.fmg_solve(0)[0] == g["norms"][0]
        gpu_lib.MGPCG(H.mg, 0, U, F, 0.0, 1.0, 1e-10)
        pcg = api.download(H.level(0), 3, U).copy()
        assert H.fmg_solve(0)[0] == g["norms"][0]
        for l in range(1, H.num_levels):
            gpu_lib.rebuild_operator(H.level(l), H.level(l - 1), 0.0, 1.0)
        gpu_lib.zero_vector(H.level(0), U)
        gpu_lib.MGSolve(H.mg, 0, U, F, 0.0, 1.0, 1e-10)
        assert H.fmg_solve(0)[0] == g["norms"][0]
        gpu_lib.MGPCG(H.mg, 0, U, F, 0.0, 1.0, 1e-10)
        np.testing.assert_array_equal(pcg, api.download(H.level(0), 3, U))
        bottom = H.level(H.num_levels - 1).contents
        assert bottom.Krylov_iterations > 0


def test_last_norms_are_kept_per_hierarchy(gpu_lib):
    ga, gb = ob.goldens()["solves"]["4 8 gsrb"], ob.goldens()["solves"]["5 1 gsrb"]
    with api.Hierarchy(4, 8) as A, api.Hierarchy(5, 1) as B:
        A.fmg_solve(0)
        B.fmg_solve(0)
        assert gpu_lib.hpgmg_last_norm_of_residual(A.mg) == ga["norms"][0]
        assert gpu_lib.hpgmg_last_norm_of_residual(B.mg) == gb["norms"][0]
        assert gpu_lib.hpgmg_last_norm_of_F(A.mg) == ga["norm_of_F"] and gpu_lib.hpgmg_last_norm_of_F(B.mg) == gb["norm_of_F"]


def test_multibox_bottom_level_solves_without_recording(gpu_lib):
    """MGBuild(minCoarseGridDim=16) on `4 8` stops at a 16^3 bottom level of 8 boxes: the bottom solve is the
    host-driven BiCGStab (dots and norms read back every iteration), which must not be stream-captured."""
    U, F = api.VECTOR_U, api.VECTOR_F
    H = api.Hierarchy(4, 8, build_operator=False, use_graphs=True)
    R = reference(4, 8, build_operator=False)
    try:
        gpu_lib.initialize_problem(H.level_h, H.h, 0.0, 1.0)
        gpu_lib.rebuild_operator(H.level_h, None, 0.0, 1.0)
        gpu_lib.MGBuild(H.mg, H.level_h, 0.0, 1.0, 16)
        H.built = True
        assert H.num_levels == 2
        if R is not None:
            with ob.quiet():
                R.L.initialize_problem(R.level_h, R.h, 0.0, 1.0)
                R.L.rebuild_operator(R.level_h, None, 0.0, 1.0)
                R.L.MGBuild(R.mg, R.level_h, 0.0, 1.0, 16)
            R.built = True
            assert R.num_levels == 2
            with ob.ref_threads(1):              # the reference's dots are sums over tiles: order defined on one thread
                R.call("zero_vector", R.level(0), U)
                R.call("FMGSolve", R.mg, 0, U, F, 0.0, 1.0, 1e-10)
        for _ in range(2):                       # twice: a recorded graph would be replayed the second time
            gpu_lib.zero_vector(H.level(0), U)
            gpu_lib.FMGSolve(H.mg, 0, U, F, 0.0, 1.0, 1e-10)
            gpu_lib.hpgmg_b200_sync()
            assert_level_equal(H, R, 0, U, "in", "FMGSolve with a multi-box bottom level")
    finally:
        H.close()


def test_chebyshev_smoother_equals_reference(gpu_lib):
    with api.Hierarchy(4, 8, smoother=api.SMOOTHER_CHEBY, use_graphs=False) as H:
        R = reference(4, 8, cheby=True)
        rng = np.random.default_rng(7)
        mirror_random(H, R, rng, (0,), (api.VECTOR_U, api.VECTOR_R, api.VECTOR_TEMP))
        eig = H.level(0).contents.dominant_eigenvalue_of_DinvA
        ref_eig = R.level(0).contents.dominant_eigenvalue_of_DinvA if R else None
        assert R is None or eig == ref_eig
        ob.pin("chebyshev eig", eig, ref_eig)
        gpu_lib.smooth(H.level(0), api.VECTOR_U, api.VECTOR_R, 0.0, 1.0)
        if R is not None:
            R.call("smooth", R.level(0), api.VECTOR_U, api.VECTOR_R, 0.0, 1.0)
        assert_level_equal(H, R, 0, api.VECTOR_U, "in", "chebyshev")
        assert_level_equal(H, R, 0, api.VECTOR_TEMP, "in", "chebyshev")
    gpu_lib.hpgmg_b200_set_smoother(api.SMOOTHER_GSRB)


# ------------------------------------------------------------------------------ against the C oracle
def test_setup_and_solution_equal_oracle_cell_by_cell(gpu_lib):
    """One 32^3 box: Dinv, betas (with first ghost layer), and U/R of every level after an F-cycle."""
    O = ob.oracle()
    Ho = O.oracle_build(5, 0)
    nF = C.c_double()
    r_or = O.oracle_fmg_solve(Ho, 0, C.byref(nF))
    with api.Hierarchy(5, 1) as H:
        r, rel = H.fmg_solve(0)
        assert r == r_or and rel == pytest.approx(r_or / nF.value, rel=1e-15)
        for l in range(H.num_levels):
            n = H.level(l).contents.box_dim
            inner, ring = slice(2, 2 + n), slice(1, 3 + n)
            for vid in (api.VECTOR_DINV, api.VECTOR_U, api.VECTOR_R):
                np.testing.assert_array_equal(api.download(H.level(l), 0, vid)[inner, inner, inner], ob.oracle_array(Ho, l, vid)[inner, inner, inner])
            for vid in (api.VECTOR_BETA_I, api.VECTOR_BETA_J, api.VECTOR_BETA_K):
                np.testing.assert_array_equal(api.download(H.level(l), 0, vid)[ring, ring, ring], ob.oracle_array(Ho, l, vid)[ring, ring, ring])
    O.oracle_destroy(Ho)


# ------------------------------------------------------------------- size-independent properties, 7 8
@pytest.fixture(scope="module")
def big(gpu_lib):
    H = api.Hierarchy(7, 8)
    yield H
    H.close()


def test_full_size_goldens_and_determinism(gpu_lib, big):
    g = ob.goldens()["solves"]["7 8 gsrb"]
    a = big.fmg_solve(0)
    b = big.fmg_solve(0)
    assert a == b
    assert a[0] == g["norms"][0] == 5.144230117437587e-07
    # the printed residual really is ||f - A u|| of the returned u
    gpu_lib.residual(big.level(0), api.VECTOR_TEMP, api.VECTOR_U, api.VECTOR_F, 0.0, 1.0)
    assert gpu_lib.norm(big.level(0), api.VECTOR_TEMP) == a[0]


def test_full_size_zero_rhs_gives_zero_solution(gpu_lib, big):
    lvl = big.level(0)
    gpu_lib.scale_vector(lvl, api.VECTOR_E, 1.0, api.VECTOR_F)            # park F
    gpu_lib.zero_vector(lvl, api.VECTOR_F)
    gpu_lib.zero_vector(lvl, api.VECTOR_U)
    gpu_lib.hpgmg_b200_use_graphs(0)
    gpu_lib.FMGSolve(big.mg, 0, api.VECTOR_U, api.VECTOR_F, 0.0, 1.0, 1e-10)
    gpu_lib.hpgmg_b200_use_graphs(1)
    assert gpu_lib.norm(lvl, api.VECTOR_U) == 0.0
    gpu_lib.scale_vector(lvl, api.VECTOR_F, 1.0, api.VECTOR_E)
    gpu_lib.exchange_boundary(lvl, api.VECTOR_F, 0)


def test_full_size_ghost_fill_is_idempotent_and_linear(gpu_lib, big):
    lvl = big.level(0)
    big.fmg_solve(0)
    gpu_lib.exchange_boundary(lvl, api.VECTOR_U, 2); gpu_lib.apply_BCs(lvl, api.VECTOR_U, 2)
    first = api.download(lvl, 5, api.VECTOR_U).copy()
    gpu_lib.exchange_boundary(lvl, api.VECTOR_U, 2); gpu_lib.apply_BCs(lvl, api.VECTOR_U, 2)
    np.testing.assert_array_equal(first, api.download(lvl, 5, api.VECTOR_U))
    # homogeneous BCs and the operator are linear: A(2u) == 2 A(u) exactly (power-of-two scaling)
    gpu_lib.apply_op(lvl, api.VECTOR_TEMP, api.VECTOR_U, 0.0, 1.0)
    Au = api.download(lvl, 2, api.VECTOR_TEMP).copy()
    gpu_lib.scale_vector(lvl, api.VECTOR_E, 2.0, api.VECTOR_U)
    gpu_lib.apply_op(lvl, api.VECTOR_TEMP, api.VECTOR_E, 0.0, 1.0)
    n = lvl.contents.box_dim
    s = slice(2, 2 + n)
    np.testing.assert_array_equal(2.0 * Au[s, s, s], api.download(lvl, 2, api.VECTOR_TEMP)[s, s, s])
    assert gpu_lib.norm(lvl, api.VECTOR_E) == 2.0 * gpu_lib.norm(lvl, api.VECTOR_U)


def test_full_size_restriction_preserves_constants_and_means(gpu_lib, big):
    l0, l1 = big.level(0), big.level(1)
    gpu_lib.init_vector(l0, api.VECTOR_E, 1.5)
    gpu_lib.restriction(l1, api.VECTOR_E, l0, api.VECTOR_E, api.RESTRICT_CELL)
    n = l1.contents.box_dim
    s = slice(2, 2 + n)
    for b in range(l1.contents.num_my_boxes):
        assert np.all(api.download(l1, b, api.VECTOR_E)[s, s, s] == 1.5)
    # cell-averaged restriction conserves the mean (up to summation rounding)
    gpu_lib.restriction(l1, api.VECTOR_E, l0, api.VECTOR_F, api.RESTRICT_CELL)
    assert gpu_lib.mean(l1, api.VECTOR_E) == pytest.approx(gpu_lib.mean(l0, api.VECTOR_F), rel=1e-9, abs=1e-16)


# --------------------------------------------------------------------------------- drop-in, literally
def test_unmodified_reference_driver_runs_on_our_library(gpu_lib):
    """hpgmg_b200/bin/hpgmg-fv-refdriver = the reference's own hpgmg-fv.c (compiled with the reference's own
    headers) linked against libhpgmg_b200.so.  Its printed F-cycle norms / error must be the goldens."""
    import os, re, subprocess
    exe = os.path.join(os.path.dirname(api.LIB_PATH), "..", "bin", "hpgmg-fv-refdriver")
    if not os.path.exists(exe):
        pytest.skip("hpgmg-fv-refdriver not built (needs /root/reference at build time)")
    out = subprocess.run([exe, "6", "1"], capture_output=True, text=True, timeout=600).stdout
    g = ob.goldens()["solves"]["6 1 gsrb"]
    norms = [float(x) for x in re.findall(r"f-cycle\s+norm=([0-9.e+-]+)", out)]
    assert norms[-3:] == pytest.approx(g["norms"], rel=1e-15), out[-2000:]      # printed with %1.15e
    assert float(re.search(r"\|\|error\|\|=([0-9.e+-]+)", out).group(1)) == pytest.approx(g["error"], rel=1e-15)
    assert "DOF/s=" in out


# ----------------------------------------------------------------------------------------- multi-GPU
def _gpu_count():
    import subprocess
    try:
        return len([l for l in subprocess.run(["nvidia-smi", "-L"], capture_output=True, text=True).stdout.splitlines() if l.startswith("GPU ")])
    except Exception:
        return 0


@pytest.mark.parametrize("ranks", [2, 4, 8])
def test_multi_gpu_fmg_equals_single_process_reference(gpu_lib, ranks):
    """One process per GPU under torchrun: NVLink peer ghost exchange (LL protocol) + NCCL transfers.  The
    N-rank solve must reproduce, bit for bit, the goldens of the reference run with N x the boxes
    (5 16 -> 2^3 boxes, 5 32 -> 3^3 boxes with shrinking rank counts, 5 64 -> 4^3 boxes)."""
    import os, subprocess, sys
    if _gpu_count() < ranks:
        pytest.skip(f"needs {ranks} GPUs")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={ranks}", "--master-addr", "127.0.0.1",
           "--master-port", str(29600 + ranks), os.path.join(root, "tools", "check_multigpu.py"), "5", "8", "cells"]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert "PARITY OK (bit-exact)" in r.stdout, r.stdout[-2000:] + r.stderr[-2000:]
    if ob.have_ref():                          # and u itself, every cell of every box on every rank
        assert "cell by cell: u of every box on every rank equals" in r.stdout, r.stdout[-2000:]


# ------------------------------------------------------------------------- the other solve drivers of mg.c
@pytest.mark.parametrize("driver", ["MGSolve", "FMGSolve2", "MGPCG"])
def test_other_solve_drivers_equal_reference(gpu_lib, driver):
    """MGSolve (V-cycles to rtol, mg.c:1168-1233), FMGSolve2 (mg.c:1348-1495) and MGPCG (mg.c:1500-1607) are part of the
    API surface of the path (SURVEY.md 8a20): same solution as the reference library, cell by cell.  The reference
    runs on one OpenMP thread: MGPCG's dots are sums over tiles whose order is only defined there."""
    with api.Hierarchy(5, 8, verbose=False) as H:
        R = reference(5, 8)
        if R is not None:
            with ob.ref_threads(1):
                R.call("zero_vector", R.level(0), api.VECTOR_U)
                R.call(driver, R.mg, 0, api.VECTOR_U, api.VECTOR_F, 0.0, 1.0, 1e-10)
        gpu_lib.zero_vector(H.level(0), api.VECTOR_U)
        getattr(gpu_lib, driver)(H.mg, 0, api.VECTOR_U, api.VECTOR_F, 0.0, 1.0, 1e-10)
        gpu_lib.hpgmg_b200_sync()
        assert_level_equal(H, R, 0, api.VECTOR_U, "in", driver)


def test_operator_timers_fill_the_reference_table(gpu_lib, capfd):
    """hpgmg_b200_profile_operators(1): every operator adds its time to level->timers.* like the reference's getTime()
    brackets, so MGPrintTiming prints the reference's table; the solve itself must not change."""
    g = ob.goldens()["solves"]["5 8 gsrb"]
    with api.Hierarchy(5, 8, verbose=False) as H:
        gpu_lib.hpgmg_b200_profile_operators(1)
        try:
            gpu_lib.MGResetTimers(H.mg)
            r, _ = H.fmg_solve(0)
            t = H.level(0).contents.timers
            assert r == g["norms"][0]
            assert t.smooth > 0.0 and t.residual > 0.0 and t.restriction_total > 0.0 and t.interpolation_total > 0.0 and t.ghostZone_total > 0.0
            gpu_lib.MGPrintTiming(H.mg, 0)
        finally:
            gpu_lib.hpgmg_b200_profile_operators(0)
    C.CDLL(None).fflush(None)
    out = capfd.readouterr().out
    assert "smooth" in out and "residual" in out and "Total by level" in out


# ------------------------------------------------------------------------- kernel variants behind switches
VARIANTS = [
    {"HPGMG_B200_TMA_BLOCKS": "37"},                              # uneven split: blocks own several partial columns
    {"HPGMG_B200_TMA_BLOCKS": "301", "HPGMG_B200_ZIGZAG": "0"},
    {"HPGMG_B200_DIAG": "0"},                                     # Dinv always from memory
    {"HPGMG_B200_TMA": "0"},                                      # boxes >= 32^3 through the pair kernel
    {"HPGMG_B200_GENERIC_STENCIL": "1"},                          # one thread per cell everywhere
    {"HPGMG_B200_PAIR_KERNEL": "0"},                              # small boxes through the generic kernel
    {"HPGMG_B200_NO_COARSE_KERNEL": "1"},
    {"HPGMG_B200_COARSE_FAST": "0"},                              # coarse kernel: generic bodies instead of the size-specialised ones
    {"HPGMG_B200_BOX_FUSED_MAX": "0"},                            # small boxes: separate ghost-fill kernel + operator kernel
    {"HPGMG_B200_BOX_FUSED_MAX": "32"},                           # fill-fused box kernel also on 32^3 boxes (instead of the TMA kernel)
    {"HPGMG_B200_FUSE_RESTRICT": "0"},                            # residual and restriction as two kernels in MGVCycle
    {"HPGMG_B200_FUSE_NORM": "0"},                                # norm as a separate kernel after residual / R=F
    {"HPGMG_B200_INTERP_MARCH": "0"},                             # tiled interpolation on every level
    {"HPGMG_B200_INTERP_MARCH": "64"},                            # k-marching interpolation down to 16^3 boxes
]


@pytest.mark.parametrize("env", VARIANTS, ids=lambda e: ",".join(f"{k[11:]}={v}" for k, v in e.items()))
def test_kernel_variants_give_the_same_bits(gpu_lib, env):
    """Every alternative kernel / schedule kept in the tree behind an environment switch (DESIGN.md section 4)
    must reproduce the reference goldens of `hpgmg-fv 6 8` (64^3 and 32^3 boxes: the TMA kernel on two levels)."""
    import os, subprocess, sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    e = dict(os.environ)
    e.update(env)
    e.pop("RANK", None); e.pop("WORLD_SIZE", None)
    r = subprocess.run([sys.executable, os.path.join(root, "tools", "check_multigpu.py"), "6", "8"], capture_output=True, text=True, timeout=300, env=e)
    assert "PARITY OK (bit-exact)" in r.stdout, r.stdout[-2000:] + r.stderr[-2000:]
