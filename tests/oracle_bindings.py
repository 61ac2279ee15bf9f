"""Test-side bindings of the two checkers (TEST INFRASTRUCTURE, never imported by hpgmg_b200/):

* the plain-C oracle restatement  oracle/hpgmg_oracle.c -> oracle/_build/libhpgmg_oracle.so
* the UNMODIFIED reference        /root/reference/finite-volume/source -> oracle/_ref/libhpgmg_ref[_cheby].so
  (built here by oracle/Makefile; travels to the GPU box as a prebuilt file; may be absent elsewhere)
"""
import contextlib
import ctypes as C
import functools
import hashlib
import json
import os
import subprocess
import sys
import zlib

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
import hpgmg_b200.api as api  # noqa: E402
from hpgmg_b200._structs import level_type, mg_type  # noqa: E402

ORACLE_SO = os.path.join(ROOT, "oracle", "_build", "libhpgmg_oracle.so")
REF_DIR = os.path.join(ROOT, "oracle", "_ref")
GOLDEN = os.path.join(ROOT, "tests", "golden", "goldens.json")


@functools.lru_cache(None)
def goldens():
    with open(GOLDEN) as f:
        return json.load(f)


# ---------------------------------------------------------------------------------------------- pins
# The reference library is built only where its sources are present.  What a reference comparison compares against is
# also stored in tests/golden/pins.json, recorded from the reference itself, so that the comparison holds on a machine
# without the reference too.  HPGMG_B200_RECORD_PINS=<file> records the reference's values into <file>; recording
# refuses to run without the reference build.
PINS = os.path.join(ROOT, "tests", "golden", "pins.json")
PIN_SAMPLES = 8                 # values stored beside an array's hash, at evenly spaced positions, for the failure message
_recorded = {}


@functools.lru_cache(None)
def pins():
    with open(PINS) as f:
        return json.load(f)


def seed(*parts):
    """A seed for np.random.default_rng that is the same in every process (hash() of a str is not)."""
    return zlib.crc32(" ".join(map(str, parts)).encode())


def fingerprint(value):
    """Exact fingerprint: a float as float.hex, an int as itself, a str as its sha1; an array or a list of arrays as a sha1
    of their float64 bytes, their size and PIN_SAMPLES of their values."""
    if isinstance(value, (int, np.integer)) and not isinstance(value, bool):
        return int(value)
    if isinstance(value, (float, np.floating)):
        return float(value).hex()
    h = hashlib.sha1()
    if isinstance(value, str):
        h.update(value.encode())
        return h.hexdigest()[:24]
    flat = np.concatenate([np.ascontiguousarray(a, dtype=np.float64).reshape(-1) for a in (value if isinstance(value, list) else [value])])
    h.update(flat.tobytes())
    at = np.linspace(0, flat.size - 1, min(PIN_SAMPLES, flat.size)).astype(np.int64) if flat.size else []
    return {"sha1": h.hexdigest()[:24], "size": int(flat.size), "sample": {str(int(i)): float(flat[i]).hex() for i in at}}


def _mismatch(fp, want):
    if not isinstance(want, dict) or not isinstance(fp, dict):
        return f"{fp!r} differs from the reference's {want!r}"
    if fp["size"] != want["size"]:
        return f"{fp['size']} values, the reference has {want['size']}"
    diffs = {i: (float.fromhex(fp["sample"][i]), float.fromhex(v)) for i, v in want["sample"].items() if fp["sample"][i] != v}
    return (f"cells differ from the reference's (hash {fp['sha1']} vs {want['sha1']}); at the sampled positions "
            + (", ".join(f"[{i}] {a!r} vs {b!r}" for i, (a, b) in diffs.items()) if diffs else "all values agree"))


def pin(key, ours, theirs):
    """Assert that ours equals the reference's value stored under key.  theirs is the reference's value computed in this
    process, or None where the reference is not built; recording stores theirs."""
    out = os.environ.get("HPGMG_B200_RECORD_PINS")
    if out:
        assert theirs is not None, f"{key}: HPGMG_B200_RECORD_PINS records the reference's values; build it first (make -C oracle ref)"
        _recorded[key] = fingerprint(theirs)
        with open(out, "w") as f:
            json.dump(_recorded, f, indent=0, sort_keys=True)
        return                  # the test itself compares ours with theirs
    stored = pins()
    assert key in stored, f"{key}: nothing recorded in tests/golden/pins.json"
    fp = fingerprint(ours)
    assert fp == stored[key], f"{key}: {_mismatch(fp, stored[key])}"


class NoReference:
    """Stands in for the reference's hierarchy or library where the reference is not built: every call does nothing and
    returns None, so that a test runs its own side and checks it against the pins alone."""
    mg = None

    def level(self, l):
        return None

    def __getattr__(self, name):
        return lambda *args: None


# ---------------------------------------------------------------------------------------------- oracle
@functools.lru_cache(None)
def oracle():
    if not os.path.exists(ORACLE_SO):
        subprocess.run(["make", "oracle"], cwd=os.path.join(ROOT, "oracle"), check=True, capture_output=True)
    L = C.CDLL(ORACLE_SO)
    vp, i, d = C.c_void_p, C.c_int, C.c_double
    sig = {"oracle_build": (vp, [i, i]), "oracle_destroy": (None, [vp]),
           "oracle_fmg_solve": (d, [vp, i, C.POINTER(d)]),
           "oracle_richardson": (None, [vp, C.POINTER(d), C.POINTER(d), C.POINTER(d)]),
           "oracle_vector": (C.POINTER(d), [vp, i, i]), "oracle_level": (vp, [vp, i]),
           "oracle_level_dim": (i, [vp, i]), "oracle_level_jstride": (i, [vp, i]), "oracle_level_volume": (i, [vp, i]),
           "oracle_level_eig": (d, [vp, i]), "oracle_num_levels": (i, [vp]), "oracle_krylov_iterations": (i, [vp]),
           "oracle_apply_BCs_v2": (None, [vp, i, i]), "oracle_apply_BCs_v4": (None, [vp, i, i]),
           "oracle_apply_op": (None, [vp, i, i, d]), "oracle_residual": (None, [vp, i, i, i, d]),
           "oracle_smooth_gsrb": (None, [vp, i, i, d]), "oracle_smooth_cheby": (None, [vp, i, i, d]),
           "oracle_restriction": (None, [vp, i, vp, i, i]),
           "oracle_interpolation_v2": (None, [vp, i, d, vp, i]), "oracle_interpolation_v4": (None, [vp, i, d, vp, i]),
           "oracle_norm": (d, [vp, i]), "oracle_extrapolate_betas": (None, [vp])}
    for name, (res, args) in sig.items():
        fn = getattr(L, name)
        fn.restype, fn.argtypes = res, args
    return L


def oracle_array(H, level, vec_id):
    """View of an oracle vector as [k][j][i] (ghosts + padding included); writes go through."""
    O = oracle()
    n, jS, vol = O.oracle_level_dim(H, level), O.oracle_level_jstride(H, level), O.oracle_level_volume(H, level)
    flat = np.ctypeslib.as_array(O.oracle_vector(H, level, vec_id), shape=(vol,))
    return flat.reshape(n + 4, n + 4, jS)


@functools.lru_cache(None)
def oracle_fmg_norms(log2_dim, cheby=False):
    """(||r|| on levels 0,1,2), richardson error, order, [eig per level], krylov its -- from the oracle."""
    O = oracle()
    H = O.oracle_build(log2_dim, 1 if cheby else 0)
    norms = (C.c_double * 3)()
    err, order = C.c_double(), C.c_double()
    O.oracle_richardson(H, norms, C.byref(err), C.byref(order))
    eigs = [O.oracle_level_eig(H, l) for l in range(O.oracle_num_levels(H))]
    out = (list(norms), err.value, order.value, eigs, O.oracle_krylov_iterations(H))
    O.oracle_destroy(H)
    return out


# ------------------------------------------------------------------------------------------- reference
def have_ref(cheby=False):
    return os.path.exists(os.path.join(REF_DIR, "libhpgmg_ref_cheby.so" if cheby else "libhpgmg_ref.so"))


_REF_SYMBOLS = ["create_level", "destroy_level", "create_vectors", "reset_level_timers",
                "stencil_get_radius", "stencil_get_shape", "apply_op", "residual", "smooth", "rebuild_operator",
                "rebuild_operator_blackbox", "restriction", "interpolation_vcycle", "interpolation_fcycle",
                "interpolation_v2", "interpolation_v4", "exchange_boundary", "apply_BCs", "apply_BCs_v1", "apply_BCs_v2",
                "apply_BCs_v4", "extrapolate_betas", "dot", "norm", "mean", "error", "add_vectors", "scale_vector",
                "zero_vector", "shift_vector", "mul_vectors", "invert_vector", "init_vector", "color_vector",
                "random_vector", "initialize_problem", "evaluateBeta", "evaluateF", "MGBuild", "MGSolve", "FMGSolve", "FMGSolve2", "MGPCG",
                "MGVCycle", "MGDestroy", "MGResetTimers", "richardson_error", "IterativeSolver", "IterativeSolver_NumVectors"]


@functools.lru_cache(None)
def ref(cheby=False):
    """The reference compiled as a shared library, bound with the same signatures as ours."""
    path = os.path.join(REF_DIR, "libhpgmg_ref_cheby.so" if cheby else "libhpgmg_ref.so")
    L = C.CDLL(path)           # RTLD_LOCAL: its symbols (smooth, norm, ...) must not clash with ours
    if hasattr(L, "create_level"):
        return api.bind(L, {k: api.SIGNATURES[k] for k in _REF_SYMBOLS})
    return _bind_by_symbol_table(L, path)


def _bind_by_symbol_table(L, path):
    """A reference build that does not export its functions (its hpgmg-fv executable, made loadable by clearing the PIE
    flag of its dynamic section): the functions at the load address plus their symbol-table values."""
    value = {}
    for line in subprocess.run(["nm", "--defined-only", path], capture_output=True, text=True, check=True).stdout.splitlines():
        f = line.split()
        if len(f) == 3 and f[1] in "Tt":
            value[f[2]] = int(f[0], 16)
    link_map = C.c_void_p()
    assert C.CDLL(None).dlinfo(C.c_void_p(L._handle), 2, C.byref(link_map)) == 0       # RTLD_DI_LINKMAP
    base = C.cast(link_map, C.POINTER(C.c_size_t))[0]                                   # link_map.l_addr

    class Functions:
        pass
    out = Functions()
    for k in _REF_SYMBOLS:
        res, args = api.SIGNATURES[k]
        setattr(out, k, C.CFUNCTYPE(res, *args)(base + value[k]))
    out._keep = L
    return out


@contextlib.contextmanager
def ref_threads(n):
    """Run the reference on n OpenMP threads (its sums over tiles and its two-layer linear BCs are only
    order-defined on one thread)."""
    gomp = C.CDLL("libgomp.so.1")
    gomp.omp_get_max_threads.restype = C.c_int
    before = gomp.omp_get_max_threads()
    gomp.omp_set_num_threads(int(n))
    try:
        yield
    finally:
        gomp.omp_set_num_threads(before)


@contextlib.contextmanager
def quiet():
    """The reference printf()s its progress: park fd 1 on /dev/null while it runs."""
    sys.stdout.flush()
    saved = os.dup(1)
    devnull = os.open(os.devnull, os.O_WRONLY)
    os.dup2(devnull, 1)
    try:
        yield
    finally:
        C.CDLL(None).fflush(None)
        os.dup2(saved, 1)
        os.close(saved)
        os.close(devnull)


class RefHierarchy:
    """hpgmg-fv.c:280-308 executed by the reference library on host memory."""

    def __init__(self, log2_box_dim, target_boxes_per_rank, my_rank=0, num_ranks=1, cheby=False, build_operator=True,
                 bc=api.BC_DIRICHLET, library=None, a=0.0, b=1.0, vectors=None):
        self.L = library or ref(cheby)
        self.a, self.b = float(a), float(b)
        self.box_dim, self.boxes_in_i = api.problem_size(log2_box_dim, target_boxes_per_rank, num_ranks)
        self._level_buf = level_type()
        self.level_h = C.pointer(self._level_buf)
        self._mg_buf = mg_type()
        self.mg = C.pointer(self._mg_buf)
        self.built = False
        with quiet():
            self.L.create_level(self.level_h, self.boxes_in_i, self.box_dim, 2, api.VECTORS_RESERVED if vectors is None else vectors, bc, my_rank, num_ranks)
            self.h = 1.0 / (float(self.boxes_in_i) * float(self.box_dim))
            if build_operator:
                self.L.initialize_problem(self.level_h, self.h, self.a, self.b)
                self.L.rebuild_operator(self.level_h, None, self.a, self.b)
                if bc == api.BC_PERIODIC:              # hpgmg-fv.c:296-302
                    average = self.L.mean(self.level_h, api.VECTOR_F)
                    if average != 0.0:
                        self.L.shift_vector(self.level_h, api.VECTOR_F, api.VECTOR_F, -average)
                self.L.MGBuild(self.mg, self.level_h, self.a, self.b, 2 if bc == api.BC_PERIODIC else 1)
                self.built = True

    def build_lists_only(self):
        """MGBuild on an uninitialised problem: only the inter-level lists are meaningful."""
        with quiet():
            self.L.MGBuild(self.mg, self.level_h, self.a, self.b, 1)
        self.built = True

    @property
    def num_levels(self):
        return self._mg_buf.num_levels

    def level(self, l):
        return self._mg_buf.levels[l] if self.built else self.level_h

    def array(self, l, box, vec_id):
        """Live view [k][j][i] of a box vector in the reference's host memory."""
        Lv = self.level(l).contents
        ptr = Lv.my_boxes[box].vectors[vec_id]
        flat = np.ctypeslib.as_array((C.c_double * Lv.box_volume).from_address(ptr))
        n = Lv.box_dim + 2 * Lv.box_ghosts
        return flat.reshape(n, n, Lv.box_jStride)

    def fmg_solve(self, on_level=0):
        with quiet():
            self.L.zero_vector(self.level(on_level), api.VECTOR_U)
            self.L.FMGSolve(self.mg, on_level, api.VECTOR_U, api.VECTOR_F, self.a, self.b, 1e-10)
            self.L.residual(self.level(on_level), api.VECTOR_TEMP, api.VECTOR_U, api.VECTOR_F, self.a, self.b)
            return self.L.norm(self.level(on_level), api.VECTOR_TEMP)

    def call(self, name, *args):
        with quiet():
            return getattr(self.L, name)(*args)


# ----------------------------------------------------------------------------------------------- lists
def list_digest(ptr, n):
    """sha1 over the index content of a blockCopy_type list (pointers reduced to 'buffer or box')."""
    h = hashlib.sha1()
    for b in api.block_list(ptr, n):
        h.update(np.asarray(b, dtype=np.int64).tobytes())
    return h.hexdigest()[:16]


def level_list_summary(level):
    """Counts + digests of every block list of a level, in a fixed order, plus the neighbour tables."""
    Lv = level.contents
    out = {"dim": Lv.dim.i, "box_dim": Lv.box_dim, "boxes_in": Lv.boxes_in.i, "num_my_boxes": Lv.num_my_boxes,
           "num_ranks": Lv.num_ranks, "jStride": Lv.box_jStride, "kStride": Lv.box_kStride, "volume": Lv.box_volume,
           "tiles": [Lv.num_my_blocks, list_digest(Lv.my_blocks, Lv.num_my_blocks)],
           "rank_of_box": [Lv.rank_of_box[i] for i in range(Lv.boxes_in.i ** 3)]}
    out["bc"] = [[Lv.boundary_condition.num_blocks[s], list_digest(Lv.boundary_condition.blocks[s], Lv.boundary_condition.num_blocks[s])] for s in range(3)]

    def comm(c):
        return {"blocks": [[c.num_blocks[p], list_digest(c.blocks[p], c.num_blocks[p])] for p in range(3)],
                "send": [[c.send_ranks[n], c.send_sizes[n]] for n in range(c.num_sends)],
                "recv": [[c.recv_ranks[n], c.recv_sizes[n]] for n in range(c.num_recvs)]}
    out["exchange"] = [comm(Lv.exchange_ghosts[s]) for s in range(3)]
    out["restriction"] = [comm(Lv.restriction[t]) for t in range(4)]
    out["interpolation"] = comm(Lv.interpolation)
    return out
