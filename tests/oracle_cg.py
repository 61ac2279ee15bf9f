"""Test-side binding of tests/oracle_cg.c (TEST INFRASTRUCTURE, never imported by hpgmg_b200/): the plain-C oracle with the
reference's D^-1-preconditioned CG bottom solver.  The C file includes oracle/hpgmg_oracle.c unchanged; it is compiled once per
process, with the oracle's flags, into a temporary directory."""
import atexit
import ctypes as C
import functools
import os
import shutil
import subprocess
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "oracle_cg.c")
GSRB, CHEBY = 0, 1                 # the smoother argument of oracle_build (ohier::cheby)


@functools.lru_cache(None)
def lib():
    d = tempfile.mkdtemp(prefix="oracle_cg_")
    atexit.register(shutil.rmtree, d, True)
    so = os.path.join(d, "liboracle_cg.so")
    subprocess.run(["gcc", "-O2", "-std=gnu11", "-Wall", "-Wno-unused-function", "-ffp-contract=off", "-shared", "-fPIC",
                    SRC, "-o", so, "-lm"], check=True, capture_output=True)
    L = C.CDLL(so)
    vp, i, d_ = C.c_void_p, C.c_int, C.c_double
    sig = {"oracle_build": (vp, [i, i]), "oracle_destroy": (None, [vp]),
           "oracle_cg": (i, [vp, i, i, i, d_]),
           "oracle_cg_fmg_solve": (d_, [vp, i, C.POINTER(d_)]),
           "oracle_cg_richardson": (None, [vp, C.POINTER(d_), C.POINTER(d_), C.POINTER(d_)]),
           "oracle_richardson": (None, [vp, C.POINTER(d_), C.POINTER(d_), C.POINTER(d_)]),
           "oracle_apply_op": (None, [vp, i, i, d_]), "oracle_residual": (None, [vp, i, i, i, d_]),
           "oracle_vector": (C.POINTER(d_), [vp, i, i]), "oracle_level": (vp, [vp, i]),
           "oracle_level_dim": (i, [vp, i]), "oracle_level_jstride": (i, [vp, i]), "oracle_level_volume": (i, [vp, i]),
           "oracle_num_levels": (i, [vp]), "oracle_krylov_iterations": (i, [vp])}
    for name, (res, args) in sig.items():
        fn = getattr(L, name)
        fn.restype, fn.argtypes = res, args
    return L


def array(H, level, vec_id):
    """View of a vector of the hierarchy as [k][j][i] (ghosts + padding included); writes go through."""
    O = lib()
    n, jS, vol = O.oracle_level_dim(H, level), O.oracle_level_jstride(H, level), O.oracle_level_volume(H, level)
    return np.ctypeslib.as_array(O.oracle_vector(H, level, vec_id), shape=(vol,)).reshape(n + 4, n + 4, jS)


def richardson(log2, smoother):
    """The driver's three solves (hpgmg-fv.c:351-366) on `hpgmg-fv <log2> 1` with the CG bottom solver: (norms on levels
    0,1,2, error, order, CG iterations of the three solves)."""
    O = lib()
    H = O.oracle_build(log2, smoother)
    norms = (C.c_double * 3)()
    err, order = C.c_double(), C.c_double()
    O.oracle_cg_richardson(H, norms, C.byref(err), C.byref(order))
    out = (list(norms), err.value, order.value, O.oracle_krylov_iterations(H))
    O.oracle_destroy(H)
    return out
