"""Test-side binding of tests/oracle_fv2_helmholtz.c (TEST INFRASTRUCTURE, never imported by hpgmg_b200/): the plain-C
restatement of the library's fv2 Helmholtz flavour on one-box-per-level hierarchies.  The C file includes tests/oracle_fv2.c
unchanged; it is compiled once per process, with the oracle's flags, into a temporary directory.  It has not been diffed
against the reference's operators.fv2.c (not available): it restates the library's fv2 and Helmholtz code."""
import atexit
import ctypes as C
import functools
import os
import shutil
import subprocess
import tempfile

import numpy as np

from oracle_fv2 import BICGSTAB, CG, CHEBY, G, GSRB, JACOBI, L1JACOBI  # noqa: F401

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "oracle_fv2_helmholtz.c")
A, B = 1.0, 1.0                                     # hpgmg-fv.c:286-288


@functools.lru_cache(None)
def lib():
    d = tempfile.mkdtemp(prefix="oracle_fv2_helmholtz_")
    atexit.register(shutil.rmtree, d, True)
    so = os.path.join(d, "liboracle_fv2_helmholtz.so")
    subprocess.run(["gcc", "-O2", "-std=gnu11", "-Wall", "-Wno-unused-function", "-ffp-contract=off", "-shared", "-fPIC",
                    SRC, "-o", so, "-lm"], check=True, capture_output=True)
    L = C.CDLL(so)
    vp, i, d_ = C.c_void_p, C.c_int, C.c_double
    sig = {"fvh_build": (vp, [i, i, i, d_, d_]), "fv2_destroy": (None, [vp]), "fv2_hier": (vp, [vp]),
           "fvh_fmg_solve": (d_, [vp, i, C.POINTER(d_)]),
           "fvh_richardson": (None, [vp, C.POINTER(d_), C.POINTER(d_), C.POINTER(d_)]),
           "fvh_level_apply_op": (None, [vp, i, i, i]), "fvh_level_residual": (None, [vp, i, i, i, i]),
           "fvh_level_smooth": (None, [vp, i, i, i]), "fvh_alpha_id": (i, []), "fvh_l1_id": (i, []),
           "oracle_vector": (C.POINTER(d_), [vp, i, i]), "oracle_level_dim": (i, [vp, i]),
           "oracle_level_jstride": (i, [vp, i]), "oracle_level_volume": (i, [vp, i]), "oracle_level_eig": (d_, [vp, i]),
           "oracle_num_levels": (i, [vp]), "oracle_krylov_iterations": (i, [vp])}
    for name, (res, args) in sig.items():
        fn = getattr(L, name)
        fn.restype, fn.argtypes = res, args
    return L


class Hier:
    """`hpgmg-fv <log2> 1` with the fv2 Helmholtz operator: build, then solve / apply operators level by level."""

    def __init__(self, log2, smoother=GSRB, bottom=BICGSTAB, a=A, b=B):
        self.O = lib()
        self.F = self.O.fvh_build(log2, smoother, bottom, a, b)
        self.H = self.O.fv2_hier(self.F)
        self.ALPHA, self.L1 = self.O.fvh_alpha_id(), self.O.fvh_l1_id()

    def num_levels(self):
        return self.O.oracle_num_levels(self.H)

    def eig(self, level):
        return self.O.oracle_level_eig(self.H, level)

    def array(self, level, vec_id):
        """View of a vector as [k][j][i] (the oracle's 2 ghost layers + padding included); writes go through."""
        O, H = self.O, self.H
        n, jS, vol = O.oracle_level_dim(H, level), O.oracle_level_jstride(H, level), O.oracle_level_volume(H, level)
        return np.ctypeslib.as_array(O.oracle_vector(H, level, vec_id), shape=(vol,)).reshape(n + 2 * G, n + 2 * G, jS)

    def interior(self, level, vec_id):
        n = self.O.oracle_level_dim(self.H, level)
        return self.array(level, vec_id)[G:G + n, G:G + n, G:G + n].copy()

    def fmg_solve(self, on_level=0):
        nf = C.c_double()
        r = self.O.fvh_fmg_solve(self.F, on_level, C.byref(nf))
        return r, nf.value

    def krylov(self):
        return self.O.oracle_krylov_iterations(self.H)

    def close(self):
        if self.F:
            self.O.fv2_destroy(self.F)
            self.F = None

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()


def richardson(log2, smoother=GSRB, bottom=BICGSTAB, a=A, b=B):
    """The driver's three solves (hpgmg-fv.c:351-366) on `hpgmg-fv <log2> 1`: (norms on levels 0,1,2, error, order, Krylov
    iterations of the three solves)."""
    with Hier(log2, smoother, bottom, a, b) as h:
        norms = (C.c_double * 3)()
        err, order = C.c_double(), C.c_double()
        h.O.fvh_richardson(h.F, norms, C.byref(err), C.byref(order))
        return list(norms), err.value, order.value, h.krylov()
