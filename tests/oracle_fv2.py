"""Test-side binding of tests/oracle_fv2.c (TEST INFRASTRUCTURE, never imported by hpgmg_b200/): the plain-C restatement of
the library's fv2 flavour on one-box-per-level hierarchies.  The C file includes oracle/hpgmg_oracle.c unchanged; it is
compiled once per process, with the oracle's flags, into a temporary directory."""
import atexit
import ctypes as C
import functools
import os
import shutil
import subprocess
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "oracle_fv2.c")
GSRB, CHEBY, JACOBI, L1JACOBI = 0, 1, 2, 3          # = HPGMG_SMOOTHER_*
BICGSTAB, CG = 0, 1                                 # = HPGMG_BOTTOM_*
G = 2                                               # the oracle's ghost layout (only the first layer is used by fv2)


@functools.lru_cache(None)
def lib():
    d = tempfile.mkdtemp(prefix="oracle_fv2_")
    atexit.register(shutil.rmtree, d, True)
    so = os.path.join(d, "liboracle_fv2.so")
    subprocess.run(["gcc", "-O2", "-std=gnu11", "-Wall", "-Wno-unused-function", "-ffp-contract=off", "-shared", "-fPIC",
                    SRC, "-o", so, "-lm"], check=True, capture_output=True)
    L = C.CDLL(so)
    vp, i, d_ = C.c_void_p, C.c_int, C.c_double
    sig = {"fv2_build": (vp, [i, i, i]), "fv2_destroy": (None, [vp]), "fv2_hier": (vp, [vp]),
           "fv2_fmg_solve": (d_, [vp, i, C.POINTER(d_)]),
           "fv2_richardson": (None, [vp, C.POINTER(d_), C.POINTER(d_), C.POINTER(d_)]),
           "fv2_level_apply_op": (None, [vp, i, i, i]), "fv2_level_residual": (None, [vp, i, i, i, i]),
           "fv2_level_smooth": (None, [vp, i, i, i]), "fv2_level_interpolation_p0": (None, [vp, i, i, d_, i]),
           "oracle_vector": (C.POINTER(d_), [vp, i, i]), "oracle_level_dim": (i, [vp, i]),
           "oracle_level_jstride": (i, [vp, i]), "oracle_level_volume": (i, [vp, i]), "oracle_level_eig": (d_, [vp, i]),
           "oracle_num_levels": (i, [vp]), "oracle_krylov_iterations": (i, [vp])}
    for name, (res, args) in sig.items():
        fn = getattr(L, name)
        fn.restype, fn.argtypes = res, args
    return L


class Hier:
    """`hpgmg-fv <log2> 1` with the fv2 operator: build, then solve / apply operators level by level."""

    def __init__(self, log2, smoother=GSRB, bottom=BICGSTAB):
        self.O = lib()
        self.F = self.O.fv2_build(log2, smoother, bottom)
        self.H = self.O.fv2_hier(self.F)

    def num_levels(self):
        return self.O.oracle_num_levels(self.H)

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
        r = self.O.fv2_fmg_solve(self.F, on_level, C.byref(nf))
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


def richardson(log2, smoother=GSRB, bottom=BICGSTAB):
    """The driver's three solves (hpgmg-fv.c:351-366) on `hpgmg-fv <log2> 1`: (norms on levels 0,1,2, error, order, Krylov
    iterations of the three solves)."""
    with Hier(log2, smoother, bottom) as h:
        norms = (C.c_double * 3)()
        err, order = C.c_double(), C.c_double()
        h.O.fv2_richardson(h.F, norms, C.byref(err), C.byref(order))
        return list(norms), err.value, order.value, h.krylov()
