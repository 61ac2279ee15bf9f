"""Python host layer over the C-ABI of libhpgmg_b200.so (include/*.h).

It mirrors the reference's own C interface for the FMG path -- same names, same argument order
(finite-volume/source/level.h:204-215, operators.h:9-50, mg.h:37-45, solvers.h:9-10) -- so a test
written against the reference (`create_level`, `initialize_problem`, `rebuild_operator`, `MGBuild`,
`FMGSolve`, `richardson_error` ...) reads the same here.  Everything numerical happens in the
hand-written sm_100a kernels inside the shared library; this module only moves pointers.  If the
library has not been built (``python -c 'import __graft_entry__ as g; g.build()'``) or there is no
CUDA device, the calls fail loudly: there is no CPU fallback.
"""
import ctypes as C
import os

import numpy as np

from ._structs import (blockCopy_type, box_type, communicator_type, level_type, mg_type,  # noqa: F401
                       block_tuple, STENCIL_MAX_SHAPES)

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libhpgmg_b200.so")
# the 2nd-order operator (the reference linked with operators.fv2.c): one ghost layer, bind with bind(ctypes.CDLL(FV2_LIB_PATH))
# and pass it as Hierarchy(..., library=...)
FV2_LIB_PATH = os.path.join(_HERE, "lib", "libhpgmg_b200_fv2.so")
# the same with -DUSE_HELMHOLTZ (the reference's operators.fv2.c with -DUSE_HELMHOLTZ): a*alpha*u - b*div(beta grad u), the
# Helmholtz vector map (VECTOR_ALPHA 9, VECTOR_L1INV 10, VECTORS_RESERVED 11: pass vectors=11 to Hierarchy)
FV2_HELMHOLTZ_LIB_PATH = os.path.join(_HERE, "lib", "libhpgmg_b200_fv2_helmholtz.so")

# defines.h:28-38
VECTOR_TEMP, VECTOR_U, VECTOR_F, VECTOR_E, VECTOR_R, VECTOR_DINV, VECTOR_BETA_I, VECTOR_BETA_J, VECTOR_BETA_K = range(9)
VECTORS_RESERVED = 9
BC_PERIODIC, BC_DIRICHLET = 0, 1
STENCIL_SHAPE_BOX, STENCIL_SHAPE_STAR, STENCIL_SHAPE_NO_CORNERS = 0, 1, 2
RESTRICT_CELL, RESTRICT_FACE_I, RESTRICT_FACE_J, RESTRICT_FACE_K = 0, 1, 2, 3
SMOOTHER_GSRB, SMOOTHER_CHEBY, SMOOTHER_JACOBI, SMOOTHER_L1JACOBI = 0, 1, 2, 3    # include/hpgmg_b200.h
BOTTOM_BICGSTAB, BOTTOM_CG = 0, 1                                                 # include/hpgmg_b200.h

ALLGATHER_FN = C.CFUNCTYPE(None, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p)
BARRIER_FN = C.CFUNCTYPE(None, C.c_void_p)

_lib = None

_LP = C.POINTER(level_type)
_MP = C.POINTER(mg_type)
_D, _I, _V = C.c_double, C.c_int, None

# name -> (restype, argtypes): the whole exported surface (tests check every symbol resolves)
SIGNATURES = {
    # hpgmg_b200.h
    "hpgmg_b200_init": (_I, [_I]), "hpgmg_b200_finalize": (_V, []), "hpgmg_b200_sync": (_V, []),
    "hpgmg_b200_backend": (C.c_char_p, []), "hpgmg_b200_device": (_I, []),
    "hpgmg_b200_set_smoother": (_V, [_I]), "hpgmg_b200_get_smoother": (_I, []),
    "hpgmg_b200_set_bottom_solver": (_V, [_I]), "hpgmg_b200_get_bottom_solver": (_I, []),
    "hpgmg_b200_set_verbose": (_V, [_I]), "hpgmg_b200_use_graphs": (_V, [_I]),
    "hpgmg_b200_profile_operators": (_V, [_I]), "hpgmg_b200_use_coarse_kernel": (_V, [_I]), "hpgmg_b200_coarse_profile": (_V, [_I, C.c_void_p]), "hpgmg_b200_coarse_levels_in_smem": (_V, [_I]), "hpgmg_b200_set_layout_only": (_V, [_I]),
    "hpgmg_download_box_vector": (_V, [_LP, _I, _I, C.c_void_p]),
    "hpgmg_upload_box_vector": (_V, [_LP, _I, _I, C.c_void_p]),
    "hpgmg_download_l1inv": (_V, [_LP, _I, C.c_void_p]),
    "hpgmg_b200_host_alloc_pinned": (C.c_void_p, [C.c_size_t]), "hpgmg_b200_host_free_pinned": (_V, [C.c_void_p]),
    "hpgmg_fmg_solve_host": (_D, [_MP, _I, _I, _I, _D, _D, _D, C.c_void_p, C.c_void_p]),
    "hpgmg_fmg_solve_host_bytes": (C.c_ulonglong, [_MP, _I]),
    "hpgmg_fmg_solve_host_submit": (_I, [_MP, _I, _I, _I, _D, _D, _D, C.c_void_p, C.c_void_p]),
    "hpgmg_fmg_solve_host_wait": (_D, [_MP, _I]),
    "hpgmg_fmg_solve_device": (_D, [_MP, _I, _I, _I, _D, _D, _D, C.c_void_p, C.c_void_p, C.c_void_p]),
    "hpgmg_last_norm_of_F": (_D, [_MP]), "hpgmg_last_norm_of_residual": (_D, [_MP]),
    "hpgmg_last_richardson_error": (_D, []), "hpgmg_last_richardson_order": (_D, []),
    "hpgmg_b200_kernel_launches": (C.c_ulonglong, []), "hpgmg_b200_device_seconds_last_solve": (_D, []),
    "hpgmg_b200_recorded_graphs": (C.c_ulonglong, []),
    "hpgmg_b200_bench_mark": (_V, [_I]), "hpgmg_b200_bench_elapsed_ms": (_D, [_I, _I]),
    "hpgmg_b200_profiler_start": (_V, []), "hpgmg_b200_profiler_stop": (_V, []),
    "hpgmg_b200_gsrb_sweep": (_V, [_LP, _I, _I, _I, _D, _D, _I]),
    "hpgmg_b200_smoother_sweep": (_V, [_LP, _I, _I, _I, _D, _D, _I]),
    "hpgmg_b200_set_comm": (_V, [_I, _I, ALLGATHER_FN, BARRIER_FN, C.c_void_p]),
    "hpgmg_b200_comm_finalize": (_V, []), "hpgmg_b200_p2p_enabled": (_I, []),
    "hpgmg_b200_set_fmg_post_vcycles": (_V, [_I]),
    "hpgmg_b200_set_agglomeration": (_V, [_I]), "hpgmg_b200_get_agglomeration": (_I, []),
    # level.h
    "create_level": (_V, [_LP, _I, _I, _I, _I, _I, _I, _I]), "destroy_level": (_V, [_LP]),
    "create_vectors": (_V, [_LP, _I]), "reset_level_timers": (_V, [_LP]),
    # operators.h
    "stencil_get_radius": (_I, []), "stencil_get_shape": (_I, []),
    "apply_op": (_V, [_LP, _I, _I, _D, _D]), "residual": (_V, [_LP, _I, _I, _I, _D, _D]),
    "smooth": (_V, [_LP, _I, _I, _D, _D]),
    "rebuild_operator": (_V, [_LP, _LP, _D, _D]), "rebuild_operator_blackbox": (_V, [_LP, _D, _D, _I]),
    "restriction": (_V, [_LP, _I, _LP, _I, _I]),
    "interpolation_vcycle": (_V, [_LP, _I, _D, _LP, _I]), "interpolation_fcycle": (_V, [_LP, _I, _D, _LP, _I]),
    "interpolation_v2": (_V, [_LP, _I, _D, _LP, _I]), "interpolation_v4": (_V, [_LP, _I, _D, _LP, _I]),
    "interpolation_p0": (_V, [_LP, _I, _D, _LP, _I]),
    "exchange_boundary": (_V, [_LP, _I, _I]),
    "apply_BCs": (_V, [_LP, _I, _I]), "apply_BCs_v1": (_V, [_LP, _I, _I]),
    "apply_BCs_v2": (_V, [_LP, _I, _I]), "apply_BCs_v4": (_V, [_LP, _I, _I]),
    "extrapolate_betas": (_V, [_LP]),
    "dot": (_D, [_LP, _I, _I]), "norm": (_D, [_LP, _I]), "mean": (_D, [_LP, _I]), "error": (_D, [_LP, _I, _I]),
    "add_vectors": (_V, [_LP, _I, _D, _I, _D, _I]), "scale_vector": (_V, [_LP, _I, _D, _I]),
    "zero_vector": (_V, [_LP, _I]), "shift_vector": (_V, [_LP, _I, _I, _D]),
    "mul_vectors": (_V, [_LP, _I, _D, _I, _I]), "invert_vector": (_V, [_LP, _I, _D, _I]),
    "init_vector": (_V, [_LP, _I, _D]), "color_vector": (_V, [_LP, _I, _I, _I, _I, _I]),
    "random_vector": (_V, [_LP, _I]),
    "initialize_problem": (_V, [_LP, _D, _D, _D]),
    "evaluateBeta": (_D, [_D, _D, _D, _D, _I, _I, _I]), "evaluateF": (_D, [_D, _D, _D, _D, _I, _I, _I]),
    # mg.h, solvers.h
    "MGBuild": (_V, [_MP, _LP, _D, _D, _I]), "MGSolve": (_V, [_MP, _I, _I, _I, _D, _D, _D]),
    "FMGSolve": (_V, [_MP, _I, _I, _I, _D, _D, _D]), "FMGSolve2": (_V, [_MP, _I, _I, _I, _D, _D, _D]),
    "MGPCG": (_V, [_MP, _I, _I, _I, _D, _D, _D]), "MGVCycle": (_V, [_MP, _I, _I, _D, _D, _I]),
    "MGDestroy": (_V, [_MP]), "MGPrintTiming": (_V, [_MP, _I]), "MGResetTimers": (_V, [_MP]),
    "richardson_error": (_V, [_MP, _I, _I]),
    "IterativeSolver": (_V, [_LP, _I, _I, _D, _D, _D]), "IterativeSolver_NumVectors": (_I, []),
}


def bind(cdll, signatures=None):
    """Attach restype/argtypes; raises AttributeError naming the first missing symbol."""
    for name, (res, args) in (signatures or SIGNATURES).items():
        fn = getattr(cdll, name)
        fn.restype = res
        fn.argtypes = args
    return cdll


def lib():
    """The loaded C-ABI library.  Built in-tree by __graft_entry__.build() (make in hpgmg_b200/csrc)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: build it with `make -C hpgmg_b200/csrc` (or __graft_entry__.build()). "
                "hpgmg_b200 has no CPU fallback.")
        _lib = bind(C.CDLL(LIB_PATH))
    return _lib


def init(device=0):
    rc = lib().hpgmg_b200_init(int(device))
    if rc != 0:
        raise RuntimeError(f"hpgmg_b200_init({device}) failed with code {rc}: a B200 (sm_100a) device is required; there is no CPU fallback")


# ------------------------------------------------------------------------------------------------
def box_view(level, flat, box=0):
    """View a flat box array (volume doubles) as [k][j][i] including ghosts and padding."""
    L = level.contents if isinstance(level, _LP) else level
    n = L.box_dim + 2 * L.box_ghosts
    return np.asarray(flat).reshape(-1)[: L.box_volume].reshape(n, n, L.box_jStride)


def download(level, box, vec_id):
    """Copy one box vector (ghosts included) to the host: ndarray [k][j][i] of shape (n+2g, n+2g, jStride)."""
    L = level.contents
    out = np.empty(L.box_volume, dtype=np.float64)
    lib().hpgmg_download_box_vector(level, box, vec_id, out.ctypes.data_as(C.c_void_p))
    return box_view(level, out)


def upload(level, box, vec_id, array):
    L = level.contents
    a = np.ascontiguousarray(array, dtype=np.float64).reshape(-1)
    assert a.size == L.box_volume, (a.size, L.box_volume)
    lib().hpgmg_upload_box_vector(level, box, vec_id, a.ctypes.data_as(C.c_void_p))


def interior(level, arr):
    L = level.contents
    g, n = L.box_ghosts, L.box_dim
    return arr[g:g + n, g:g + n, g:g + n]


def block_list(ptr, n):
    return [block_tuple(ptr[i]) for i in range(n)]


def problem_size(log2_box_dim, target_boxes_per_rank, num_ranks=1, max_coarse_dim=11):
    """boxes_in_i exactly as the reference driver picks it (hpgmg-fv.c:184-197)."""
    box_dim = 1 << log2_box_dim
    target = target_boxes_per_rank * num_ranks
    best = -1
    for bi in range(1, 1000):
        if bi ** 3 <= target:
            odd = box_dim * bi
            while odd % 2 == 0:
                odd //= 2
            if odd <= max_coarse_dim:
                best = bi
    return box_dim, best


class Hierarchy:
    """The reference driver's setup sequence (hpgmg-fv.c:280-308) as an object.

    level_h -> initialize_problem -> rebuild_operator -> MGBuild, for `hpgmg-fv <log2_box_dim>
    <target_boxes_per_rank>` on `num_ranks` ranks (this process being `my_rank`).  `smoother`, `bottom_solver`, `verbose`
    and `use_graphs` are process-wide selections of the library; they are set only when `library` is None.
    """

    def __init__(self, log2_box_dim, target_boxes_per_rank, my_rank=0, num_ranks=1, a=0.0, b=1.0,
                 smoother=SMOOTHER_GSRB, verbose=False, use_graphs=True, build_operator=True, library=None,
                 bc=BC_DIRICHLET, vectors=None, bottom_solver=BOTTOM_BICGSTAB):
        self.L = library or lib()
        self.a, self.b = float(a), float(b)
        self.box_dim, self.boxes_in_i = problem_size(log2_box_dim, target_boxes_per_rank, num_ranks)
        if self.boxes_in_i < 1:
            raise ValueError("failed to find an acceptable problem size")
        if library is None:
            self.L.hpgmg_b200_set_verbose(1 if verbose else 0)
            self.L.hpgmg_b200_set_smoother(smoother)
            self.L.hpgmg_b200_set_bottom_solver(bottom_solver)
            self.L.hpgmg_b200_use_graphs(1 if use_graphs else 0)
        self._level_buf = level_type()
        self.level_h = C.pointer(self._level_buf)
        self.bc = bc
        self.L.create_level(self.level_h, self.boxes_in_i, self.box_dim, self.L.stencil_get_radius(),
                            VECTORS_RESERVED if vectors is None else vectors, bc, my_rank, num_ranks)
        self.h = 1.0 / (float(self.boxes_in_i) * float(self.box_dim))
        self._mg_buf = mg_type()
        self.mg = C.pointer(self._mg_buf)
        self.built = False
        if build_operator:
            self.L.initialize_problem(self.level_h, self.h, self.a, self.b)
            self.L.rebuild_operator(self.level_h, None, self.a, self.b)
            if bc == BC_PERIODIC:                  # remove any constant from the RHS (hpgmg-fv.c:296-302)
                average = self.L.mean(self.level_h, VECTOR_F)
                if average != 0.0:
                    self.L.shift_vector(self.level_h, VECTOR_F, VECTOR_F, -average)
            self.L.MGBuild(self.mg, self.level_h, self.a, self.b, 2 if bc == BC_PERIODIC else 1)   # hpgmg-fv.c:278,281
            self.built = True

    # -- accessors -------------------------------------------------------------------------------
    @property
    def num_levels(self):
        return self._mg_buf.num_levels

    def level(self, l):
        return self._mg_buf.levels[l] if self.built else self.level_h

    def dof(self, l=0):
        d = self.level(l).contents.dim
        return d.i * d.j * d.k

    # -- the hot path ----------------------------------------------------------------------------
    def fmg_solve(self, on_level=0, u_id=VECTOR_U, f_id=VECTOR_F, rtol=1e-10, zero_u=True):
        """zero_vector(U) + FMGSolve, as bench_hpgmg does (hpgmg-fv.c:78-80).  Returns (||r||, ||r||/||f||)."""
        if zero_u:
            self.L.zero_vector(self.level(on_level), u_id)
        self.L.FMGSolve(self.mg, on_level, u_id, f_id, self.a, self.b, rtol)
        r, f = self.L.hpgmg_last_norm_of_residual(self.mg), self.L.hpgmg_last_norm_of_F(self.mg)
        return r, (r / f if f != 0 else float("nan"))

    def fmg_solve_device(self, f, out=None, on_level=0, rtol=1e-10):
        """FMG solve of A u = f with f and u as CUDA tensors of the level's whole domain (hpgmg_fmg_solve_device).

        `f` and `out` are contiguous float64 tensors of shape (dim.k, dim.j, dim.i) on the library's device; element [k, j, i] is
        cell (i, j, k).  `out` may be `f` itself (solved in place); None allocates torch.zeros_like(f).  Only the cells of this
        rank's boxes are read and written.  The solve starts after the work already queued on the current torch stream and
        returns after u is written.  Returns (u, (||r||, ||r||/||f||)) with the F-cycle residual max-norm, as fmg_solve does."""
        import torch
        lvl = self.level(on_level).contents
        shape = (lvl.dim.k, lvl.dim.j, lvl.dim.i)
        device = self.L.hpgmg_b200_device()
        _check_grid_tensor("f", f, shape, device)
        if out is None:
            out = torch.zeros_like(f)
        _check_grid_tensor("out", out, shape, device)
        stream = torch.cuda.current_stream(f.device).cuda_stream
        r = self.L.hpgmg_fmg_solve_device(self.mg, on_level, VECTOR_U, VECTOR_F, self.a, self.b, rtol, f.data_ptr(), out.data_ptr(), stream)
        nf = self.L.hpgmg_last_norm_of_F(self.mg)
        return out, (r, (r / nf if nf != 0 else float("nan")))

    def restrict_rhs_to(self, l):
        """restriction(level l, F <- level l-1, F) as the driver does before solving on level l (hpgmg-fv.c:322)."""
        self.L.restriction(self.level(l), VECTOR_F, self.level(l - 1), VECTOR_F, RESTRICT_CELL)

    def richardson(self, rtol=1e-10):
        """The reference's own correctness check (hpgmg-fv.c:351-366, mg.c:1113-1131): (||error||, order)."""
        norms = []
        for l in range(3):
            if l > 0:
                self.restrict_rhs_to(l)
            norms.append(self.fmg_solve(l, rtol=rtol))
        self.L.richardson_error(self.mg, 0, VECTOR_U)
        return self.L.hpgmg_last_richardson_error(), self.L.hpgmg_last_richardson_order(), norms

    def close(self):
        if self.built:
            self.L.MGDestroy(self.mg)
            self.built = False
        if self.level_h is not None:
            self.L.destroy_level(self.level_h)
            self.level_h = None

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()


def _check_grid_tensor(name, t, shape, device):
    """What hpgmg_fmg_solve_device needs of an array, as TypeError / ValueError instead of the library's exit(1)."""
    import torch
    if not isinstance(t, torch.Tensor):
        raise TypeError(f"{name} must be a torch.Tensor, not {type(t).__name__}")
    if t.dtype != torch.float64:
        raise TypeError(f"{name} must be float64, not {t.dtype}")
    if t.device.type != "cuda" or t.device.index != device:
        raise ValueError(f"{name} is on {t.device}; the library runs on cuda:{device}")
    if tuple(t.shape) != shape:
        raise ValueError(f"{name} has shape {tuple(t.shape)}; the level's domain is (dim.k, dim.j, dim.i) = {shape}")
    if not t.is_contiguous():
        raise ValueError(f"{name} must be contiguous (strides {t.stride()})")
    if t.data_ptr() % 16:
        raise ValueError(f"{name} must start on a 16-byte boundary (data_ptr {t.data_ptr():#x})")


# ------------------------------------------------------------------------------------------------
_comm_keepalive = []


def init_distributed():
    """One process per GPU under torchrun: pick the GPU, create the torch.distributed group and hand
    the library the two setup-time callbacks it needs to build its NCCL communicator."""
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    init(local)
    if world == 1:
        return rank, world
    import torch
    import torch.distributed as dist
    torch.cuda.set_device(local)
    if not dist.is_initialized():
        dist.init_process_group(backend="nccl", device_id=torch.device("cuda", local))

    def _allgather(send, recv, nbytes, ctx):
        src = torch.frombuffer((C.c_char * nbytes).from_address(send), dtype=torch.uint8).cuda()
        out = [torch.empty_like(src) for _ in range(world)]
        dist.all_gather(out, src)
        flat = torch.cat(out).cpu().numpy().tobytes()
        C.memmove(recv, flat, nbytes * world)

    def _barrier(ctx):
        dist.barrier()

    ag, br = ALLGATHER_FN(_allgather), BARRIER_FN(_barrier)
    _comm_keepalive.extend([ag, br])
    lib().hpgmg_b200_set_comm(rank, world, ag, br, None)
    return rank, world
