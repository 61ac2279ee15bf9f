/*
 * hpgmg_b200.h -- extension C-ABI of the B200 build (everything the reference API cannot say
 * because it assumes host memory and compile-time variant selection).
 *
 * Plain C, plain pointers and sizes; no CUDA or torch types cross this boundary.  The Python
 * host layer (hpgmg_b200/api.py) binds these with ctypes; a C caller links libhpgmg_b200.so.
 *
 * Reference counterparts are cited per function; where there is none the reason is given.
 */
#ifndef HPGMG_B200_H
#define HPGMG_B200_H

#include "hpgmg_defines.h"
#include "hpgmg_level.h"
#include "hpgmg_operators.h"
#include "hpgmg_solvers.h"
#include "hpgmg_mg.h"

#ifdef __cplusplus
extern "C" {
#endif

/* ---- runtime ------------------------------------------------------------------------------
 * The reference has no device to select (hpgmg-fv.c:103-140 only does MPI_Init).  One process
 * drives one GPU; call once before create_level().  Returns 0 on success; on a machine without
 * a usable sm_100 device it prints the CUDA error and returns non-zero -- there is no CPU path. */
int  hpgmg_b200_init(int device_ordinal);
void hpgmg_b200_finalize(void);
void hpgmg_b200_sync(void);                      /* drain the compute stream                    */
const char *hpgmg_b200_backend(void);            /* "cuda-sm_100a": there is no other backend    */
int  hpgmg_b200_device(void);                    /* ordinal of the library's device; -1 before init */

/* ---- variant selection ----------------------------------------------------------------------
 * The reference picks the smoother at compile time (-DUSE_GSRB | -DUSE_CHEBY | -DUSE_JACOBI | -DUSE_L1JACOBI,
 * operators.fv4.c:176-195, hpgmgconf.py:114-126).  Here it is a runtime switch.  Any other value is refused
 * (a message on stderr; the current selection stays).
 * L1-Jacobi needs the L1 row inverse of every level, which rebuild_operator_blackbox stores only while it is the
 * selected smoother: select it before rebuild_operator / MGBuild.  Smoothing a level without it is a fatal error. */
#define HPGMG_SMOOTHER_GSRB     0                /* 3x red-black = 6 sweeps   (NUM_SMOOTHS 3)   */
#define HPGMG_SMOOTHER_CHEBY    1                /* one degree-6 polynomial   (CHEBYSHEV_DEGREE) */
#define HPGMG_SMOOTHER_JACOBI   2                /* 6 weighted Jacobi sweeps, w = 2/3, D^-1      (operators/jacobi.c) */
#define HPGMG_SMOOTHER_L1JACOBI 3                /* 6 L1-Jacobi sweeps, w = 1, 1/(Aii + sum|Aij|/2) (operators/jacobi.c) */
void hpgmg_b200_set_smoother(int which);
int  hpgmg_b200_get_smoother(void);
/* The bottom solver, likewise: the reference picks it at compile time (-DUSE_BICGSTAB, the default, | -DUSE_CG; solvers.c).
 * Any other value is refused (a message on stderr; the current selection stays).  It is read when a bottom solve is
 * enqueued, so it may change on a built hierarchy; recorded graphs are kept per selection. */
#define HPGMG_BOTTOM_BICGSTAB   0                /* D^-1-preconditioned BiCGStab (solvers/bicgstab.c) */
#define HPGMG_BOTTOM_CG         1                /* D^-1-preconditioned CG       (solvers/cg.c)       */
void hpgmg_b200_set_bottom_solver(int which);
int  hpgmg_b200_get_bottom_solver(void);

/* 0: silent; 1: the reference's progress lines on stdout (default, rank 0 only). */
void hpgmg_b200_set_verbose(int on);

/* 1 (default): FMGSolve/MGSolve record their kernel sequence once per (level,ids) into a CUDA
 * graph and replay it.  0: plain stream launches (used by the per-operator timers). */
void hpgmg_b200_use_graphs(int on);

/* 1 (default): levels of <= 4096 cells that live entirely on this GPU run their whole sub-cycle
 * (smooths, residual, transfers, bottom solve) inside ONE single-thread-block kernel instead of
 * ~45 launches per level visit.  0: one launch per operator everywhere (same bits). */
void hpgmg_b200_use_coarse_kernel(int on);
/* 1 (default): inside that kernel the coarsest levels (as many as fit in 227 KB, from the bottom up)
 * are held in shared memory.  0: they stay in global memory (same bits; for A/B timing). */
void hpgmg_b200_coarse_levels_in_smem(int on);
/* phase clocks of the coarse kernel: on=1 makes the next launches record SM cycles per category; out9 (may be NULL)
 * receives those of the last launch: load, ghost fill, stencil, restriction, zero, interpolation, bottom solve, store, total */
void hpgmg_b200_coarse_profile(int on, long long *out9);

/* 1: each operator synchronises and adds its device time to level->timers.* like the reference's
 * getTime() brackets (e.g. gsrb.c:37,130).  0 (default): timers only hold MGSolve totals. */
void hpgmg_b200_profile_operators(int on);

/* 1: build only the host-side data model (decomposition, block lists, level table): allocations
 * become inaccessible address-space reservations and any kernel launch aborts.  Lets the index
 * mapping be diffed against the reference on a machine without a GPU; it is not a compute path. */
void hpgmg_b200_set_layout_only(int on);

/* The reference's -DUNLIMIT_FMG_ITERATIONS (mg.c:1243-1247): up to n V-cycles after the F-cycle
 * until ||r||/||f|| < rtol.  Default 0, as in the benchmark. */
void hpgmg_b200_set_fmg_post_vcycles(int n);

/* values richardson_error() last printed (mg.c:1128-1130) */
double hpgmg_last_richardson_error(void);
double hpgmg_last_richardson_order(void);

/* ---- moving data across the boundary ------------------------------------------------------
 * The reference reads box arrays directly (e.g. problem.fv.c:129-135).  Device memory needs an
 * explicit copy: `host` holds box->volume doubles in the box's own [k][j][i] layout, ghosts
 * included.  The *_async forms require pinned host memory to overlap; all go through the
 * compute stream so they are ordered with the operators. */
void hpgmg_download_box_vector(level_type *level, int box, int id, double *host);
void hpgmg_upload_box_vector(level_type *level, int box, int id, const double *host);
/* The L1 row inverse L1-Jacobi smooths with (rebuild.c: 1/Aii or 1/(Aii + sum|Aij|/2)), in the same layout.  The
 * Helmholtz build reads VECTOR_L1INV; the default build keeps it outside the vector map, in an array of the level
 * that exists only if L1-Jacobi was selected when the operator was rebuilt (otherwise: a fatal error).  Ghost cells
 * are not meaningful. */
void hpgmg_download_l1inv(level_type *level, int box, double *host);
void *hpgmg_b200_host_alloc_pinned(size_t bytes);
void  hpgmg_b200_host_free_pinned(void *p);

/* FMGSolve with HOST buffers (the end-to-end call of bench.py): f and u hold the CELLS of this rank's boxes, dense:
 * num_my_boxes x box_dim^3 doubles, box-major (the level's box order), [k][j][i] inside a box; pinned memory
 * (hpgmg_b200_host_alloc_pinned) makes the copies asynchronous.  Uploads f into F_id, zeroes u_id, runs FMGSolve
 * (mg.c:1237) and downloads u_id into u; the download overlaps the final residual and norm.  Returns the F-cycle residual
 * max-norm (the number mg.c:1325-1329 prints).  hpgmg_fmg_solve_host_bytes: bytes moved per call and direction. */
double hpgmg_fmg_solve_host(mg_type *all_grids, int onLevel, int u_id, int F_id, double a, double b,
                            double rtol, const double *f_host, double *u_host);
unsigned long long hpgmg_fmg_solve_host_bytes(mg_type *all_grids, int onLevel);
/* The same call split in two for a stream of solves: submit() enqueues upload + solve + download and returns a ticket
 * (0 or 1) at once, wait() blocks until that solve's u_host is complete and returns its residual norm.  Up to two solves
 * may be in flight; the upload of the next and the download of the previous solve then overlap the running one, each on
 * its own stream.  Same bits as hpgmg_fmg_solve_host.  f_host / u_host of a submitted solve belong to the library until
 * wait() returns. */
int    hpgmg_fmg_solve_host_submit(mg_type *all_grids, int onLevel, int u_id, int F_id, double a, double b,
                                   double rtol, const double *f_host, double *u_host);
double hpgmg_fmg_solve_host_wait(mg_type *all_grids, int ticket);
/* FMGSolve with DEVICE arrays of the whole domain, for a caller whose f is already on the GPU (a torch.Tensor, another
 * library's output).  f_dev and u_dev hold dim.k x dim.j x dim.i doubles of level onLevel, [k][j][i] with i fastest: element
 * (k*dim.j + j)*dim.i + i is global cell (i, j, k) -- a contiguous (N, N, N) tensor, NOT the box-major layout of the host call.
 * Only the cells of this rank's boxes are read from f_dev and written to u_dev; the other cells of u_dev are left untouched,
 * so on several ranks the ranks' results combine by summing zero-initialised u.  f_dev == u_dev solves in place (f is read
 * before u is written); arrays that overlap only in part give undefined results.
 * Before it reads f, the library's compute stream waits for everything enqueued on `stream` so far (a cudaStream_t of the
 * library's device; NULL is the legacy default stream).  Returns, after u is written, the F-cycle residual max-norm, and
 * records the norms and the bottom solver's iteration count as hpgmg_fmg_solve_host does, with the same bits for the same f.
 * No staging buffers are allocated.  Refused with a message and exit(1): NULL, host, managed or other-device pointers,
 * pointers not 16-byte aligned, odd box sizes and inactive levels. */
double hpgmg_fmg_solve_device(mg_type *all_grids, int onLevel, int u_id, int F_id, double a, double b,
                              double rtol, const double *f_dev, double *u_dev, void *stream);

/* Norms of the last FMGSolve/MGSolve on this hierarchy: ||F||, ||r|| after the F-cycle (or
 * last V-cycle).  The reference only prints them (mg.c:1325-1329); tests need the values. */
double hpgmg_last_norm_of_F(const mg_type *all_grids);
double hpgmg_last_norm_of_residual(const mg_type *all_grids);

/* ---- evidence ------------------------------------------------------------------------------ */
unsigned long long hpgmg_b200_kernel_launches(void);  /* kernels enqueued so far (graph replays count their nodes) */
double hpgmg_b200_device_seconds_last_solve(void);    /* CUDA-event time of the last FMGSolve/MGSolve body */
unsigned long long hpgmg_b200_recorded_graphs(void);  /* recorded solves (CUDA graphs) the library holds now */

/* event marks on the library's compute stream, for timing several calls from outside (bench.py) */
void   hpgmg_b200_bench_mark(int idx);                /* idx 0..7 */
double hpgmg_b200_bench_elapsed_ms(int from_idx, int to_idx);
/* cudaProfilerStart/Stop around a region, for `ncu --profile-from-start off` captures */
void   hpgmg_b200_profiler_start(void);
void   hpgmg_b200_profiler_stop(void);
/* exactly one GSRB sweep kernel of smooth() (gsrb.c:41-129), without the ghost fill: dst = sweep s of src */
void   hpgmg_b200_gsrb_sweep(level_type *level, int src_id, int dst_id, int rhs_id, double a, double b, int s);
/* the same for whichever smoother is selected (Chebyshev: step s of chebyshev.c:51-97, x_{n-1} = dst; Jacobi and
 * L1-Jacobi: one sweep of jacobi.c, s is ignored) */
void   hpgmg_b200_smoother_sweep(level_type *level, int src_id, int dst_id, int rhs_id, double a, double b, int s);

/* ---- multi-GPU plumbing -----------------------------------------------------------------------
 * The reference talks MPI (exchange_boundary.c:33-97, restriction.c:128-192, misc.c:276,324).
 * Here ranks are processes launched by torchrun, one per GPU.  The host layer provides two
 * callbacks (backed by torch.distributed) that are used only at SETUP time: an allgather of small
 * byte blobs (to distribute the NCCL unique id) and a barrier.  The timed path never calls back
 * into Python: ghost exchanges are direct peer stores into the neighbour GPU's receive buffer plus a
 * flag (CUDA IPC over NVLink; comm.cu), inter-level messages are grouped ncclSend/ncclRecv on the
 * compute stream, norms are an 8-byte ncclAllReduce on a device scalar. */
typedef void (*hpgmg_allgather_fn)(const void *send, void *recv, size_t bytes_per_rank, void *ctx);
typedef void (*hpgmg_barrier_fn)(void *ctx);
void hpgmg_b200_set_comm(int my_rank, int num_ranks, hpgmg_allgather_fn allgather, hpgmg_barrier_fn barrier, void *ctx);
void hpgmg_b200_comm_finalize(void);
/* Multi-GPU only: levels whose boxes have at most `box_dim` cells per side or that are at most 4*box_dim cells wide, and all
 * coarser ones, are owned by rank 0 (default 16, i.e. boxes <= 16^3 or levels <= 64^3; 0 = exactly the reference's rank_of_box).  Same boxes, same bits; call before MGBuild on every rank. */
void hpgmg_b200_set_agglomeration(int box_dim);
int  hpgmg_b200_get_agglomeration(void);
/* 1 if ghost exchanges go through direct peer stores (CUDA IPC over NVLink), 0 if through ncclSend/ncclRecv */
int  hpgmg_b200_p2p_enabled(void);

#ifdef __cplusplus
}
#endif
#endif
