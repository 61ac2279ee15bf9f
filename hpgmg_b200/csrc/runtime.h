/*
 * runtime.h -- internal seam between the C host code (level.c, mg.c, solvers.c, problem.c) and
 * the CUDA translation units.  Nothing here is part of the public C-ABI (see include/).
 *
 * The host code never dereferences vector or buffer memory; it goes through these calls.
 */
#ifndef HPGMG_B200_RUNTIME_H
#define HPGMG_B200_RUNTIME_H

#include <stddef.h>
#include "hpgmg_b200.h"

/* The device mirror of a level (lists, slab geometry) hangs off level_type::fluxes -- a pointer the
 * reference only uses in its experimental flux smoother (level.h, `fluxes`) -- so that level_type
 * keeps EXACTLY the reference's size and layout and a caller compiled against the reference's own
 * level.h can hand us its struct. */
struct hpgmg_device_level;
#define HPGMG_DEV(level)        ((struct hpgmg_device_level *)(level)->fluxes)
#define HPGMG_SET_DEV(level, p) ((level)->fluxes = (double *)(p))

#ifdef __cplusplus
extern "C" {
#endif

/* process-wide settings (runtime.cu) */
int  hpgmg_rt_verbose(void);          /* print reference-style progress lines?            */
int  hpgmg_rt_smoother(void);
int  hpgmg_rt_bottom_solver(void);    /* HPGMG_BOTTOM_BICGSTAB | HPGMG_BOTTOM_CG              */
int  hpgmg_rt_use_graphs(void);
int  hpgmg_rt_profile(void);
int  hpgmg_rt_sm_count(void);         /* multiprocessors of the current device            */
int  hpgmg_rt_layout_only(void);   /* host data model only: no device, kernels refuse to launch */
double hpgmg_rt_wtime(void);          /* host wall clock, seconds                         */

/* device memory (zero-filled) and copies, all ordered on the compute stream */
void *hpgmg_rt_alloc_zero(size_t bytes);
void  hpgmg_rt_free(void *p);
void  hpgmg_rt_copy_d2d(void *dst, const void *src, size_t bytes);
void  hpgmg_rt_copy_h2d(void *dst, const void *src, size_t bytes);
void  hpgmg_rt_copy_d2h(void *dst, const void *src, size_t bytes);
void  hpgmg_rt_sync(void);

/* device mirror of a level's lists (device_level.cu) */
void hpgmg_device_level_create(level_type *level);            /* after lists of create_level exist */
void hpgmg_device_level_rebind_vectors(level_type *level);    /* after create_vectors() regrew     */
void hpgmg_device_level_upload_transfer_lists(level_type *level); /* after build_restriction/interpolation */
void hpgmg_device_level_destroy(level_type *level);

/* CUDA-graph capture of a whole solve (graphs.cu).  `key` identifies the recorded sequence.
 * begin returns 1 if the caller must now enqueue the work (recording), 0 if a recorded graph was
 * replayed and the caller must skip enqueueing. */
int  hpgmg_graph_begin(const void *owner, long long key);
void hpgmg_graph_end(const void *owner, long long key);
void hpgmg_graph_drop_all(const void *owner);

/* device-side scalars: results of norm/dot that stay on the GPU inside a captured solve */
double *hpgmg_rt_scalar_slots(void);                  /* device array of HPGMG_NUM_SCALARS doubles */
void    hpgmg_rt_read_scalars(double *host, int first, int count); /* sync + copy */
#define HPGMG_NUM_SCALARS 64
#define HPGMG_SLOT_NORM_F   0
#define HPGMG_SLOT_NORM_R   1
#define HPGMG_SLOT_KRYLOV   2   /* bottom-solver iterations of the current solve (as a double) */
#define HPGMG_SLOT_SCRATCH  8
#define HPGMG_SLOT_BARRIER  32  /* grid-barrier counter of the persistent smoother */

/* async reductions that leave their result in a scalar slot (no host sync) */
void hpgmg_norm_async(level_type *level, int id_a, int slot);
void hpgmg_copy_norm_async(level_type *level, int id_c, int id_a, int slot);          /* norm(a) and c = 1.0*a in one pass */
void hpgmg_residual_norm_async(level_type *level, int res_id, int x_id, int rhs_id, double a, double b, int slot);  /* residual, then its norm */

/* residual(level, res <- rhs - A x) followed by restriction(level_c, rc <- res, RESTRICT_CELL): one kernel where the level allows it (smooth.cu) */
void hpgmg_restriction_map_prepare(level_type *level, level_type *level_c);          /* MGBuild: the per-box map the fused kernel needs */
void hpgmg_residual_then_restriction(level_type *level_c, int rc_id, level_type *level, int res_id, int x_id, int rhs_id, double a, double b);

/* on-device bottom solver; returns 0 if the level is not eligible (caller falls back to the
 * host-driven BiCGStab in solvers.c) */
int  hpgmg_bicgstab_device(level_type *level, int x_id, int R_id, double a, double b, double rtol);

void hpgmg_rt_zero_scalar(int slot);                  /* async, capturable */

/* peer-visible device memory for receive buffers and flags (comm.cu); plain device memory on one rank */
void  *hpgmg_rt_alloc_comm(size_t bytes);
int    hpgmg_rt_is_comm_memory(const void *p);
void   hpgmg_rt_free_comm(void *p);
void   hpgmg_comm_recycle_arena(void);                              /* collective; start of create_level */
void   hpgmg_comm_register_exchange(level_type *level, int shape);   /* collective over all ranks */
void   hpgmg_comm_unregister(communicator_type *C);
void   hpgmg_comm_register_transfer(communicator_type *Cs, communicator_type *Cr);   /* collective; MGBuild */
void   hpgmg_comm_unregister_transfer(communicator_type *C);
int    hpgmg_comm_xfer_send_lookup(communicator_type *Cs, const blockCopy_type **pack, int *npack);
int    hpgmg_comm_xfer_recv_lookup(communicator_type *Cr);
void   hpgmg_comm_xfer_pre(communicator_type *Cs);
void   hpgmg_comm_xfer_post(communicator_type *Cs);
void   hpgmg_comm_xfer_wait(communicator_type *Cr);
void   hpgmg_comm_xfer_ack(communicator_type *Cr);

/* inter-GPU plumbing (comm.cu): no-ops on a single rank */
int    hpgmg_comm_rank(void);
int    hpgmg_comm_size(void);
void   hpgmg_comm_barrier(void);
double hpgmg_comm_allreduce_max(level_type *level, double v);
double hpgmg_comm_allreduce_sum(level_type *level, double v);
double hpgmg_comm_allreduce_max_world(level_type *level, double v);
void   hpgmg_comm_allreduce_slot_max(level_type *level, int slot);
void   hpgmg_comm_exchange(level_type *level, communicator_type *C, int tag);
void   hpgmg_comm_exchange_wait(level_type *level, communicator_type *C);
void   hpgmg_comm_transfer(level_type *level_send, communicator_type *Cs, level_type *level_recv, communicator_type *Cr, int tag);
void   hpgmg_comm_transfer_wait(level_type *level_send, communicator_type *Cs, level_type *level_recv, communicator_type *Cr);

/* default build: the L1 row inverse of a level (smooth.cu); a fatal error if the level was built without it */
double *hpgmg_l1inv_array(level_type *level);

/* coarse end of the cycle as one single-block kernel (coarse.cu): levels from..bottom */
int  hpgmg_coarse_chain_eligible(mg_type *MG, int from);
void hpgmg_coarse_cycle(mg_type *MG, int from, int mode_ftail, int zero_bottom, int e_id, int R_id, double a, double b);

/* end-to-end solve with host buffers (mg.c: hpgmg_fmg_solve_host): dense staging buffers, the side stream the download runs
 * on, and the kernels that move cells between a dense [box][k][j][i] buffer and the padded boxes (blas1.cu) */
void *hpgmg_rt_staging(int which, size_t bytes);
void  hpgmg_rt_side_begin(void);
void  hpgmg_rt_side_end(void);
void  hpgmg_rt_side_join(void);
void  hpgmg_rt_pipe_upload(int slot, void *stage, const void *host, size_t bytes);      /* pipelined solves: upload / download streams */
void  hpgmg_rt_pipe_download(int slot, void *host, const void *stage, size_t bytes);
void  hpgmg_rt_pipe_scalars(int slot);
void  hpgmg_rt_pipe_wait(int slot, double *scalars3);
void  hpgmg_rt_pipe_destroy(void);
void  hpgmg_unpack_copy_norm_async(level_type *level, int id_f, int id_r, const double *dense, int slot);   /* F = dense; R = 1.0*F; slot = max|F| */
void  hpgmg_pack_async(level_type *level, int id, double *dense);
void  hpgmg_unpack_async(level_type *level, int id, const double *dense);
/* end-to-end solve with device arrays of the whole domain (mg.c: hpgmg_fmg_solve_device): the same moves to and from a
 * [k][j][i] array of the level's dim.k x dim.j x dim.i cells, each box at its low corner (blas1.cu) */
void  hpgmg_grid_unpack_copy_norm_async(level_type *level, int id_f, int id_r, const double *grid, int slot);
void  hpgmg_grid_pack_async(level_type *level, int id, double *grid);
void  hpgmg_rt_check_device_array(const char *who, const char *name, const void *p);  /* exit(1) unless 16-byte aligned memory of this device */
void  hpgmg_rt_wait_for_stream(void *stream);                                         /* the compute stream waits for what `stream` holds now */

/* event timing of a solve body */
void hpgmg_rt_timer_start(void);
void hpgmg_rt_timer_stop(void);

#ifdef __cplusplus
}
#endif
#endif
