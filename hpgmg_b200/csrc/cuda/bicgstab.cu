/*
 * bicgstab.cu -- the bottom solver as ONE single-thread-block kernel: BiCGStab (bicgstab_kernel) or, when
 * HPGMG_BOTTOM_CG is selected, D^-1-preconditioned CG (cg_kernel, the restatement of solvers.c:cg_host_driven).
 *
 * Restates solvers/bicgstab.c:14-97 (diagonally right-preconditioned BiCGStab, <=200 iterations,
 * stop when ||s||inf or ||r||inf < rtol*||r0||inf, exact-zero breakdown tests).  In the reference
 * every scalar (6 per iteration) steers a host branch; here the coarsest grid is one box of at
 * most 11^3 cells, so a single CTA runs the whole solve with the scalars in registers: no host
 * round trip, no launch per BLAS1 op, and the kernel can sit inside a captured CUDA graph.
 *
 * Bit-exactness: dot products are accumulated in the reference's order (k, j, i; one tile) by one
 * thread over products staged in shared memory; the max-norm is order-free; apply_op / residual use
 * the same device bodies (stencil.cuh, bc.cuh) as the level-wide kernels.
 */
#include "bicgstab.cuh"

__global__ void __launch_bounds__(BOTTOM_THREADS) bicgstab_kernel(const BottomArgs A)
{
  PDL_WAIT();
  __shared__ double prod[BOTTOM_MAX_CELLS];
  __shared__ double red[36];
  bicgstab_solve(A, prod, red);
}
__global__ void __launch_bounds__(BOTTOM_THREADS) cg_kernel(const BottomArgs A)
{
  PDL_WAIT();
  __shared__ double prod[BOTTOM_MAX_CELLS];
  __shared__ double red[36];
  cg_solve(A, prod, red);
}

/* Returns 1 if the solve (of the selected bottom solver) was enqueued on the device, 0 if the level is not eligible (more
 * than one box on this rank, other ranks involved, a periodic problem that needs mean subtraction, or a box larger than the
 * kernel's shared-memory staging) and the caller must use the host-driven loop.  Eligibility does not depend on the solver. */
/* side-effect free: would hpgmg_bicgstab_device() take this level?  (mg.c uses it to decide whether a solve can be
 * recorded into a CUDA graph: the host-driven fallback synchronises on every dot / norm) */
extern "C" int hpgmg_bicgstab_device_eligible(const level_type *level)
{
#if defined(VECTOR_ALPHA) && !defined(HPGMG_FV2)
  return 0;                                        /* fv4 Helmholtz build: host-driven solvers over the public operators (solvers.c) */
#endif
  if (level->must_subtract_mean == 1) return 0;
  if (level->boundary_condition.type != BC_DIRICHLET) return 0;
  if (level->num_my_boxes != 1) return 0;
  if (level->boxes_in.i != 1 || level->boxes_in.j != 1 || level->boxes_in.k != 1) return 0;
  if (level->box_dim > BOTTOM_MAX_DIM || level->box_dim < STENCIL_RADIUS) return 0;      /* fv4: 2^3 and up; fv2: 1^3 and up */
  if (level->box_ghosts != STENCIL_RADIUS) return 0;
  const hpgmg_device_level *D = HPGMG_DEV(level);
  /* the fill tables are rebuilt for the new vector count when IterativeSolver grows the level (create_vectors) */
  if (D->fill_nvec == 0 || D->fill[STENCIL_SHAPE].nlate > 0) return 0;
  return 1;
}

extern "C" int hpgmg_bicgstab_device(level_type *level, int x_id, int R_id, double a, double b, double rtol)
{
  if (!hpgmg_bicgstab_device_eligible(level)) return 0;
  hpgmg_device_level *D = HPGMG_DEV(level);
  BottomArgs A;
  A.L = D->L;
  if (D->fill_nvec != level->numVectors) return 0;
  A.bc = D->fill[STENCIL_SHAPE].bc;  A.nbc = D->fill[STENCIL_SHAPE].nbc;
  A.x_id = x_id;  A.R_id = R_id;  A.a = a;  A.b = b;
  A.ids = bottom_ids_identity();
  A.h2inv = 1.0 / (level->h * level->h);
  A.rtol = rtol;
  A.iters = hpgmg_rt_scalar_slots() + HPGMG_SLOT_KRYLOV;
  if (hpgmg_rt_bottom_solver() == HPGMG_BOTTOM_CG) LAUNCH(cg_kernel, 1, BOTTOM_THREADS, 0, A);
  else                                             LAUNCH(bicgstab_kernel, 1, BOTTOM_THREADS, 0, A);
  return 1;
}

