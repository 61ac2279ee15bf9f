/*
 * solvers.c -- bottom solver of the V/F-cycle.
 *
 * Two solvers, chosen at run time with hpgmg_b200_set_bottom_solver (the reference's -DUSE_BICGSTAB / -DUSE_CG):
 *  - BiCGStab (the default) restates /root/reference/finite-volume/source/solvers.c:27-105 and solvers/bicgstab.c:14-97:
 *    right-preconditioned (D^-1) BiCGStab, at most 200 iterations, stop when the max-norm of the intermediate or updated
 *    residual drops below rtol*||r0||, with the reference's exact-zero breakdown tests.
 *  - CG is the D^-1-preconditioned conjugate gradient of solvers/cg.c in the same style: the same cap, stopping test and
 *    exact-zero breakdown tests, the shape of MGPCG (mg.c) with the V-cycle replaced by z = D^-1 r.
 *
 * Every scalar of either solver steers a host branch in the reference (six device->host round trips per BiCGStab
 * iteration if run naively).  The coarsest grid of the benchmark is one box of at most 11^3 cells, so the fast path
 * (hpgmg_bicgstab_device, csrc/cuda) runs the whole solver in ONE thread block with the scalars in registers and can be
 * captured in a CUDA graph.  The host-driven loops below are the general path (multi-box bottoms, periodic problems, the
 * Helmholtz build); they are built from the same public operators and synchronise on every dot/norm.
 */
#include <math.h>
#include <stdio.h>

#include "hpgmg_b200.h"
#include "runtime.h"

/* r0 r p q s t Ap As (solvers.c:92-96).  CG uses the first five (r0 r p Ap z); the bottom level is sized once by MGBuild and
 * the solver may change afterwards, so the count does not depend on the selection (hpgmg_solvers.h). */
int IterativeSolver_NumVectors(void) { return 8; }

static void bicgstab_host_driven(level_type *L, int x_id, int R_id, double a, double b, double rtol)
{
  const int r0 = VECTORS_RESERVED + 0, r = VECTORS_RESERVED + 1, p = VECTORS_RESERVED + 2, q = VECTORS_RESERVED + 3;
  const int s = VECTORS_RESERVED + 4, t = VECTORS_RESERVED + 5, Ap = VECTORS_RESERVED + 6, As = VECTORS_RESERVED + 7;
  const int jMax = 200;
  int j = 0, failed = 0, converged = 0;

  residual(L, r0, x_id, R_id, a, b);
  if (L->must_subtract_mean == 1) { double m = mean(L, r0); shift_vector(L, r0, r0, -m); }
  scale_vector(L, r, 1.0, r0);
  scale_vector(L, p, 1.0, r0);
  double r_dot_r0 = dot(L, r, r0);
  double norm_of_r0 = norm(L, r);
  if (r_dot_r0 == 0.0 || norm_of_r0 == 0.0) converged = 1;
  while (j < jMax && !failed && !converged) {
    j++;  L->Krylov_iterations++;
    mul_vectors(L, q, 1.0, VECTOR_DINV, p);
    apply_op(L, Ap, q, a, b);
    double Ap_dot_r0 = dot(L, Ap, r0);
    if (Ap_dot_r0 == 0.0) { failed = 1; break; }
    double alpha = r_dot_r0 / Ap_dot_r0;
    if (isinf(alpha)) { failed = 2; break; }
    add_vectors(L, x_id, 1.0, x_id, alpha, q);
    add_vectors(L, s, 1.0, r, -alpha, Ap);
    if (L->must_subtract_mean == 1) { double m = mean(L, s); shift_vector(L, s, s, -m); }
    double norm_of_s = norm(L, s);
    if (norm_of_s == 0.0) { converged = 1; break; }
    if (norm_of_s < rtol * norm_of_r0) { converged = 1; break; }
    mul_vectors(L, t, 1.0, VECTOR_DINV, s);
    apply_op(L, As, t, a, b);
    double As_dot_As = dot(L, As, As);
    double As_dot_s  = dot(L, As, s);
    if (As_dot_As == 0.0) { converged = 1; break; }
    double omega = As_dot_s / As_dot_As;
    if (omega == 0.0) { failed = 3; break; }
    if (isinf(omega)) { failed = 4; break; }
    add_vectors(L, x_id, 1.0, x_id, omega, t);
    add_vectors(L, r, 1.0, s, -omega, As);
    if (L->must_subtract_mean == 1) { double m = mean(L, r); shift_vector(L, r, r, -m); }
    double norm_of_r = norm(L, r);
    if (norm_of_r == 0.0) { converged = 1; break; }
    if (norm_of_r < rtol * norm_of_r0) { converged = 1; break; }
    double r_dot_r0_new = dot(L, r, r0);
    if (r_dot_r0_new == 0.0) { failed = 5; break; }
    double beta = (r_dot_r0_new / r_dot_r0) * (alpha / omega);
    if (isinf(beta)) { failed = 6; break; }
    add_vectors(L, VECTOR_TEMP, 1.0, p, -omega, Ap);
    add_vectors(L, p, 1.0, r, beta, VECTOR_TEMP);
    r_dot_r0 = r_dot_r0_new;
  }
  (void)failed;
}

/* D^-1-preconditioned CG (solvers/cg.c).  The device body cg_solve (cuda/bicgstab.cuh) is the same sequence of operations. */
static void cg_host_driven(level_type *L, int x_id, int R_id, double a, double b, double rtol)
{
  const int r0 = VECTORS_RESERVED + 0, r = VECTORS_RESERVED + 1, p = VECTORS_RESERVED + 2, Ap = VECTORS_RESERVED + 3, z = VECTORS_RESERVED + 4;
  const int jMax = 200;
  int j = 0, failed = 0, converged = 0;

  residual(L, r0, x_id, R_id, a, b);
  if (L->must_subtract_mean == 1) { double m = mean(L, r0); shift_vector(L, r0, r0, -m); }
  scale_vector(L, r, 1.0, r0);
  mul_vectors(L, z, 1.0, VECTOR_DINV, r);
  scale_vector(L, p, 1.0, z);
  double r_dot_z = dot(L, r, z);
  double norm_of_r0 = norm(L, r);
  if (r_dot_z == 0.0 || norm_of_r0 == 0.0) converged = 1;
  while (j < jMax && !failed && !converged) {
    j++;  L->Krylov_iterations++;
    apply_op(L, Ap, p, a, b);
    double Ap_dot_p = dot(L, Ap, p);
    if (Ap_dot_p == 0.0) { failed = 1; break; }
    double alpha = r_dot_z / Ap_dot_p;
    if (isinf(alpha)) { failed = 2; break; }
    add_vectors(L, x_id, 1.0, x_id, alpha, p);
    add_vectors(L, r, 1.0, r, -alpha, Ap);
    if (L->must_subtract_mean == 1) { double m = mean(L, r); shift_vector(L, r, r, -m); }
    double norm_of_r = norm(L, r);
    if (norm_of_r == 0.0) { converged = 1; break; }
    if (norm_of_r < rtol * norm_of_r0) { converged = 1; break; }
    mul_vectors(L, z, 1.0, VECTOR_DINV, r);
    double r_dot_z_new = dot(L, r, z);
    if (r_dot_z_new == 0.0) { failed = 3; break; }
    double beta = r_dot_z_new / r_dot_z;
    if (isinf(beta)) { failed = 4; break; }
    add_vectors(L, p, 1.0, z, beta, p);
    r_dot_z = r_dot_z_new;
  }
  (void)failed;
}

void IterativeSolver(level_type *L, int u_id, int f_id, double a, double b, double desired_reduction_in_norm)
{
  if (!L->active) return;
  if (L->must_subtract_mean == -1) {                                               /* solvers.c:30-38 */
#ifdef VECTOR_ALPHA
    const int alpha_is_zero = (dot(L, VECTOR_ALPHA, VECTOR_ALPHA) == 0.0);
    L->must_subtract_mean = (L->boundary_condition.type == BC_PERIODIC && (a == 0 || alpha_is_zero)) ? 1 : 0;
#else
    L->must_subtract_mean = (L->boundary_condition.type == BC_PERIODIC) ? 1 : 0;
#endif
  }
  if (L->numVectors < VECTORS_RESERVED + IterativeSolver_NumVectors())
    create_vectors(L, VECTORS_RESERVED + IterativeSolver_NumVectors());
  if (hpgmg_bicgstab_device(L, u_id, f_id, a, b, desired_reduction_in_norm)) return;     /* either solver, one kernel */
  if (hpgmg_rt_bottom_solver() == HPGMG_BOTTOM_CG) cg_host_driven(L, u_id, f_id, a, b, desired_reduction_in_norm);
  else                                             bicgstab_host_driven(L, u_id, f_id, a, b, desired_reduction_in_norm);
}
