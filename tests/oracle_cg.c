/*
 * oracle_cg.c -- TEST INFRASTRUCTURE ONLY: the reference's D^-1-preconditioned CG bottom solver (solvers/cg.c, selected there
 * with -DUSE_CG, solvers.c) on top of the plain-C oracle.
 *
 * The oracle (oracle/hpgmg_oracle.c) is included unchanged, so the setup, the operator, the boundary conditions, the
 * transfers and the smoothers (GSRB, or Chebyshev when ohier::cheby is set) are its own; this file adds cg() and the cycles
 * that call it instead of bicgstab() (the oracle's MGVCycle / FMGSolve / Richardson pass, same order of operations).  It is
 * compiled by tests/oracle_cg.py with the oracle's flags (-O2 -ffp-contract=off); nothing under hpgmg_b200/ may use it.
 *
 * cg() is the algorithm the library implements (solvers.c:cg_host_driven, cuda/bicgstab.cuh:cg_solve): vectors r0, r, p, Ap,
 * z are VECTORS_RESERVED+0..4, at most 200 iterations, stop when max|r| < rtol*max|r0|, exact-zero breakdown tests.  The
 * oracle's bottom level has 8 Krylov vectors, of which it uses the first 5.
 */
#include "../oracle/hpgmg_oracle.c"

int cg(olevel *L, int x_id, int R_id, double b, double rtol)
{
  const int r0 = V_RESERVED, r = V_RESERVED + 1, p = V_RESERVED + 2, Ap = V_RESERVED + 3, z = V_RESERVED + 4;
  int j = 0, failed = 0, converged = 0;
  oracle_residual(L, r0, x_id, R_id, b);                     /* one box, Dirichlet: no mean to subtract */
  scale_vec(L, r, 1.0, r0);
  mul_vec(L, z, 1.0, V_DINV, r);
  scale_vec(L, p, 1.0, z);
  double r_dot_z = dot_vec(L, r, z), norm_of_r0 = oracle_norm(L, r);
  if (r_dot_z == 0.0) converged = 1;
  if (norm_of_r0 == 0.0) converged = 1;
  while (j < 200 && !failed && !converged) {
    j++;
    oracle_apply_op(L, Ap, p, b);
    double Ap_dot_p = dot_vec(L, Ap, p);
    if (Ap_dot_p == 0.0) { failed = 1; break; }
    double alpha = r_dot_z / Ap_dot_p;
    if (isinf(alpha)) { failed = 2; break; }
    add_vec(L, x_id, 1.0, x_id, alpha, p);
    add_vec(L, r, 1.0, r, -alpha, Ap);
    double norm_of_r = oracle_norm(L, r);
    if (norm_of_r == 0.0) { converged = 1; break; }
    if (norm_of_r < rtol * norm_of_r0) { converged = 1; break; }
    mul_vec(L, z, 1.0, V_DINV, r);
    double r_dot_z_new = dot_vec(L, r, z);
    if (r_dot_z_new == 0.0) { failed = 3; break; }
    double beta = r_dot_z_new / r_dot_z;
    if (isinf(beta)) { failed = 4; break; }
    add_vec(L, p, 1.0, z, beta, p);
    r_dot_z = r_dot_z_new;
  }
  return j;
}

/* cg() on level `level` of the hierarchy (test hook: x and R are whatever the caller left in them) */
int oracle_cg(ohier *H, int level, int x_id, int R_id, double rtol) { return cg(&H->L[level], x_id, R_id, H->b, rtol); }

/* mg.c:1135-1164, as vcycle() of the oracle */
static void cgvcycle(ohier *H, int e_id, int R_id, int l)
{
  if (l == H->nlevels - 1) { H->krylov += cg(&H->L[l], e_id, R_id, H->b, 1e-3); return; }
  smooth(H, &H->L[l], e_id, R_id);
  oracle_residual(&H->L[l], V_TEMP, e_id, R_id, H->b);
  oracle_restriction(&H->L[l + 1], R_id, &H->L[l], V_TEMP, OR_RESTRICT_CELL);
  zero_vec(&H->L[l + 1], e_id);
  cgvcycle(H, e_id, R_id, l + 1);
  oracle_interpolation_v2(&H->L[l], e_id, 1.0, &H->L[l + 1], e_id);
  smooth(H, &H->L[l], e_id, R_id);
}

/* mg.c:1237-1344, as oracle_fmg_solve() */
double oracle_cg_fmg_solve(ohier *H, int onLevel, double *norm_of_F)
{
  const int e_id = V_U, R_id = V_R, bottom = H->nlevels - 1;
  zero_vec(&H->L[onLevel], V_U);
  const double nF = oracle_norm(&H->L[onLevel], V_F);
  scale_vec(&H->L[onLevel], R_id, 1.0, V_F);
  for (int l = onLevel; l < bottom; l++) oracle_restriction(&H->L[l + 1], R_id, &H->L[l], R_id, OR_RESTRICT_CELL);
  if (bottom > onLevel) zero_vec(&H->L[bottom], e_id);
  H->krylov += cg(&H->L[bottom], e_id, R_id, H->b, 1e-3);
  for (int l = bottom - 1; l >= onLevel; l--) {
    oracle_interpolation_v4(&H->L[l], e_id, 0.0, &H->L[l + 1], e_id);
    cgvcycle(H, e_id, R_id, l);
  }
  oracle_residual(&H->L[onLevel], V_TEMP, e_id, V_F, H->b);
  if (norm_of_F) *norm_of_F = nF;
  return oracle_norm(&H->L[onLevel], V_TEMP);
}

/* hpgmg-fv.c:351-366, mg.c:1113-1131, as oracle_richardson() */
void oracle_cg_richardson(ohier *H, double norms[3], double *err, double *order)
{
  for (int l = 0; l < 3; l++) {
    if (l > 0) oracle_restriction(&H->L[l], V_F, &H->L[l - 1], V_F, OR_RESTRICT_CELL);
    norms[l] = oracle_cg_fmg_solve(H, l, NULL);
  }
  oracle_restriction(&H->L[1], V_TEMP, &H->L[0], V_U, OR_RESTRICT_CELL);
  oracle_restriction(&H->L[2], V_TEMP, &H->L[1], V_U, OR_RESTRICT_CELL);
  add_vec(&H->L[1], V_TEMP, 1.0, V_U, -1.0, V_TEMP);
  add_vec(&H->L[2], V_TEMP, 1.0, V_U, -1.0, V_TEMP);
  const double e2h = oracle_norm(&H->L[1], V_TEMP), e4h = oracle_norm(&H->L[2], V_TEMP);
  *err = e2h;
  *order = log(e4h / e2h) / log(2);
}
