/*
 * oracle_fv2_helmholtz.c -- TEST INFRASTRUCTURE ONLY: a plain-C restatement of the library's fv2 Helmholtz flavour (the
 * reference's operators.fv2.c built with -DUSE_HELMHOLTZ) for one-box-per-level hierarchies (`hpgmg-fv L 1`).
 *
 *   A x = a*alpha[ijk]*x[ijk] - b*h2inv*( bi[i+1](x[i+1]-x) + bi[i](x[i-1]-x) + ... j ... k )
 *
 * tests/oracle_fv2.c (and through it oracle/hpgmg_oracle.c) is included unchanged: its setup, boundary conditions, transfers
 * and BLAS1 are used as they are.  This file restates the parts that apply the operator with a and alpha threaded through:
 * the operator and residual, the four smoothers, the 2-colour black-box diagonal (Aii with the a*alpha term, the fallback
 * a + b*h2inv), BiCGStab, CG and the cycles.  alpha is 1.0 on the index range initialize_problem writes (cells 0..dim
 * inclusive, problem.fv.c) and is restricted with RESTRICT_CELL by rebuild_operator; the driver solves a = b = 1
 * (hpgmg-fv.c:286-288).
 *
 * The reference sources were not available: this follows the Helmholtz form of operators.fv4.c:56-85 applied to the fv2
 * operator as the library states it, and has not been diffed against the reference's operators.fv2.c.
 */
#include "oracle_fv2.c"

#define V_ALPHA (V_RESERVED + 9)       /* after the 8 Krylov vectors and the L1 row inverse of oracle_fv2.c */

static inline double fvh_op_ijk(const double *x, const double *alpha, const double *bi, const double *bj, const double *bk, int q, int jS, int kS,
                                double a, double b, double h2inv)
{
  return a * alpha[q] * x[q] - b * h2inv * (bi[q + 1] * (x[q + 1] - x[q]) + bi[q] * (x[q - 1] - x[q])
                                          + bj[q + jS] * (x[q + jS] - x[q]) + bj[q] * (x[q - jS] - x[q])
                                          + bk[q + kS] * (x[q + kS] - x[q]) + bk[q] * (x[q - kS] - x[q]));
}
#define FVH_OP(L, x, q, a, b, h2inv) fvh_op_ijk(x, cell0(L, V_ALPHA), cell0(L, V_BI), cell0(L, V_BJ), cell0(L, V_BK), q, (L)->jS, (L)->kS, a, b, h2inv)

void fvh_apply_op(const olevel *L, int Ax_id, int x_id, double a, double b)
{
  fv2_fill(L, x_id);
  const double h2inv = 1.0 / (L->h * L->h);
  const double *x = cell0(L, x_id);
  double *Ax = cell0(L, Ax_id);
  for (int k = 0; k < L->n; k++) for (int j = 0; j < L->n; j++) for (int i = 0; i < L->n; i++) {
    const int q = IDX(L, i, j, k);
    Ax[q] = FVH_OP(L, x, q, a, b, h2inv);
  }
}
void fvh_residual(const olevel *L, int res_id, int x_id, int rhs_id, double a, double b)
{
  fv2_fill(L, x_id);
  const double h2inv = 1.0 / (L->h * L->h);
  const double *x = cell0(L, x_id), *rhs = cell0(L, rhs_id);
  double *res = cell0(L, res_id);
  for (int k = 0; k < L->n; k++) for (int j = 0; j < L->n; j++) for (int i = 0; i < L->n; i++) {
    const int q = IDX(L, i, j, k);
    res[q] = rhs[q] - FVH_OP(L, x, q, a, b, h2inv);
  }
}

/* smooth(): FV2_SWEEPS sweeps x -> TEMP -> x, each after a ghost fill of its source (oracle_fv2.c's fv2_smooth with the term) */
void fvh_smooth(const olevel *L, int smoother, int x_id, int rhs_id, double a, double b)
{
  const double h2inv = 1.0 / (L->h * L->h);
  double c1[FV2_CHEBY_DEGREE], c2[FV2_CHEBY_DEGREE];                                 /* chebyshev.c:22-40 */
  {
    double beta = 1.000 * L->eig, alpha = 0.125000 * beta, theta = 0.5 * (beta + alpha), delta = 0.5 * (beta - alpha);
    double sigma = theta / delta, rho_n = 1 / sigma;
    c1[0] = 0.0;  c2[0] = 1 / theta;
    for (int s = 1; s < FV2_CHEBY_DEGREE; s++) { double rho_nm1 = rho_n; rho_n = 1.0 / (2.0 * sigma - rho_nm1); c1[s] = rho_n * rho_nm1; c2[s] = rho_n * 2.0 / delta; }
  }
  const double weight = smoother == FV2_L1JACOBI ? 1.0 : 2.0 / 3.0;
  const double *rhs = cell0(L, rhs_id), *Dinv = cell0(L, V_DINV);
  const double *lam = smoother == FV2_L1JACOBI ? cell0(L, V_L1) : Dinv;
  for (int s = 0; s < FV2_SWEEPS; s++) {
    const int src = (s & 1) ? V_TEMP : x_id, dst = (s & 1) ? x_id : V_TEMP;
    fv2_fill(L, src);
    const double *xn = cell0(L, src);
    double *xp = cell0(L, dst);
    for (int k = 0; k < L->n; k++) for (int j = 0; j < L->n; j++) for (int i = 0; i < L->n; i++) {
      const int q = IDX(L, i, j, k);
      if (smoother == FV2_GSRB && ((i ^ j ^ k ^ s) & 1)) { xp[q] = xn[q]; continue; }   /* box low = (0,0,0) */
      const double Ax = FVH_OP(L, xn, q, a, b, h2inv);
      if (smoother == FV2_GSRB)       xp[q] = xn[q] + Dinv[q] * (rhs[q] - Ax);
      else if (smoother == FV2_CHEBY) xp[q] = xn[q] + c1[s % FV2_CHEBY_DEGREE] * (xn[q] - xp[q]) + c2[s % FV2_CHEBY_DEGREE] * Dinv[q] * (rhs[q] - Ax);
      else                            xp[q] = xn[q] + (weight * lam[q]) * (rhs[q] - Ax);
    }
  }
}

/* rebuild_operator_blackbox(level, a, b, 2) (rebuild.c:47-208) with the a*alpha term; the L1 row inverse is kept in V_L1 */
static void fvh_rebuild_blackbox(olevel *L, double a, double b)
{
  int colors = 2;
  if (L->n < colors) colors = L->n;
  const double h2inv = 1.0 / (L->h * L->h);
  zero_vec(L, V_DINV);  zero_vec(L, V_E);
  double *x = cell0(L, V_TEMP), *Aii = cell0(L, V_DINV), *sum = cell0(L, V_E), *l1 = cell0(L, V_L1);
  for (int kc = 0; kc < colors; kc++) for (int jc = 0; jc < colors; jc++) for (int ic = 0; ic < colors; ic++) {
    for (int k = 0; k < L->n; k++) for (int j = 0; j < L->n; j++) for (int i = 0; i < L->n; i++)
      x[IDX(L, i, j, k)] = (((i + ic) % colors) == 0 ? 1.0 : 0.0) * (((j + jc) % colors) == 0 ? 1.0 : 0.0) * (((k + kc) % colors) == 0 ? 1.0 : 0.0);
    fv2_fill(L, V_TEMP);
    for (int k = 0; k < L->n; k++) for (int j = 0; j < L->n; j++) for (int i = 0; i < L->n; i++) {
      const int q = IDX(L, i, j, k);
      const double Ax = FVH_OP(L, x, q, a, b, h2inv);
      Aii[q] += (x[q]) * Ax;
      sum[q] += fabs((1.0 - x[q]) * Ax);
    }
  }
  double eig = -1e9;
  for (int k = 0; k < L->n; k++) for (int j = 0; j < L->n; j++) for (int i = 0; i < L->n; i++) {
    const int q = IDX(L, i, j, k);
    if (Aii[q] == 0.0) Aii[q] = a + b * h2inv;
    double Di = (Aii[q] + sum[q]) / Aii[q];
    if (Di > eig) eig = Di;
    if (Aii[q] >= 1.5 * sum[q]) sum[q] = 1.0 / (Aii[q]); else sum[q] = 1.0 / (Aii[q] + 0.5 * sum[q]);
    l1[q] = sum[q];
    Aii[q] = 1.0 / Aii[q];
  }
  L->eig = eig;
}
static void fvh_rebuild_operator(olevel *L, const olevel *from, double a, double b)
{
  if (from) {
    oracle_restriction(L, V_ALPHA, from, V_ALPHA, OR_RESTRICT_CELL);
    oracle_restriction(L, V_BI, from, V_BI, OR_RESTRICT_FACE_I);
    oracle_restriction(L, V_BJ, from, V_BJ, OR_RESTRICT_FACE_J);
    oracle_restriction(L, V_BK, from, V_BK, OR_RESTRICT_FACE_K);
  }
  fvh_rebuild_blackbox(L, a, b);
}

/* ---- bottom solvers: oracle_fv2.c's fv2_bicgstab / fv2_cg over the Helmholtz operator ---- */
int fvh_bicgstab(olevel *L, int x_id, int R_id, double a, double b, double rtol)
{
  const int r0 = V_RESERVED, r = V_RESERVED + 1, p = V_RESERVED + 2, q = V_RESERVED + 3, s = V_RESERVED + 4, t = V_RESERVED + 5, Ap = V_RESERVED + 6, As = V_RESERVED + 7;
  int j = 0, failed = 0, converged = 0;
  fvh_residual(L, r0, x_id, R_id, a, b);
  scale_vec(L, r, 1.0, r0);
  scale_vec(L, p, 1.0, r0);
  double r_dot_r0 = dot_vec(L, r, r0), norm_of_r0 = oracle_norm(L, r);
  if (r_dot_r0 == 0.0) converged = 1;
  if (norm_of_r0 == 0.0) converged = 1;
  while (j < 200 && !failed && !converged) {
    j++;
    mul_vec(L, q, 1.0, V_DINV, p);
    fvh_apply_op(L, Ap, q, a, b);
    double Ap_dot_r0 = dot_vec(L, Ap, r0);
    if (Ap_dot_r0 == 0.0) { failed = 1; break; }
    double alpha = r_dot_r0 / Ap_dot_r0;
    if (isinf(alpha)) { failed = 2; break; }
    add_vec(L, x_id, 1.0, x_id, alpha, q);
    add_vec(L, s, 1.0, r, -alpha, Ap);
    double norm_of_s = oracle_norm(L, s);
    if (norm_of_s == 0.0) { converged = 1; break; }
    if (norm_of_s < rtol * norm_of_r0) { converged = 1; break; }
    mul_vec(L, t, 1.0, V_DINV, s);
    fvh_apply_op(L, As, t, a, b);
    double As_dot_As = dot_vec(L, As, As), As_dot_s = dot_vec(L, As, s);
    if (As_dot_As == 0.0) { converged = 1; break; }
    double omega = As_dot_s / As_dot_As;
    if (omega == 0.0) { failed = 3; break; }
    if (isinf(omega)) { failed = 4; break; }
    add_vec(L, x_id, 1.0, x_id, omega, t);
    add_vec(L, r, 1.0, s, -omega, As);
    double norm_of_r = oracle_norm(L, r);
    if (norm_of_r == 0.0) { converged = 1; break; }
    if (norm_of_r < rtol * norm_of_r0) { converged = 1; break; }
    double r_dot_r0_new = dot_vec(L, r, r0);
    if (r_dot_r0_new == 0.0) { failed = 5; break; }
    double beta = (r_dot_r0_new / r_dot_r0) * (alpha / omega);
    if (isinf(beta)) { failed = 6; break; }
    add_vec(L, V_TEMP, 1.0, p, -omega, Ap);
    add_vec(L, p, 1.0, r, beta, V_TEMP);
    r_dot_r0 = r_dot_r0_new;
  }
  return j;
}
int fvh_cg(olevel *L, int x_id, int R_id, double a, double b, double rtol)
{
  const int r0 = V_RESERVED, r = V_RESERVED + 1, p = V_RESERVED + 2, Ap = V_RESERVED + 3, z = V_RESERVED + 4;
  int j = 0, failed = 0, converged = 0;
  fvh_residual(L, r0, x_id, R_id, a, b);
  scale_vec(L, r, 1.0, r0);
  mul_vec(L, z, 1.0, V_DINV, r);
  scale_vec(L, p, 1.0, z);
  double r_dot_z = dot_vec(L, r, z), norm_of_r0 = oracle_norm(L, r);
  if (r_dot_z == 0.0) converged = 1;
  if (norm_of_r0 == 0.0) converged = 1;
  while (j < 200 && !failed && !converged) {
    j++;
    fvh_apply_op(L, Ap, p, a, b);
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

/* ---- cycles: mg.c:1135-1164 (MGVCycle), :1237-1344 (FMGSolve); the same as oracle_fv2.c with a threaded through ---- */
static int fvh_bottom(fv2hier *F, int x_id, int R_id)
{
  olevel *L = &F->H.L[F->H.nlevels - 1];
  return F->bottom == FV2_CG ? fvh_cg(L, x_id, R_id, F->H.a, F->H.b, 1e-3) : fvh_bicgstab(L, x_id, R_id, F->H.a, F->H.b, 1e-3);
}
static void fvh_vcycle(fv2hier *F, int e_id, int R_id, int l)
{
  ohier *H = &F->H;
  if (l == H->nlevels - 1) { H->krylov += fvh_bottom(F, e_id, R_id); return; }
  fvh_smooth(&H->L[l], F->smoother, e_id, R_id, H->a, H->b);
  fvh_residual(&H->L[l], V_TEMP, e_id, R_id, H->a, H->b);
  oracle_restriction(&H->L[l + 1], R_id, &H->L[l], V_TEMP, OR_RESTRICT_CELL);
  zero_vec(&H->L[l + 1], e_id);
  fvh_vcycle(F, e_id, R_id, l + 1);
  fv2_interpolation_p0(&H->L[l], e_id, 1.0, &H->L[l + 1], e_id);
  fvh_smooth(&H->L[l], F->smoother, e_id, R_id, H->a, H->b);
}
double fvh_fmg_solve(fv2hier *F, int onLevel, double *norm_of_F)
{
  ohier *H = &F->H;
  const int e_id = V_U, R_id = V_R, bottom = H->nlevels - 1;
  zero_vec(&H->L[onLevel], V_U);
  const double nF = oracle_norm(&H->L[onLevel], V_F);
  scale_vec(&H->L[onLevel], R_id, 1.0, V_F);
  for (int l = onLevel; l < bottom; l++) oracle_restriction(&H->L[l + 1], R_id, &H->L[l], R_id, OR_RESTRICT_CELL);
  if (bottom > onLevel) zero_vec(&H->L[bottom], e_id);
  H->krylov += fvh_bottom(F, e_id, R_id);
  for (int l = bottom - 1; l >= onLevel; l--) {
    fv2_interpolation_v2(&H->L[l], e_id, 0.0, &H->L[l + 1], e_id);
    fvh_vcycle(F, e_id, R_id, l);
  }
  fvh_residual(&H->L[onLevel], V_TEMP, e_id, V_F, H->a, H->b);
  if (norm_of_F) *norm_of_F = nF;
  return oracle_norm(&H->L[onLevel], V_TEMP);
}

/* hpgmg-fv.c:280-308 + MGBuild for `hpgmg-fv log2_dim 1` with the radius-1 stencil, solving a*alpha*u - b*div(beta grad u) = f */
fv2hier *fvh_build(int log2_dim, int smoother, int bottom, double a, double b)
{
  fv2hier *F = (fv2hier *)calloc(1, sizeof(fv2hier));
  ohier *H = &F->H;
  F->smoother = smoother;  F->bottom = bottom;
  H->a = a;  H->b = b;  H->cheby = 0;
  H->nlevels = log2_dim + 1;
  H->L = (olevel *)calloc((size_t)H->nlevels, sizeof(olevel));
  for (int l = 0; l < H->nlevels; l++) level_init(&H->L[l], 1 << (log2_dim - l), V_RESERVED + 10);
  initialize_problem(&H->L[0], 1.0 / (double)(1 << log2_dim));
  {
    olevel *L = &H->L[0];
    double *alpha = cell0(L, V_ALPHA);
    for (int k = 0; k <= L->n; k++) for (int j = 0; j <= L->n; j++) for (int i = 0; i <= L->n; i++) alpha[IDX(L, i, j, k)] = 1.0;
  }
  fvh_rebuild_operator(&H->L[0], NULL, H->a, H->b);
  for (int l = 1; l < H->nlevels; l++) { H->L[l].h = 2.0 * H->L[l - 1].h; fvh_rebuild_operator(&H->L[l], &H->L[l - 1], H->a, H->b); }
  return F;
}

/* the driver's Richardson pass (hpgmg-fv.c:351-366) */
void fvh_richardson(fv2hier *F, double norms[3], double *err, double *order)
{
  ohier *H = &F->H;
  for (int l = 0; l < 3; l++) {
    if (l > 0) oracle_restriction(&H->L[l], V_F, &H->L[l - 1], V_F, OR_RESTRICT_CELL);
    norms[l] = fvh_fmg_solve(F, l, NULL);
  }
  oracle_restriction(&H->L[1], V_TEMP, &H->L[0], V_U, OR_RESTRICT_CELL);
  oracle_restriction(&H->L[2], V_TEMP, &H->L[1], V_U, OR_RESTRICT_CELL);
  add_vec(&H->L[1], V_TEMP, 1.0, V_U, -1.0, V_TEMP);
  add_vec(&H->L[2], V_TEMP, 1.0, V_U, -1.0, V_TEMP);
  const double e2h = oracle_norm(&H->L[1], V_TEMP), e4h = oracle_norm(&H->L[2], V_TEMP);
  *err = e2h;
  *order = log(e4h / e2h) / log(2);
}

/* raw access for Python */
void fvh_level_apply_op(fv2hier *F, int l, int Ax_id, int x_id) { fvh_apply_op(&F->H.L[l], Ax_id, x_id, F->H.a, F->H.b); }
void fvh_level_residual(fv2hier *F, int l, int res_id, int x_id, int rhs_id) { fvh_residual(&F->H.L[l], res_id, x_id, rhs_id, F->H.a, F->H.b); }
void fvh_level_smooth(fv2hier *F, int l, int x_id, int rhs_id) { fvh_smooth(&F->H.L[l], F->smoother, x_id, rhs_id, F->H.a, F->H.b); }
int fvh_alpha_id(void) { return V_ALPHA; }
int fvh_l1_id(void) { return V_L1; }
