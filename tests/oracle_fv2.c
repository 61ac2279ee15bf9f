/*
 * oracle_fv2.c -- TEST INFRASTRUCTURE ONLY: a plain-C restatement of the library's fv2 flavour (the reference linked with
 * operators.fv2.c) for one-box-per-level hierarchies (`hpgmg-fv L 1`: 2^L, 2^(L-1), ... 2, 1 cells per side, because the
 * radius-1 stencil lets boxes shrink to one cell).
 *
 * The oracle (oracle/hpgmg_oracle.c) is included unchanged.  Its setup (initialize_problem), restriction, interpolation_v2
 * and BLAS1 are used as they are; its levels keep their 2-layer layout, of which only the first ghost layer is ever read
 * here.  This file adds the fv2 operator, its boundary conditions (apply_BCs_v2 on the STAR shape, v1 below 2^3), the
 * piecewise-constant interpolation_p0, the 2-colour black-box diagonal (no extrapolate_betas), the 4-sweep smoothers
 * (GSRB RBRB, Chebyshev degree 4, Jacobi 2/3 and L1-Jacobi), BiCGStab and CG over the fv2 operator, and the cycles
 * (V-cycle interpolation p0, F-cycle interpolation v2).  It is compiled by tests/oracle_fv2.py with the oracle's flags.
 */
#include "../oracle/hpgmg_oracle.c"

#define FV2_SWEEPS 4
#define FV2_CHEBY_DEGREE 4
#define V_L1 (V_RESERVED + 8)          /* the L1 row inverse (every level has 8 Krylov vectors and this one) */
enum { FV2_GSRB = 0, FV2_CHEBY = 1, FV2_JACOBI = 2, FV2_L1JACOBI = 3 };
enum { FV2_BICGSTAB = 0, FV2_CG = 1 };

typedef struct { ohier H; int smoother, bottom; } fv2hier;

/* A x at one cell: -b h2inv (bi[i+1](x[i+1]-x) + bi[i](x[i-1]-x) + ... j ... k), left to right */
static inline double fv2_op_ijk(const double *x, const double *bi, const double *bj, const double *bk, int q, int jS, int kS, double b, double h2inv)
{
  return -b * h2inv * (bi[q + 1] * (x[q + 1] - x[q]) + bi[q] * (x[q - 1] - x[q])
                     + bj[q + jS] * (x[q + jS] - x[q]) + bj[q] * (x[q - jS] - x[q])
                     + bk[q + kS] * (x[q + kS] - x[q]) + bk[q] * (x[q - kS] - x[q]));
}

/* apply_BCs_v1 (boundary_fv.c:6-90) with one ghost layer: a ghost cell is the cell one step inward along every normal axis,
 * times -1 on faces and corners, +1 on edges */
static void fv2_bc_v1(const olevel *L, int id, int shape)
{
  double *x = cell0(L, id);
  const int n = L->n;
  for (int dk = -1; dk <= 1; dk++) for (int dj = -1; dj <= 1; dj++) for (int di = -1; di <= 1; di++) {
    if (!shape_has(shape, di, dj, dk)) continue;
    const int m = (di != 0) + (dj != 0) + (dk != 0);
    const double scale = (m == 2) ? 1.0 : -1.0;
    const int lo[3] = { di < 0 ? -1 : (di > 0 ? n : 0), dj < 0 ? -1 : (dj > 0 ? n : 0), dk < 0 ? -1 : (dk > 0 ? n : 0) };
    const int ext[3] = { di ? 1 : n, dj ? 1 : n, dk ? 1 : n };
    const int stride = -di - dj * L->jS - dk * L->kS;
    for (int c = 0; c < ext[2]; c++) for (int bb = 0; bb < ext[1]; bb++) for (int a = 0; a < ext[0]; a++) {
      const int q = IDX(L, a + lo[0], bb + lo[1], c + lo[2]);
      x[q] = scale * x[q + stride];
    }
  }
}
/* apply_BCs_v2, v1 below 2^3 */
static void fv2_bcs(const olevel *L, int id, int shape)
{
  if (L->n < 2) fv2_bc_v1(L, id, shape); else oracle_apply_BCs_v2(L, id, shape);
}
static void fv2_fill(const olevel *L, int id) { fv2_bcs(L, id, OR_SHAPE_STAR); }   /* exchange_boundary is empty for one box */

void fv2_apply_op(const olevel *L, int Ax_id, int x_id, double b)
{
  fv2_fill(L, x_id);
  const double h2inv = 1.0 / (L->h * L->h);
  const double *x = cell0(L, x_id), *bi = cell0(L, V_BI), *bj = cell0(L, V_BJ), *bk = cell0(L, V_BK);
  double *Ax = cell0(L, Ax_id);
  for (int k = 0; k < L->n; k++) for (int j = 0; j < L->n; j++) for (int i = 0; i < L->n; i++) {
    const int q = IDX(L, i, j, k);
    Ax[q] = fv2_op_ijk(x, bi, bj, bk, q, L->jS, L->kS, b, h2inv);
  }
}
void fv2_residual(const olevel *L, int res_id, int x_id, int rhs_id, double b)
{
  fv2_fill(L, x_id);
  const double h2inv = 1.0 / (L->h * L->h);
  const double *x = cell0(L, x_id), *rhs = cell0(L, rhs_id), *bi = cell0(L, V_BI), *bj = cell0(L, V_BJ), *bk = cell0(L, V_BK);
  double *res = cell0(L, res_id);
  for (int k = 0; k < L->n; k++) for (int j = 0; j < L->n; j++) for (int i = 0; i < L->n; i++) {
    const int q = IDX(L, i, j, k);
    res[q] = rhs[q] - fv2_op_ijk(x, bi, bj, bk, q, L->jS, L->kS, b, h2inv);
  }
}

/* smooth(): FV2_SWEEPS sweeps x -> TEMP -> x, each after a ghost fill of its source */
void fv2_smooth(const olevel *L, int smoother, int x_id, int rhs_id, double b)
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
  const double *rhs = cell0(L, rhs_id), *bi = cell0(L, V_BI), *bj = cell0(L, V_BJ), *bk = cell0(L, V_BK), *Dinv = cell0(L, V_DINV);
  const double *lam = smoother == FV2_L1JACOBI ? cell0(L, V_L1) : Dinv;
  for (int s = 0; s < FV2_SWEEPS; s++) {
    const int src = (s & 1) ? V_TEMP : x_id, dst = (s & 1) ? x_id : V_TEMP;
    fv2_fill(L, src);
    const double *xn = cell0(L, src);
    double *xp = cell0(L, dst);
    for (int k = 0; k < L->n; k++) for (int j = 0; j < L->n; j++) for (int i = 0; i < L->n; i++) {
      const int q = IDX(L, i, j, k);
      if (smoother == FV2_GSRB && ((i ^ j ^ k ^ s) & 1)) { xp[q] = xn[q]; continue; }   /* box low = (0,0,0) */
      const double Ax = fv2_op_ijk(xn, bi, bj, bk, q, L->jS, L->kS, b, h2inv);
      if (smoother == FV2_GSRB)       xp[q] = xn[q] + Dinv[q] * (rhs[q] - Ax);
      else if (smoother == FV2_CHEBY) xp[q] = xn[q] + c1[s % FV2_CHEBY_DEGREE] * (xn[q] - xp[q]) + c2[s % FV2_CHEBY_DEGREE] * Dinv[q] * (rhs[q] - Ax);
      else                            xp[q] = xn[q] + (weight * lam[q]) * (rhs[q] - Ax);
    }
  }
}

/* interpolation_p0: fine = prescale*fine + coarse parent */
void fv2_interpolation_p0(const olevel *Lf, int id_f, double prescale, const olevel *Lc, int id_c)
{
  const double *rd = cell0(Lc, id_c);
  double *wr = cell0(Lf, id_f);
  for (int k = 0; k < Lf->n; k++) for (int j = 0; j < Lf->n; j++) for (int i = 0; i < Lf->n; i++) {
    const int q = IDX(Lf, i, j, k);
    wr[q] = prescale * wr[q] + rd[IDX(Lc, i >> 1, j >> 1, k >> 1)];
  }
}
/* interpolation_v2 with the coarse BCs of this flavour: the oracle's own, except from a 1^3 level, where apply_BCs_v2 is v1 */
void fv2_interpolation_v2(const olevel *Lf, int id_f, double prescale, const olevel *Lc, int id_c)
{
  if (Lc->n >= 2) { oracle_interpolation_v2(Lf, id_f, prescale, Lc, id_c); return; }
  fv2_bc_v1(Lc, id_c, OR_SHAPE_BOX);
  const double *rd = cell0(Lc, id_c);
  double *wr = cell0(Lf, id_f);
  double fi[2][3][3], fj[2][2][3];
  for (int K = 0; K < 3; K++) for (int J = 0; J < 3; J++) pro(3, rd + IDX(Lc, 0, J - 1, K - 1), 1, &fi[0][J][K], &fi[1][J][K]);
  for (int K = 0; K < 3; K++) for (int I = 0; I < 2; I++) {
    double col[3] = { fi[I][0][K], fi[I][1][K], fi[I][2][K] };
    pro(3, col + 1, 1, &fj[I][0][K], &fj[I][1][K]);
  }
  for (int J = 0; J < 2; J++) for (int I = 0; I < 2; I++) {
    double col[3] = { fj[I][J][0], fj[I][J][1], fj[I][J][2] }, lo, hi;
    pro(3, col + 1, 1, &lo, &hi);
    double *w0 = wr + IDX(Lf, I, J, 0);
    w0[0] = prescale * w0[0] + lo;
    w0[Lf->kS] = prescale * w0[Lf->kS] + hi;
  }
}

/* rebuild_operator_blackbox(level, a, b, 2) (rebuild.c:47-208); the L1 row inverse is kept in V_L1 */
static void fv2_rebuild_blackbox(olevel *L, double a, double b)
{
  int colors = 2;
  if (L->n < colors) colors = L->n;
  const double h2inv = 1.0 / (L->h * L->h);
  zero_vec(L, V_DINV);  zero_vec(L, V_E);
  double *x = cell0(L, V_TEMP), *Aii = cell0(L, V_DINV), *sum = cell0(L, V_E), *l1 = cell0(L, V_L1);
  const double *bi = cell0(L, V_BI), *bj = cell0(L, V_BJ), *bk = cell0(L, V_BK);
  for (int kc = 0; kc < colors; kc++) for (int jc = 0; jc < colors; jc++) for (int ic = 0; ic < colors; ic++) {
    for (int k = 0; k < L->n; k++) for (int j = 0; j < L->n; j++) for (int i = 0; i < L->n; i++)
      x[IDX(L, i, j, k)] = (((i + ic) % colors) == 0 ? 1.0 : 0.0) * (((j + jc) % colors) == 0 ? 1.0 : 0.0) * (((k + kc) % colors) == 0 ? 1.0 : 0.0);
    fv2_fill(L, V_TEMP);
    for (int k = 0; k < L->n; k++) for (int j = 0; j < L->n; j++) for (int i = 0; i < L->n; i++) {
      const int q = IDX(L, i, j, k);
      const double Ax = fv2_op_ijk(x, bi, bj, bk, q, L->jS, L->kS, b, h2inv);
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
static void fv2_rebuild_operator(olevel *L, const olevel *from, double a, double b)
{
  if (from) {
    oracle_restriction(L, V_BI, from, V_BI, OR_RESTRICT_FACE_I);
    oracle_restriction(L, V_BJ, from, V_BJ, OR_RESTRICT_FACE_J);
    oracle_restriction(L, V_BK, from, V_BK, OR_RESTRICT_FACE_K);
  }
  fv2_rebuild_blackbox(L, a, b);
}

/* ---- bottom solvers over the fv2 operator: solvers/bicgstab.c:14-97 and the library's CG (oracle_cg.c) ---- */
int fv2_bicgstab(olevel *L, int x_id, int R_id, double b, double rtol)
{
  const int r0 = V_RESERVED, r = V_RESERVED + 1, p = V_RESERVED + 2, q = V_RESERVED + 3, s = V_RESERVED + 4, t = V_RESERVED + 5, Ap = V_RESERVED + 6, As = V_RESERVED + 7;
  int j = 0, failed = 0, converged = 0;
  fv2_residual(L, r0, x_id, R_id, b);
  scale_vec(L, r, 1.0, r0);
  scale_vec(L, p, 1.0, r0);
  double r_dot_r0 = dot_vec(L, r, r0), norm_of_r0 = oracle_norm(L, r);
  if (r_dot_r0 == 0.0) converged = 1;
  if (norm_of_r0 == 0.0) converged = 1;
  while (j < 200 && !failed && !converged) {
    j++;
    mul_vec(L, q, 1.0, V_DINV, p);
    fv2_apply_op(L, Ap, q, b);
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
    fv2_apply_op(L, As, t, b);
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
int fv2_cg(olevel *L, int x_id, int R_id, double b, double rtol)
{
  const int r0 = V_RESERVED, r = V_RESERVED + 1, p = V_RESERVED + 2, Ap = V_RESERVED + 3, z = V_RESERVED + 4;
  int j = 0, failed = 0, converged = 0;
  fv2_residual(L, r0, x_id, R_id, b);
  scale_vec(L, r, 1.0, r0);
  mul_vec(L, z, 1.0, V_DINV, r);
  scale_vec(L, p, 1.0, z);
  double r_dot_z = dot_vec(L, r, z), norm_of_r0 = oracle_norm(L, r);
  if (r_dot_z == 0.0) converged = 1;
  if (norm_of_r0 == 0.0) converged = 1;
  while (j < 200 && !failed && !converged) {
    j++;
    fv2_apply_op(L, Ap, p, b);
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

/* ---- cycles: mg.c:1135-1164 (MGVCycle), :1237-1344 (FMGSolve) ---- */
static int fv2_bottom(fv2hier *F, int x_id, int R_id)
{
  olevel *L = &F->H.L[F->H.nlevels - 1];
  return F->bottom == FV2_CG ? fv2_cg(L, x_id, R_id, F->H.b, 1e-3) : fv2_bicgstab(L, x_id, R_id, F->H.b, 1e-3);
}
static void fv2_vcycle(fv2hier *F, int e_id, int R_id, int l)
{
  ohier *H = &F->H;
  if (l == H->nlevels - 1) { H->krylov += fv2_bottom(F, e_id, R_id); return; }
  fv2_smooth(&H->L[l], F->smoother, e_id, R_id, H->b);
  fv2_residual(&H->L[l], V_TEMP, e_id, R_id, H->b);
  oracle_restriction(&H->L[l + 1], R_id, &H->L[l], V_TEMP, OR_RESTRICT_CELL);
  zero_vec(&H->L[l + 1], e_id);
  fv2_vcycle(F, e_id, R_id, l + 1);
  fv2_interpolation_p0(&H->L[l], e_id, 1.0, &H->L[l + 1], e_id);
  fv2_smooth(&H->L[l], F->smoother, e_id, R_id, H->b);
}
double fv2_fmg_solve(fv2hier *F, int onLevel, double *norm_of_F)
{
  ohier *H = &F->H;
  const int e_id = V_U, R_id = V_R, bottom = H->nlevels - 1;
  zero_vec(&H->L[onLevel], V_U);
  const double nF = oracle_norm(&H->L[onLevel], V_F);
  scale_vec(&H->L[onLevel], R_id, 1.0, V_F);
  for (int l = onLevel; l < bottom; l++) oracle_restriction(&H->L[l + 1], R_id, &H->L[l], R_id, OR_RESTRICT_CELL);
  if (bottom > onLevel) zero_vec(&H->L[bottom], e_id);
  H->krylov += fv2_bottom(F, e_id, R_id);
  for (int l = bottom - 1; l >= onLevel; l--) {
    fv2_interpolation_v2(&H->L[l], e_id, 0.0, &H->L[l + 1], e_id);
    fv2_vcycle(F, e_id, R_id, l);
  }
  fv2_residual(&H->L[onLevel], V_TEMP, e_id, V_F, H->b);
  if (norm_of_F) *norm_of_F = nF;
  return oracle_norm(&H->L[onLevel], V_TEMP);
}

/* hpgmg-fv.c:280-308 + MGBuild for `hpgmg-fv log2_dim 1` with the radius-1 stencil: 2^log2_dim ... 1 */
fv2hier *fv2_build(int log2_dim, int smoother, int bottom)
{
  fv2hier *F = (fv2hier *)calloc(1, sizeof(fv2hier));
  ohier *H = &F->H;
  F->smoother = smoother;  F->bottom = bottom;
  H->a = 0.0;  H->b = 1.0;  H->cheby = 0;
  H->nlevels = log2_dim + 1;
  H->L = (olevel *)calloc((size_t)H->nlevels, sizeof(olevel));
  for (int l = 0; l < H->nlevels; l++) level_init(&H->L[l], 1 << (log2_dim - l), V_RESERVED + 9);
  initialize_problem(&H->L[0], 1.0 / (double)(1 << log2_dim));
  fv2_rebuild_operator(&H->L[0], NULL, H->a, H->b);
  for (int l = 1; l < H->nlevels; l++) { H->L[l].h = 2.0 * H->L[l - 1].h; fv2_rebuild_operator(&H->L[l], &H->L[l - 1], H->a, H->b); }
  return F;
}
void fv2_destroy(fv2hier *F)
{
  for (int l = 0; l < F->H.nlevels; l++) level_free(&F->H.L[l]);
  free(F->H.L);
  free(F);
}

/* the driver's Richardson pass (hpgmg-fv.c:351-366) */
void fv2_richardson(fv2hier *F, double norms[3], double *err, double *order)
{
  ohier *H = &F->H;
  for (int l = 0; l < 3; l++) {
    if (l > 0) oracle_restriction(&H->L[l], V_F, &H->L[l - 1], V_F, OR_RESTRICT_CELL);
    norms[l] = fv2_fmg_solve(F, l, NULL);
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
ohier *fv2_hier(fv2hier *F) { return &F->H; }
void fv2_level_apply_op(fv2hier *F, int l, int Ax_id, int x_id) { fv2_apply_op(&F->H.L[l], Ax_id, x_id, F->H.b); }
void fv2_level_residual(fv2hier *F, int l, int res_id, int x_id, int rhs_id) { fv2_residual(&F->H.L[l], res_id, x_id, rhs_id, F->H.b); }
void fv2_level_smooth(fv2hier *F, int l, int x_id, int rhs_id) { fv2_smooth(&F->H.L[l], F->smoother, x_id, rhs_id, F->H.b); }
void fv2_level_interpolation_p0(fv2hier *F, int lf, int id_f, double prescale, int id_c) { fv2_interpolation_p0(&F->H.L[lf], id_f, prescale, &F->H.L[lf + 1], id_c); }
