/*
 * oracle_jacobi.c -- TEST INFRASTRUCTURE ONLY: the reference's weighted Jacobi and L1-Jacobi smoothers (operators/jacobi.c,
 * selected there with -DUSE_JACOBI / -DUSE_L1JACOBI, operators.fv4.c:176-195) on top of the plain-C oracle.
 *
 * The oracle (oracle/hpgmg_oracle.c) is included unchanged, so the setup, the operator, the boundary conditions, the
 * transfers and the BiCGStab bottom solver are its own; this file adds the smoother and the cycles that call it (the
 * oracle's MGVCycle / FMGSolve / Richardson pass with the smoother swapped, same order of operations).  It is compiled by
 * tests/oracle_jacobi.py with the oracle's flags (-O2 -ffp-contract=off); nothing under hpgmg_b200/ may use it.
 *
 * The L1 row inverse: the oracle's rebuild_blackbox leaves 1/Aii or 1/(Aii + sum|Aij|/2) (rebuild.c) in V_E; a copy is
 * kept in one more vector of every level, appended after the oracle's own (VECTOR_L1INV of the reference's -DUSE_L1JACOBI
 * map, defines.h:12-26).
 */
#include "../oracle/hpgmg_oracle.c"

#define OJ_JACOBI   2
#define OJ_L1JACOBI 3

/* the id of the appended L1-inverse vector of a level */
static int l1_id(const olevel *L) { return L->nvec - 1; }

/* jacobi.c: NUM_SMOOTHS 6; x ping-pongs through VECTOR_TEMP like GSRB; before each sweep exchange_boundary + apply_BCs on the
 * source; every cell x_np1 = x_n + weight*lambda*(rhs - Ax_n), evaluated left to right */
void oracle_smooth_jacobi(const olevel *L, int x_id, int rhs_id, double b, double weight, int lambda_id)
{
  const double h2inv = 1.0 / (L->h * L->h);
  const double *rhs = cell0(L, rhs_id), *bi = cell0(L, V_BI), *bj = cell0(L, V_BJ), *bk = cell0(L, V_BK), *lambda = cell0(L, lambda_id);
  for (int s = 0; s < 6; s++) {
    const int src = (s & 1) ? V_TEMP : x_id, dst = (s & 1) ? x_id : V_TEMP;
    fill_ghosts(L, src);
    const double *xn = cell0(L, src);
    double *xp = cell0(L, dst);
    for (int k = 0; k < L->n; k++) for (int j = 0; j < L->n; j++) for (int i = 0; i < L->n; i++) {
      const int ijk = IDX(L, i, j, k);
      const double Ax_n = apply_op_ijk(xn, bi, bj, bk, ijk, L->jS, L->kS, b, h2inv);
      xp[ijk] = xn[ijk] + weight * lambda[ijk] * (rhs[ijk] - Ax_n);
    }
  }
}

/* the hierarchy keeps its smoother in ohier::cheby (OJ_JACOBI or OJ_L1JACOBI here) */
static void jsmooth(const ohier *H, const olevel *L, int x_id, int rhs_id)
{
  if (H->cheby == OJ_L1JACOBI) oracle_smooth_jacobi(L, x_id, rhs_id, H->b, 1.0, l1_id(L));
  else                         oracle_smooth_jacobi(L, x_id, rhs_id, H->b, 2.0 / 3.0, V_DINV);
}

/* oracle_build + a copy of the L1 inverse on every level; smoother: OJ_JACOBI or OJ_L1JACOBI */
ohier *oracle_jacobi_build(int log2_dim, int smoother)
{
  ohier *H = oracle_build(log2_dim, 0);
  H->cheby = smoother;
  for (int l = 0; l < H->nlevels; l++) {
    olevel *L = &H->L[l];
    L->v = (double **)realloc(L->v, (size_t)(L->nvec + 1) * sizeof(double *));
    L->v[L->nvec] = (double *)malloc((size_t)L->vol * sizeof(double));
    memcpy(L->v[L->nvec], L->v[V_E], (size_t)L->vol * sizeof(double));
    L->nvec++;
  }
  return H;
}

/* mg.c:1135-1164, as vcycle() of the oracle */
static void jvcycle(ohier *H, int e_id, int R_id, int l)
{
  if (l == H->nlevels - 1) { H->krylov += bicgstab(&H->L[l], e_id, R_id, H->b, 1e-3); return; }
  jsmooth(H, &H->L[l], e_id, R_id);
  oracle_residual(&H->L[l], V_TEMP, e_id, R_id, H->b);
  oracle_restriction(&H->L[l + 1], R_id, &H->L[l], V_TEMP, OR_RESTRICT_CELL);
  zero_vec(&H->L[l + 1], e_id);
  jvcycle(H, e_id, R_id, l + 1);
  oracle_interpolation_v2(&H->L[l], e_id, 1.0, &H->L[l + 1], e_id);
  jsmooth(H, &H->L[l], e_id, R_id);
}

/* mg.c:1237-1344, as oracle_fmg_solve() */
double oracle_jacobi_fmg_solve(ohier *H, int onLevel, double *norm_of_F)
{
  const int e_id = V_U, R_id = V_R, bottom = H->nlevels - 1;
  zero_vec(&H->L[onLevel], V_U);
  const double nF = oracle_norm(&H->L[onLevel], V_F);
  scale_vec(&H->L[onLevel], R_id, 1.0, V_F);
  for (int l = onLevel; l < bottom; l++) oracle_restriction(&H->L[l + 1], R_id, &H->L[l], R_id, OR_RESTRICT_CELL);
  if (bottom > onLevel) zero_vec(&H->L[bottom], e_id);
  H->krylov += bicgstab(&H->L[bottom], e_id, R_id, H->b, 1e-3);
  for (int l = bottom - 1; l >= onLevel; l--) {
    oracle_interpolation_v4(&H->L[l], e_id, 0.0, &H->L[l + 1], e_id);
    jvcycle(H, e_id, R_id, l);
  }
  oracle_residual(&H->L[onLevel], V_TEMP, e_id, V_F, H->b);
  if (norm_of_F) *norm_of_F = nF;
  return oracle_norm(&H->L[onLevel], V_TEMP);
}

/* hpgmg-fv.c:351-366, mg.c:1113-1131, as oracle_richardson() */
void oracle_jacobi_richardson(ohier *H, double norms[3], double *err, double *order)
{
  for (int l = 0; l < 3; l++) {
    if (l > 0) oracle_restriction(&H->L[l], V_F, &H->L[l - 1], V_F, OR_RESTRICT_CELL);
    norms[l] = oracle_jacobi_fmg_solve(H, l, NULL);
  }
  oracle_restriction(&H->L[1], V_TEMP, &H->L[0], V_U, OR_RESTRICT_CELL);
  oracle_restriction(&H->L[2], V_TEMP, &H->L[1], V_U, OR_RESTRICT_CELL);
  add_vec(&H->L[1], V_TEMP, 1.0, V_U, -1.0, V_TEMP);
  add_vec(&H->L[2], V_TEMP, 1.0, V_U, -1.0, V_TEMP);
  const double e2h = oracle_norm(&H->L[1], V_TEMP), e4h = oracle_norm(&H->L[2], V_TEMP);
  *err = e2h;
  *order = log(e4h / e2h) / log(2);
}

int oracle_jacobi_l1inv_id(ohier *H, int level) { return l1_id(&H->L[level]); }
