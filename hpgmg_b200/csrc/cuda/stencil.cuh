/*
 * stencil.cuh -- the 4th-order variable-coefficient finite-volume operator at one cell.
 *
 * Restates the Poisson form of the reference macro apply_op_ijk (operators.fv4.c:87-114) with the
 * SAME association order, because the parity target is bit-for-bit agreement with the gcc -O2
 * (no FMA) build of the reference: C evaluates a+b+c as (a+b)+c, and the library is compiled
 * with -fmad=false so nvcc emits separate DMUL/DADD exactly as written here.
 *
 *   A x = -b h^-2 { 1/12 * SUM_6faces  beta_face * ( 15 (x_nbr - x) - (x_nbr2 - x_opp) )
 *                 + 1/48 * SUM_12      (transverse difference of beta_face) * (4-point mixed difference of x) }
 *
 * beta_d[ijk] is the coefficient on the LOW d-face of cell ijk.  25 x-points (axis +-1,+-2 and the
 * 12 in-plane diagonals: ghost faces + edges, never corners), 30 beta-points.
 *
 * The arithmetic is written ONCE, over four "loaders" X, BI, BJ, BK that return the value at an
 * offset (di,dj,dk) from the cell: the global-memory kernels pass pointer loaders, the tiled kernels
 * pass shared-memory loaders; both therefore produce identical bits.
 *
 * The smoothers' cell updates, the GSRB colouring and the smoothers' per-level coefficients live here too, so
 * that every kernel family (smooth.cu, stencil_tma.cuh, stencil_box.cuh, coarse.cu) evaluates the same expressions.
 */
#ifndef HPGMG_B200_STENCIL_CUH
#define HPGMG_B200_STENCIL_CUH

#include "hpgmg_b200.h"

/* what an operator kernel computes; kernel symbols are named by these values (stencil_tma_kernel<2,...> is the GSRB sweep) */
enum { OP_APPLY = 0, OP_RESIDUAL = 1, OP_GSRB = 2, OP_CHEBY = 3, OP_REBUILD = 4,
       OP_RESRES = 5,     /* residual fused with the cell restriction that follows it in MGVCycle (k-marching kernel only) */
       OP_JACOBI = 6 };   /* one Jacobi sweep: x + (weight*lambda)*(rhs - A x) */

#define STENCIL_TWELFTH (0.0833333333333333333)

/* aii (optional): the diagonal entry of A at this cell, i.e. the same expression evaluated on the unit vector
 * (x_c = 1, every other point 0) -- what rebuild_operator_blackbox (rebuild.c:127-133) accumulates into Aii for a
 * cell whose stencil does not reach a boundary-condition ghost cell: 15*(0-1)-(0-0) = -15 on each face, every
 * mixed difference (+-0)*beta = +-0, so Aii = -b*h2inv*(1/12 * SUM_faces beta*(-15)) with the faces added in the
 * macro's order.  Dinv = 1.0/Aii (rebuild.c:181) can then be formed in registers instead of being read. */
template <class XL, class BIL, class BJL, class BKL>
__device__ __forceinline__ double fv4_apply_op_at(const XL &X, const BIL &BI, const BJL &BJ, const BKL &BK, const double b, const double h2inv, double *aii = nullptr)
{
  const double xc = X(0, 0, 0);
  const double xw = X(-1, 0, 0), xe = X(1, 0, 0), xww = X(-2, 0, 0), xee = X(2, 0, 0);
  const double xs = X(0, -1, 0), xn = X(0, 1, 0), xss = X(0, -2, 0), xnn = X(0, 2, 0);
  const double xd = X(0, 0, -1), xu = X(0, 0, 1), xdd = X(0, 0, -2), xuu = X(0, 0, 2);
  const double xwn = X(-1, 1, 0), xws = X(-1, -1, 0), xen = X(1, 1, 0), xes = X(1, -1, 0);
  const double xwu = X(-1, 0, 1), xwd = X(-1, 0, -1), xeu = X(1, 0, 1), xed = X(1, 0, -1);
  const double xsu = X(0, -1, 1), xsd = X(0, -1, -1), xnu = X(0, 1, 1), xnd = X(0, 1, -1);

  const double bi0 = BI(0, 0, 0), bi1 = BI(1, 0, 0), bj0 = BJ(0, 0, 0), bj1 = BJ(0, 1, 0), bk0 = BK(0, 0, 0), bk1 = BK(0, 0, 1);
  const double axial =
      bi0 * (15.0 * (xw - xc) - (xww - xe))
    + bi1 * (15.0 * (xe - xc) - (xee - xw))
    + bj0 * (15.0 * (xs - xc) - (xss - xn))
    + bj1 * (15.0 * (xn - xc) - (xnn - xs))
    + bk0 * (15.0 * (xd - xc) - (xdd - xu))
    + bk1 * (15.0 * (xu - xc) - (xuu - xd));
  if (aii) {
    const double unit = bi0 * (-15.0) + bi1 * (-15.0) + bj0 * (-15.0) + bj1 * (-15.0) + bk0 * (-15.0) + bk1 * (-15.0);
    *aii = -b * h2inv * (STENCIL_TWELFTH * unit);
  }

  const double mixed =
      (BI(0, 1, 0) - BI(0, -1, 0)) * (xwn - xn - xws + xs)
    + (BI(0, 0, 1) - BI(0, 0, -1)) * (xwu - xu - xwd + xd)
    + (BJ(1, 0, 0) - BJ(-1, 0, 0)) * (xes - xe - xws + xw)
    + (BJ(0, 0, 1) - BJ(0, 0, -1)) * (xsu - xu - xsd + xd)
    + (BK(1, 0, 0) - BK(-1, 0, 0)) * (xed - xe - xwd + xw)
    + (BK(0, 1, 0) - BK(0, -1, 0)) * (xnd - xn - xsd + xs)

    + (BI(1, 1, 0) - BI(1, -1, 0)) * (xen - xn - xes + xs)
    + (BI(1, 0, 1) - BI(1, 0, -1)) * (xeu - xu - xed + xd)
    + (BJ(1, 1, 0) - BJ(-1, 1, 0)) * (xen - xe - xwn + xw)
    + (BJ(0, 1, 1) - BJ(0, 1, -1)) * (xnu - xu - xnd + xd)
    + (BK(1, 0, 1) - BK(-1, 0, 1)) * (xeu - xe - xwu + xw)
    + (BK(0, 1, 1) - BK(0, -1, 1)) * (xnu - xn - xsu + xs);

  return -b * h2inv * (STENCIL_TWELFTH * axial + 0.25 * STENCIL_TWELFTH * mixed);
}

/* The 2nd-order variable-coefficient finite-volume operator (operators.fv2.c), the 7-point star over the same loaders:
 *   A x = -b h^-2 ( beta_i[i+1]*(x[i+1]-x) + beta_i[i]*(x[i-1]-x) + the same in j and k ),  summed left to right in that order.
 * aii (optional): the same expression on the unit vector at this cell, as rebuild_operator_blackbox accumulates it where the
 * stencil does not reach a boundary-condition ghost cell. */
template <class XL, class BIL, class BJL, class BKL>
__device__ __forceinline__ double fv2_apply_op_at(const XL &X, const BIL &BI, const BJL &BJ, const BKL &BK, const double b, const double h2inv, double *aii = nullptr)
{
  const double xc = X(0, 0, 0);
  const double bi0 = BI(0, 0, 0), bi1 = BI(1, 0, 0), bj0 = BJ(0, 0, 0), bj1 = BJ(0, 1, 0), bk0 = BK(0, 0, 0), bk1 = BK(0, 0, 1);
  if (aii) *aii = -b * h2inv * (bi1 * (0.0 - 1.0) + bi0 * (0.0 - 1.0) + bj1 * (0.0 - 1.0) + bj0 * (0.0 - 1.0) + bk1 * (0.0 - 1.0) + bk0 * (0.0 - 1.0));
  return -b * h2inv * (bi1 * (X(1, 0, 0) - xc) + bi0 * (X(-1, 0, 0) - xc)
                     + bj1 * (X(0, 1, 0) - xc) + bj0 * (X(0, -1, 0) - xc)
                     + bk1 * (X(0, 0, 1) - xc) + bk0 * (X(0, 0, -1) - xc));
}

/* ---- the flavour: which operator the library is built for (-DHPGMG_FV2: operators.fv2.c, otherwise operators.fv4.c) ----
 * STENCIL_RADIUS is stencil_get_radius(), i.e. the ghost depth of every level MGBuild makes, and the only depth the flat
 * fill tables and the fast kernels are built for; levels of another depth take the list-walking kernels.
 * Values that could not be checked against operators.fv2.c are marked (unverified); each is defined here only.
 * Either operator combines with -DUSE_HELMHOLTZ (the Helmholtz vector map of hpgmg_defines.h and HELMHOLTZ_TERM below). */
#ifdef HPGMG_FV2
#define STENCIL_RADIUS      1
#define STENCIL_SHAPE       STENCIL_SHAPE_STAR
#define SMOOTH_SWEEPS       4      /* (unverified) GSRB NUM_SMOOTHS 2 (RBRB), Jacobi / L1-Jacobi 4 sweeps, Chebyshev = its degree */
#define CHEBYSHEV_DEGREE    4      /* (unverified) */
#define BLACKBOX_COLORS     2      /* rebuild_operator_blackbox(level, a, b, 2): no two cells of a colour in one radius-1 star */
#define SMOOTH_BC_VERSION   2      /* (unverified) apply_BCs = apply_BCs_v2 (v1 below 2^3) */
#else
#define STENCIL_RADIUS      2
#define STENCIL_SHAPE       STENCIL_SHAPE_NO_CORNERS
#define SMOOTH_SWEEPS       6      /* GSRB NUM_SMOOTHS 3 (RBRBRB), Jacobi NUM_SMOOTHS 6, Chebyshev degree 6 (operators.fv4.c:176-195) */
#define CHEBYSHEV_DEGREE    6
#define BLACKBOX_COLORS     4      /* operators.fv4.c:145-173 */
#define SMOOTH_BC_VERSION   4      /* apply_BCs = apply_BCs_v4 (v2 below 4^3) */
#endif
#define CHEBYSHEV_MAX_DEGREE 6

/* the operator of this flavour at one cell */
template <class XL, class BIL, class BJL, class BKL>
__device__ __forceinline__ double op_apply_at(const XL &X, const BIL &BI, const BJL &BJ, const BKL &BK, const double b, const double h2inv, double *aii = nullptr)
{
#ifdef HPGMG_FV2
  return fv2_apply_op_at(X, BI, BJ, BK, b, h2inv, aii);
#else
  return fv4_apply_op_at(X, BI, BJ, BK, b, h2inv, aii);
#endif
}

/* The Helmholtz build (-DUSE_HELMHOLTZ, as in the reference: operators.fv4.c:56-85, and operators.fv2.c in its Helmholtz form):
 * A x = a*alpha*x - b*h2inv*(...).  Written before the operator, HELMHOLTZ_TERM(a, alpha, x) op_apply_at(...) forms that sum.
 * The reference subtracts (b*h2inv)*(...) from a*alpha*x; op_apply_at returns (-b*h2inv)*(...), the exact negation, and
 * p - q == p + (-q) in IEEE arithmetic, so the sum has the reference's bits.  Without VECTOR_ALPHA the term is empty and
 * VECTOR_ALPHA_OR_0 only keeps the call sites compiling. */
#ifdef VECTOR_ALPHA
#define HELMHOLTZ_TERM(a, alpha, x) (a) * (alpha) * (x) +
#define VECTOR_ALPHA_OR_0 VECTOR_ALPHA
#else
#define HELMHOLTZ_TERM(a, alpha, x)
#define VECTOR_ALPHA_OR_0 0
#endif

/* loader over a global-memory array: p points at cell ijk */
struct GlobalLoader {
  const double *__restrict__ p;
  int jS, kS;
  __device__ __forceinline__ double operator()(const int di, const int dj, const int dk) const { return p[di + dj * jS + dk * kS]; }
};

/* x, bi, bj, bk point at cell ijk; jS/kS are the strides (doubles). Returns A x at ijk. */
__device__ __forceinline__ double fv4_apply_op(const double *__restrict__ x,
                                               const double *__restrict__ bi,
                                               const double *__restrict__ bj,
                                               const double *__restrict__ bk,
                                               const int jS, const int kS,
                                               const double b, const double h2inv)
{
  const GlobalLoader X = { x, jS, kS }, BI = { bi, jS, kS }, BJ = { bj, jS, kS }, BK = { bk, jS, kS };
  return fv4_apply_op_at(X, BI, BJ, BK, b, h2inv);
}

/* the same for the operator of this flavour */
__device__ __forceinline__ double op_apply(const double *__restrict__ x, const double *__restrict__ bi, const double *__restrict__ bj, const double *__restrict__ bk,
                                           const int jS, const int kS, const double b, const double h2inv)
{
  const GlobalLoader X = { x, jS, kS }, BI = { bi, jS, kS }, BJ = { bj, jS, kS }, BK = { bk, jS, kS };
  return op_apply_at(X, BI, BJ, BK, b, h2inv);
}

/* ---- the smoothers at one cell: x the cell's value before the sweep, Ax = (A x) there; the reference's association order ---- */
/* gsrb.c:41-129: x + Dinv*(rhs - Ax) */
__device__ __forceinline__ double gsrb_update(const double x, const double dinv, const double rhs, const double Ax)
{
  return x + dinv * (rhs - Ax);
}

/* chebyshev.c:90: x_n + c1*(x_n - x_{n-1}) + c2*Dinv*(rhs - Ax_n) */
__device__ __forceinline__ double chebyshev_update(const double x, const double xm1, const double c1, const double c2, const double dinv, const double rhs, const double Ax)
{
  return x + c1 * (x - xm1) + c2 * dinv * (rhs - Ax);
}

/* jacobi.c: x_n + weight*lambda*(rhs - Ax_n), left to right */
__device__ __forceinline__ double jacobi_update(const double x, const double weight, const double lam, const double rhs, const double Ax)
{
  return x + (weight * lam) * (rhs - Ax);
}

/* GSRB colouring (gsrb.c:55,100): cell (i,j,k) of box `box`, whose low corner is low[3 box .. 3 box + 2], is updated
 * on sweep s iff ((i ^ j ^ k ^ gsrb_box_parity(low, box, s)) & 1) == 0.  sweep is taken by reference so that, like the
 * corner, it is a load here: taken by value, the compiler orders the xors differently (same value, other instructions). */
__device__ __forceinline__ int gsrb_box_parity(const int *low, const int box, const int &sweep)
{
  return (low[3 * box] ^ low[3 * box + 1] ^ low[3 * box + 2] ^ sweep) & 1;
}

/* ---- the smoothers' per-level coefficients and operator codes (host) ---- */
/* Chebyshev coefficients of the `degree` steps (<= CHEBYSHEV_MAX_DEGREE), exactly as chebyshev.c:22-40 */
static inline void chebyshev_coefficients(const double dominant_eigenvalue_of_DinvA, const int degree, double c1[], double c2[])
{
  double beta = 1.000 * dominant_eigenvalue_of_DinvA;
  double alpha = 0.125000 * beta;
  double theta = 0.5 * (beta + alpha);
  double delta = 0.5 * (beta - alpha);
  double sigma = theta / delta;
  double rho_n = 1 / sigma;
  c1[0] = 0.0;
  c2[0] = 1 / theta;
  for (int s = 1; s < degree; s++) {
    double rho_nm1 = rho_n;
    rho_n = 1.0 / (2.0 * sigma - rho_nm1);
    c1[s] = rho_n * rho_nm1;
    c2[s] = rho_n * 2.0 / delta;
  }
}

/* jacobi.c: weight 2/3 with lambda = Dinv (USE_JACOBI), 1 with lambda = the L1 row inverse (USE_L1JACOBI) */
static inline double jacobi_weight(const int smoother)
{
  return smoother == HPGMG_SMOOTHER_L1JACOBI ? 1.0 : 2.0 / 3.0;
}

/* the sweep operator of a smoother (HPGMG_SMOOTHER_*) */
static inline int smoother_op(const int smoother)
{
  if (smoother == HPGMG_SMOOTHER_CHEBY) return OP_CHEBY;
  if (smoother == HPGMG_SMOOTHER_JACOBI || smoother == HPGMG_SMOOTHER_L1JACOBI) return OP_JACOBI;
  return OP_GSRB;
}

#endif
