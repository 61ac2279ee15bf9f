/*
 * bicgstab.cuh -- device bodies of the single-thread-block bottom solvers, BiCGStab and CG (see bicgstab.cu), shared with
 * the coarse-grid cycle kernel (coarse.cu).
 */
#ifndef HPGMG_B200_BICGSTAB_CUH
#define HPGMG_B200_BICGSTAB_CUH
#include <math.h>
#include "common.cuh"
#include "stencil.cuh"
#include "bc.cuh"

#define BOTTOM_MAX_DIM   11
#define BOTTOM_MAX_CELLS (BOTTOM_MAX_DIM * BOTTOM_MAX_DIM * BOTTOM_MAX_DIM)
#define BOTTOM_THREADS   256   /* the stand-alone kernel; the body works for any 1-D block that is a multiple of 32 (<=1024) */

/* which vector of L plays which role: the identity (vector ids of the reference, bicgstab.c:17-24, defines.h:28-38) for the
 * stand-alone kernel; the coarse-cycle kernel keeps only the vectors a cycle touches in shared memory and passes their slots.
 * alpha (Helmholtz builds) is set by the identity only: the coarse-cycle kernel does not run in those builds. */
struct BottomIds {
  int r0, r, p, q, s, t, Ap, As;
  int dinv, temp, beta_i, beta_j, beta_k;
#ifdef VECTOR_ALPHA
  int alpha;
#endif
};
__host__ __device__ __forceinline__ BottomIds bottom_ids_identity()
{
  BottomIds I = { VECTORS_RESERVED + 0, VECTORS_RESERVED + 1, VECTORS_RESERVED + 2, VECTORS_RESERVED + 3, VECTORS_RESERVED + 4, VECTORS_RESERVED + 5,
                  VECTORS_RESERVED + 6, VECTORS_RESERVED + 7, VECTOR_DINV, VECTOR_TEMP, VECTOR_BETA_I, VECTOR_BETA_J, VECTOR_BETA_K,
#ifdef VECTOR_ALPHA
                  VECTOR_ALPHA
#endif
                };
  return I;
}

struct BottomArgs {
  DLevel L;
  const FillBC *bc;             /* BC columns of the flavour's stencil shape (NO_CORNERS; fv2: STAR) of the (single) box: flat table (device_level.cu); offsets are relative to a vector's start */
  int nbc;
  int x_id, R_id;
  BottomIds ids;
  double a, b, h2inv, rtol;
  double *iters;                /* device scalar slot: iterations are added to it */
};

struct BottomCtx {
  const BottomArgs &A;
  double *prod;                 /* shared: BOTTOM_MAX_CELLS products / scratch */
  double *red;                  /* shared: per-warp partials + broadcast slot  */
  int n, cells, jS, kS;
  int flip;                     /* which pair of result slots (red[32..33] / red[34..35]) the next reduction uses */
  __device__ int cell_offset(int c) const { return (c % n) + ((c / n) % n) * jS + (c / (n * n)) * kS; }
};

__device__ static void b_fill_ghosts(const BottomCtx &C, const int id)
{
  const DLevel &L = C.A.L;
  double *v = L.base + (size_t)id * (size_t)L.volume;
#ifdef HPGMG_FV2
  /* fv2: apply_BCs_v2 on the STAR shape, one ghost layer (nothing deeper to zero); v1 on a 1^3 box (boundary_fv.c:6-90: a face
   * ghost cell is minus the cell behind it) */
  const bool v1 = C.n < 2;
  for (int e = threadIdx.x; e < C.A.nbc; e += blockDim.x) {
    const FillBC it = C.A.bc[e];
    const BCNormal N = bc_normal(it.subtype, L.jStride, L.kStride);
    if (v1) v[it.dst] = -1.0 * v[it.src + N.d[0]];
    else    bc_v2_col(v + it.src, v + it.dst, N.m, N.d[0], N.d[1], N.d[2]);
  }
#else
  /* exchange_boundary is empty for a single box with Dirichlet BCs; apply_BCs = v4 (v2 if dim<4) */
  const bool v2 = C.n < 4;
  for (int e = threadIdx.x; e < C.A.nbc; e += blockDim.x) {
    const FillBC it = C.A.bc[e];
    const BCNormal N = bc_normal(it.subtype, L.jStride, L.kStride);
    if (v2) bc_v2_col_zero_rest(v + it.src, v + it.dst, N.m, N.d[0], N.d[1], N.d[2]);
    else    bc_v4_column(v + it.src, v + it.dst, N);
  }
#endif
  __syncthreads();
}

/* out = A in   (mode 0)   or   out = rhs - A in   (mode 1); A carries a*alpha in the Helmholtz builds */
__device__ static void b_apply(const BottomCtx &C, const int out_id, const int in_id, const int rhs_id, const int mode)
{
  b_fill_ghosts(C, in_id);
  const DLevel &L = C.A.L;
  const double *x = L.vec(0, in_id), *bi = L.vec(0, C.A.ids.beta_i), *bj = L.vec(0, C.A.ids.beta_j), *bk = L.vec(0, C.A.ids.beta_k);
  double *out = L.vec(0, out_id);
  const double *rhs = L.vec(0, rhs_id);
#ifdef VECTOR_ALPHA
  const double *alpha = L.vec(0, C.A.ids.alpha);
#endif
  for (int c = threadIdx.x; c < C.cells; c += blockDim.x) {
    const int ijk = C.cell_offset(c);
    const double Ax = HELMHOLTZ_TERM(C.A.a, alpha[ijk], x[ijk]) op_apply(x + ijk, bi + ijk, bj + ijk, bk + ijk, C.jS, C.kS, C.A.b, C.A.h2inv);
    out[ijk] = mode ? rhs[ijk] - Ax : Ax;
  }
  __syncthreads();
}

/* Every helper ends with ONE block barrier after its last write (reductions: two, around the serial sum), so that the next
 * helper may read anything; independent updates share a barrier.  Reduction results alternate between two shared slots, which
 * makes a third barrier (result read before the slot is written again) unnecessary.  The arithmetic of every cell and the
 * order of every sum are those of solvers/bicgstab.c + operators/misc.c. */

/* c = sa*a + sb*b  and  e = sd*d + sf*f   (two independent updates) */
__device__ static void b_add2(const BottomCtx &C, const int c_id, const double sa, const int a_id, const double sb, const int b_id,
                              const int e_id, const double sd, const int d_id, const double sf, const int f_id)
{
  const DLevel &L = C.A.L;
  double *c = L.vec(0, c_id), *e = L.vec(0, e_id);
  const double *a = L.vec(0, a_id), *b = L.vec(0, b_id), *d = L.vec(0, d_id), *f = L.vec(0, f_id);
  for (int q = threadIdx.x; q < C.cells; q += blockDim.x) {
    const int ijk = C.cell_offset(q);
    c[ijk] = sa * a[ijk] + sb * b[ijk];
    e[ijk] = sd * d[ijk] + sf * f[ijk];
  }
  __syncthreads();
}
/* c = sa*a + sb*b, then e = sd*d + sf*c  (the second reads the first's result in the same cell) */
__device__ static void b_add_chain(const BottomCtx &C, const int c_id, const double sa, const int a_id, const double sb, const int b_id,
                                   const int e_id, const double sd, const int d_id, const double sf)
{
  const DLevel &L = C.A.L;
  double *c = L.vec(0, c_id), *e = L.vec(0, e_id);
  const double *a = L.vec(0, a_id), *b = L.vec(0, b_id), *d = L.vec(0, d_id);
  for (int q = threadIdx.x; q < C.cells; q += blockDim.x) {
    const int ijk = C.cell_offset(q);
    const double v = sa * a[ijk] + sb * b[ijk];
    c[ijk] = v;
    e[ijk] = sd * d[ijk] + sf * v;
  }
  __syncthreads();
}
__device__ static void b_scale2(const BottomCtx &C, const int c_id, const int e_id, const double sa, const int a_id)
{
  const DLevel &L = C.A.L;
  double *c = L.vec(0, c_id), *e = L.vec(0, e_id);
  const double *a = L.vec(0, a_id);
  for (int q = threadIdx.x; q < C.cells; q += blockDim.x) {
    const int ijk = C.cell_offset(q);
    const double v = sa * a[ijk];
    c[ijk] = v;
    e[ijk] = v;
  }
  __syncthreads();
}
__device__ static void b_mul(const BottomCtx &C, const int c_id, const double s, const int a_id, const int b_id)
{
  const DLevel &L = C.A.L;
  double *c = L.vec(0, c_id);
  const double *a = L.vec(0, a_id), *b = L.vec(0, b_id);
  for (int q = threadIdx.x; q < C.cells; q += blockDim.x) {
    const int ijk = C.cell_offset(q);
    c[ijk] = s * a[ijk] * b[ijk];
  }
  __syncthreads();
}

/* dot(a,b) [and dot(a,d) if d_id >= 0]: products staged in shared memory, each sum by ONE thread in linear cell order
 * (k,j,i: the reference's order on one tile) */
__device__ static double b_dot(BottomCtx &C, const int a_id, const int b_id, const int d_id = -1, double *second = nullptr)
{
  const DLevel &L = C.A.L;
  const double *a = L.vec(0, a_id), *b = L.vec(0, b_id), *d = d_id >= 0 ? L.vec(0, d_id) : nullptr;
  double *prod2 = C.prod + C.cells;                              /* callers pass d_id only when 2*cells fit (bicgstab_solve) */
  for (int q = threadIdx.x; q < C.cells; q += blockDim.x) {
    const int ijk = C.cell_offset(q);
    C.prod[q] = a[ijk] * b[ijk];
    if (d) prod2[q] = a[ijk] * d[ijk];
  }
  __syncthreads();
  const int slot = 32 + 2 * C.flip;
  if (threadIdx.x == 0) {
    double s = 0.0;
    for (int q = 0; q < C.cells; q++) s += C.prod[q];
    C.red[slot] = s;
  } else if (d && threadIdx.x == 32) {
    double s = 0.0;
    for (int q = 0; q < C.cells; q++) s += prod2[q];
    C.red[slot + 1] = s;
  }
  __syncthreads();
  C.flip ^= 1;
  if (second) *second = C.red[slot + 1];
  return C.red[slot];
}

/* max |a| over the cells; m: this thread's partial maximum (callers that have just produced the values pass it) */
__device__ static double b_max(BottomCtx &C, double m)
{
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const double other = __shfl_down_sync(0xffffffffu, m, o);
    if (other > m) m = other;
  }
  if ((threadIdx.x & 31) == 0) C.red[threadIdx.x >> 5] = m;
  __syncthreads();
  const int slot = 32 + 2 * C.flip;
  if (threadIdx.x == 0) {
    for (int w = 1; w < (int)(blockDim.x >> 5); w++) if (C.red[w] > m) m = C.red[w];
    C.red[slot] = m;
  }
  __syncthreads();
  C.flip ^= 1;
  return C.red[slot];
}
__device__ static double b_norm(BottomCtx &C, const int a_id)
{
  const double *a = C.A.L.vec(0, a_id);
  double m = 0.0;
  for (int q = threadIdx.x; q < C.cells; q += blockDim.x) {
    const double f = fabs(a[C.cell_offset(q)]);
    if (f > m) m = f;
  }
  return b_max(C, m);
}
/* c = sa*a + sb*b; e = sd*d + sf*f; returns max |e| */
__device__ static double b_add2_norm(BottomCtx &C, const int c_id, const double sa, const int a_id, const double sb, const int b_id,
                                     const int e_id, const double sd, const int d_id, const double sf, const int f_id)
{
  const DLevel &L = C.A.L;
  double *c = L.vec(0, c_id), *e = L.vec(0, e_id);
  const double *a = L.vec(0, a_id), *b = L.vec(0, b_id), *d = L.vec(0, d_id), *f = L.vec(0, f_id);
  double m = 0.0;
  for (int q = threadIdx.x; q < C.cells; q += blockDim.x) {
    const int ijk = C.cell_offset(q);
    c[ijk] = sa * a[ijk] + sb * b[ijk];
    const double v = sd * d[ijk] + sf * f[ijk];
    e[ijk] = v;
    const double av = fabs(v);
    if (av > m) m = av;
  }
  return b_max(C, m);                                            /* its barriers also publish c and e */
}

/* the whole solve, executed cooperatively by all threads of the calling thread block;
 * prod: BOTTOM_MAX_CELLS doubles of shared memory, red: 36 doubles of shared memory */
__device__ static void bicgstab_solve(const BottomArgs &A, double *prod, double *red)
{
  BottomCtx C = { A, prod, red, A.L.dim, A.L.dim * A.L.dim * A.L.dim, A.L.jStride, A.L.kStride, 0 };

  const int r0 = A.ids.r0, r = A.ids.r, p = A.ids.p, q = A.ids.q, s = A.ids.s, t = A.ids.t, Ap = A.ids.Ap, As = A.ids.As;
  const int DINV = A.ids.dinv, TEMP = A.ids.temp;
  const int x_id = A.x_id;
  const int jMax = 200;
  const bool two_dots = 2 * C.cells <= BOTTOM_MAX_CELLS;            /* room for a second product array */
  int j = 0;
  bool failed = false, converged = false;

  b_apply(C, r0, x_id, A.R_id, 1);                        /* r0 = R - A x */
  b_scale2(C, r, p, 1.0, r0);                             /* r = r0; p = r0 */
  double r_dot_r0 = b_dot(C, r, r0);
  const double norm_of_r0 = b_norm(C, r);
  if (r_dot_r0 == 0.0) converged = true;
  if (norm_of_r0 == 0.0) converged = true;
  while ((j < jMax) && !failed && !converged) {
    j++;
    b_mul(C, q, 1.0, DINV, p);                     /* q = D^-1 p */
    b_apply(C, Ap, q, 0, 0);                              /* Ap = A q   */
    const double Ap_dot_r0 = b_dot(C, Ap, r0);
    if (Ap_dot_r0 == 0.0) { failed = true; break; }
    const double alpha = r_dot_r0 / Ap_dot_r0;
    if (isinf(alpha)) { failed = true; break; }
    const double norm_of_s = b_add2_norm(C, x_id, 1.0, x_id, alpha, q, s, 1.0, r, -alpha, Ap);      /* x += alpha q; s = r - alpha Ap */
    if (norm_of_s == 0.0) { converged = true; break; }
    if (norm_of_s < A.rtol * norm_of_r0) { converged = true; break; }
    b_mul(C, t, 1.0, DINV, s);                     /* t = D^-1 s */
    b_apply(C, As, t, 0, 0);                              /* As = A t   */
    double As_dot_s;
    double As_dot_As;
    if (two_dots) As_dot_As = b_dot(C, As, As, s, &As_dot_s);
    else { As_dot_As = b_dot(C, As, As); As_dot_s = b_dot(C, As, s); }
    if (As_dot_As == 0.0) { converged = true; break; }
    const double omega = As_dot_s / As_dot_As;
    if (omega == 0.0) { failed = true; break; }
    if (isinf(omega)) { failed = true; break; }
    const double norm_of_r = b_add2_norm(C, x_id, 1.0, x_id, omega, t, r, 1.0, s, -omega, As);      /* x += omega t; r = s - omega As */
    if (norm_of_r == 0.0) { converged = true; break; }
    if (norm_of_r < A.rtol * norm_of_r0) { converged = true; break; }
    const double r_dot_r0_new = b_dot(C, r, r0);
    if (r_dot_r0_new == 0.0) { failed = true; break; }
    const double beta = (r_dot_r0_new / r_dot_r0) * (alpha / omega);
    if (isinf(beta)) { failed = true; break; }
    b_add_chain(C, TEMP, 1.0, p, -omega, Ap, p, 1.0, r, beta);      /* TEMP = p - omega Ap; p = r + beta TEMP */
    r_dot_r0 = r_dot_r0_new;
  }
  if (threadIdx.x == 0) atomicAdd(A.iters, (double)j);
}

/* ---- CG (solvers/cg.c) ------------------------------------------------------------------------------------------------ */
/* the sum of C.prod[0..cells) by ONE thread in linear cell order, after the barrier that publishes the products (b_dot's order) */
__device__ static double b_sum_staged(BottomCtx &C)
{
  __syncthreads();
  const int slot = 32 + 2 * C.flip;
  if (threadIdx.x == 0) {
    double s = 0.0;
    for (int q = 0; q < C.cells; q++) s += C.prod[q];
    C.red[slot] = s;
  }
  __syncthreads();
  C.flip ^= 1;
  return C.red[slot];
}
/* c = sa*a + sb*b */
__device__ static void b_add(const BottomCtx &C, const int c_id, const double sa, const int a_id, const double sb, const int b_id)
{
  const DLevel &L = C.A.L;
  double *c = L.vec(0, c_id);
  const double *a = L.vec(0, a_id), *b = L.vec(0, b_id);
  for (int q = threadIdx.x; q < C.cells; q += blockDim.x) {
    const int ijk = C.cell_offset(q);
    c[ijk] = sa * a[ijk] + sb * b[ijk];
  }
  __syncthreads();
}
/* out = A in, returns dot(out, in): the products are staged in the pass that produces out */
__device__ static double b_apply_dot(BottomCtx &C, const int out_id, const int in_id)
{
  b_fill_ghosts(C, in_id);
  const DLevel &L = C.A.L;
  const double *x = L.vec(0, in_id), *bi = L.vec(0, C.A.ids.beta_i), *bj = L.vec(0, C.A.ids.beta_j), *bk = L.vec(0, C.A.ids.beta_k);
  double *out = L.vec(0, out_id);
#ifdef VECTOR_ALPHA
  const double *alpha = L.vec(0, C.A.ids.alpha);
#endif
  for (int c = threadIdx.x; c < C.cells; c += blockDim.x) {
    const int ijk = C.cell_offset(c);
    const double Ax = HELMHOLTZ_TERM(C.A.a, alpha[ijk], x[ijk]) op_apply(x + ijk, bi + ijk, bj + ijk, bk + ijk, C.jS, C.kS, C.A.b, C.A.h2inv);
    out[ijk] = Ax;
    C.prod[c] = Ax * x[ijk];
  }
  return b_sum_staged(C);
}
/* z = s*d*r, returns dot(r, z): the products are staged in the pass that writes z */
__device__ static double b_mul_dot(BottomCtx &C, const int z_id, const double s, const int d_id, const int r_id)
{
  const DLevel &L = C.A.L;
  double *z = L.vec(0, z_id);
  const double *d = L.vec(0, d_id), *r = L.vec(0, r_id);
  for (int q = threadIdx.x; q < C.cells; q += blockDim.x) {
    const int ijk = C.cell_offset(q);
    const double v = s * d[ijk] * r[ijk];
    z[ijk] = v;
    C.prod[q] = r[ijk] * v;
  }
  return b_sum_staged(C);
}
/* the start of CG in one pass: r = 1.0*r0; z = 1.0*d*r; p = 1.0*z; returns dot(r, z) and, in *norm_r, max |r| */
__device__ static double b_cg_start(BottomCtx &C, const int r_id, const int z_id, const int p_id, const int r0_id, const int d_id, double *norm_r)
{
  const DLevel &L = C.A.L;
  double *r = L.vec(0, r_id), *z = L.vec(0, z_id), *p = L.vec(0, p_id);
  const double *r0 = L.vec(0, r0_id), *d = L.vec(0, d_id);
  double m = 0.0;
  for (int q = threadIdx.x; q < C.cells; q += blockDim.x) {
    const int ijk = C.cell_offset(q);
    const double rv = 1.0 * r0[ijk];
    const double zv = 1.0 * d[ijk] * rv;
    r[ijk] = rv;
    z[ijk] = zv;
    p[ijk] = 1.0 * zv;
    C.prod[q] = rv * zv;
    const double f = fabs(rv);
    if (f > m) m = f;
  }
  const double r_dot_z = b_sum_staged(C);
  *norm_r = b_max(C, m);
  return r_dot_z;
}

/* D^-1-preconditioned CG, the restatement of solvers.c:cg_host_driven, executed cooperatively by all threads of the calling
 * thread block; prod: BOTTOM_MAX_CELLS doubles of shared memory, red: 36 doubles of shared memory.
 * Vectors: r0, r, p of BottomIds play themselves, q plays Ap and s plays z (the ids of cg.c, VECTORS_RESERVED+0..4).
 * Block barriers per iteration: 8 (ghost fill of p 1, Ap with the Ap.p sum 2, x/r update with max|r| 2, z with the r.z sum 2,
 * p update 1). */
__device__ static void cg_solve(const BottomArgs &A, double *prod, double *red)
{
  BottomCtx C = { A, prod, red, A.L.dim, A.L.dim * A.L.dim * A.L.dim, A.L.jStride, A.L.kStride, 0 };

  const int r0 = A.ids.r0, r = A.ids.r, p = A.ids.p, Ap = A.ids.q, z = A.ids.s;
  const int DINV = A.ids.dinv;
  const int x_id = A.x_id;
  const int jMax = 200;
  int j = 0;
  bool failed = false, converged = false;

  b_apply(C, r0, x_id, A.R_id, 1);                        /* r0 = R - A x */
  double norm_of_r0;
  double r_dot_z = b_cg_start(C, r, z, p, r0, DINV, &norm_of_r0);     /* r = r0; z = D^-1 r; p = z */
  if (r_dot_z == 0.0) converged = true;
  if (norm_of_r0 == 0.0) converged = true;
  while ((j < jMax) && !failed && !converged) {
    j++;
    const double Ap_dot_p = b_apply_dot(C, Ap, p);       /* Ap = A p */
    if (Ap_dot_p == 0.0) { failed = true; break; }
    const double alpha = r_dot_z / Ap_dot_p;
    if (isinf(alpha)) { failed = true; break; }
    const double norm_of_r = b_add2_norm(C, x_id, 1.0, x_id, alpha, p, r, 1.0, r, -alpha, Ap);      /* x += alpha p; r -= alpha Ap */
    if (norm_of_r == 0.0) { converged = true; break; }
    if (norm_of_r < A.rtol * norm_of_r0) { converged = true; break; }
    const double r_dot_z_new = b_mul_dot(C, z, 1.0, DINV, r);   /* z = D^-1 r */
    if (r_dot_z_new == 0.0) { failed = true; break; }
    const double beta = r_dot_z_new / r_dot_z;
    if (isinf(beta)) { failed = true; break; }
    b_add(C, p, 1.0, z, beta, p);                         /* p = z + beta p */
    r_dot_z = r_dot_z_new;
  }
  if (threadIdx.x == 0) atomicAdd(A.iters, (double)j);
}


#endif
