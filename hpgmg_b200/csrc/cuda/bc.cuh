/*
 * bc.cuh -- device bodies of the homogeneous-Dirichlet ghost-cell extrapolations, shared by the
 * list-walking kernels (ghost.cu), the single-block bottom solver (bicgstab.cuh) and the coarse-cycle
 * kernel (coarse.cu).  Reference: operators/boundary_fv.c:101-250 (quadratic), :262-569 (quartic).
 *
 * Unit of work = one COLUMN: one tangential position of a BC region.  Along each axis that is normal
 * to the domain boundary the column owns the 2 ghost cells and reads the 4 (v4) or 2 (v2) interior
 * cells behind them.  With M normal axes (1 face, 2 edge, 3 corner) the quartic version gathers 4^M
 * values and extrapolates axis by axis in ascending axis order -- the order of the reference's
 * face / 16-point edge (:404-425) / 64-point corner (:507-565) code -- so results are bit-identical.
 */
#ifndef HPGMG_B200_BC_CUH
#define HPGMG_B200_BC_CUH
#include "common.cuh"

/* 1-D quartic extrapolation of cell averages through a zero Dirichlet face (boundary_fv.c:339-340):
 * x1..x4 are the four cells nearest the boundary; near/far are the first/second ghost cell. */
__device__ __forceinline__ void quartic_pair(const double x1, const double x2, const double x3, const double x4, double &near, double &far)
{
  const double OneTwelfth = 1.0 / 12.0;
  near = OneTwelfth * (-77.0 * x1 + 43.0 * x2 - 17.0 * x3 + 3.0 * x4);
  far  = OneTwelfth * (-505.0 * x1 + 335.0 * x2 - 145.0 * x3 + 27.0 * x4);
}

/* ---- one column, quartic ------------------------------------------------------------------------ */
/* w points at the column's nearest ghost cell; r points at the SAME position in the array the interior
 * values are read from: the box itself, or -- when the column's tangential coordinates lie in a ghost
 * region that exchange_boundary would fill -- the image of that position inside the neighbouring
 * box (fused ghost fill, ghost.cu: same values, no dependency on the copy).  d0<d1<d2 (axis order) are
 * the inward strides of the normal axes; both boxes share the strides. */
/* e0<e1<e2: the same strides in the array that is written (they differ from d* when the column is written into a
 * staged shared-memory tile, stencil_box.cuh) */
__device__ __forceinline__ void bc_v4_col1(const double *r, double *w, const int d0, const int e0)
{
  double n, f;
  quartic_pair(r[d0], r[2 * d0], r[3 * d0], r[4 * d0], n, f);
  w[0] = n;
  w[-e0] = f;
}
__device__ __forceinline__ void bc_v4_col2(const double *r, double *w, const int d0, const int d1, const int e0, const int e1)
{
  double n[4], f[4];
#pragma unroll
  for (int J = 0; J < 4; J++) {
    const double *o = r + (J + 1) * d1;
    quartic_pair(o[d0], o[2 * d0], o[3 * d0], o[4 * d0], n[J], f[J]);
  }
  double nn, nf, fn, ff;
  quartic_pair(n[0], n[1], n[2], n[3], nn, nf);
  quartic_pair(f[0], f[1], f[2], f[3], fn, ff);
  w[0] = nn;
  w[-e1] = nf;
  w[-e0] = fn;
  w[-e0 - e1] = ff;
}
__device__ __forceinline__ void bc_v4_col3(const double *r, double *w, const int d0, const int d1, const int d2, const int e0, const int e1, const int e2)
{
  double nn[4], nf[4], fn[4], ff[4];
#pragma unroll
  for (int K = 0; K < 4; K++) {
    double n[4], f[4];
#pragma unroll
    for (int J = 0; J < 4; J++) {
      const double *o = r + (J + 1) * d1 + (K + 1) * d2;
      quartic_pair(o[d0], o[2 * d0], o[3 * d0], o[4 * d0], n[J], f[J]);
    }
    quartic_pair(n[0], n[1], n[2], n[3], nn[K], nf[K]);
    quartic_pair(f[0], f[1], f[2], f[3], fn[K], ff[K]);
  }
  double nnn, nnf, nfn, nff, fnn, fnf, ffn, fff;
  quartic_pair(nn[0], nn[1], nn[2], nn[3], nnn, nnf);
  quartic_pair(nf[0], nf[1], nf[2], nf[3], nfn, nff);
  quartic_pair(fn[0], fn[1], fn[2], fn[3], fnn, fnf);
  quartic_pair(ff[0], ff[1], ff[2], ff[3], ffn, fff);
  w[0] = nnn;
  w[-e2] = nnf;
  w[-e1] = nfn;
  w[-e1 - e2] = nff;
  w[-e0] = fnn;
  w[-e0 - e2] = fnf;
  w[-e0 - e1] = ffn;
  w[-e0 - e1 - e2] = fff;
}
__device__ __forceinline__ void bc_v4_col1(const double *r, double *w, const int d0) { bc_v4_col1(r, w, d0, d0); }
__device__ __forceinline__ void bc_v4_col2(const double *r, double *w, const int d0, const int d1) { bc_v4_col2(r, w, d0, d1, d0, d1); }
__device__ __forceinline__ void bc_v4_col3(const double *r, double *w, const int d0, const int d1, const int d2) { bc_v4_col3(r, w, d0, d1, d2, d0, d1, d2); }

/* ---- one column, quadratic: only the nearest ghost cell (boundary_fv.c:169, :206-209, :238-245) ---- */
__device__ __forceinline__ double bc_v2_value(const double *r, const int m, const int d0, const int d1, const int d2)
{
  if (m == 1) return -2.5 * r[d0] + 0.5 * r[2 * d0];
  if (m == 2) return 6.25 * r[d0 + d1]
                   - 1.25 * r[2 * d0 + d1]
                   - 1.25 * r[d0 + 2 * d1]
                   + 0.25 * r[2 * d0 + 2 * d1];
  return -15.625 * r[d0 + d1 + d2]
        + 3.125 * r[2 * d0 + d1 + d2]
        + 3.125 * r[d0 + 2 * d1 + d2]
        + 3.125 * r[d0 + d1 + 2 * d2]
        - 0.625 * r[2 * d0 + 2 * d1 + d2]
        - 0.625 * r[d0 + 2 * d1 + 2 * d2]
        - 0.625 * r[2 * d0 + d1 + 2 * d2]
        + 0.125 * r[2 * d0 + 2 * d1 + 2 * d2];
}
__device__ __forceinline__ void bc_v2_col(const double *r, double *w, const int m, const int d0, const int d1, const int d2)
{
  w[0] = bc_v2_value(r, m, d0, d1, d2);
}
/* the same, plus the zeroing of the column's deeper ghost cells (boundary_fv.c:139-145 zeroes the whole
 * region first; with 2 ghost layers a region is exactly the union of its columns' 2^m cells) */
__device__ __forceinline__ void bc_v2_col_zero_rest(const double *r, double *w, const int m, const int d0, const int d1, const int d2)
{
  const double v = bc_v2_value(r, m, d0, d1, d2);
  w[-d0] = 0.0;
  if (m >= 2) { w[-d1] = 0.0; w[-d0 - d1] = 0.0; }
  if (m >= 3) { w[-d2] = 0.0; w[-d0 - d2] = 0.0; w[-d1 - d2] = 0.0; w[-d0 - d1 - d2] = 0.0; }
  w[0] = v;
}

/* the v2 column of a ghost fill: fv4 levels have 2 ghost layers and zero the deeper one (above); fv2 levels (-DHPGMG_FV2) have
 * one, and there is nothing deeper to zero */
__device__ __forceinline__ void bc_v2_fill_col(const double *r, double *w, const int m, const int d0, const int d1, const int d2)
{
#ifdef HPGMG_FV2
  bc_v2_col(r, w, m, d0, d1, d2);
#else
  bc_v2_col_zero_rest(r, w, m, d0, d1, d2);
#endif
}

/* the normal axes of a domain normal `subtype` (0..26 = 13+di+3dj+9dk): their count and inward strides */
struct BCNormal {
  int m, d[3];
  int normal[3];
};
__device__ __forceinline__ BCNormal bc_normal(const int subtype, const int jS, const int kS)
{
  BCNormal N;
  N.normal[0] = (subtype % 3) - 1;
  N.normal[1] = ((subtype % 9) / 3) - 1;
  N.normal[2] = (subtype / 9) - 1;
  const int stride[3] = { 1, jS, kS };
  N.m = 0;
  N.d[0] = N.d[1] = N.d[2] = 0;
#pragma unroll
  for (int a = 0; a < 3; a++)
    if (N.normal[a]) N.d[N.m++] = (N.normal[a] < 0) ? stride[a] : -stride[a];
  return N;
}
__device__ __forceinline__ void bc_v4_column(const double *r, double *w, const BCNormal &N)
{
  if (N.m == 1)      bc_v4_col1(r, w, N.d[0]);
  else if (N.m == 2) bc_v4_col2(r, w, N.d[0], N.d[1]);
  else               bc_v4_col3(r, w, N.d[0], N.d[1], N.d[2]);
}

/* ---- one list entry (a block of columns), cooperatively by nthreads threads ---------------------- */
struct BCGeom {
  int normal[3];     /* -1 low side, +1 high side, 0 tangential   (domain normal)       */
  int t[3];          /* coordinate of the nearest ghost cell along a normal axis          */
  int stride[3];
  int lo[3], ext[3]; /* block origin and extent                                           */
};
__device__ __forceinline__ BCGeom bc_geometry(const blockCopy_type &B, const int subtype, const int dim, const int jS, const int kS)
{
  BCGeom G;
  G.normal[0] = (subtype % 3) - 1;
  G.normal[1] = ((subtype % 9) / 3) - 1;
  G.normal[2] = (subtype / 9) - 1;
  G.stride[0] = 1;  G.stride[1] = jS;  G.stride[2] = kS;
  G.lo[0] = B.read.i;  G.lo[1] = B.read.j;  G.lo[2] = B.read.k;
  G.ext[0] = B.dim.i;  G.ext[1] = B.dim.j;  G.ext[2] = B.dim.k;
#pragma unroll
  for (int a = 0; a < 3; a++) G.t[a] = (G.normal[a] < 0) ? -1 : dim;
  return G;
}
/* number of columns of a block and the offset of column c's nearest ghost cell */
__device__ __forceinline__ int bc_num_columns(const BCGeom &G)
{
  return (G.normal[0] ? 1 : G.ext[0]) * (G.normal[1] ? 1 : G.ext[1]) * (G.normal[2] ? 1 : G.ext[2]);
}
__device__ __forceinline__ int bc_column_offset(const BCGeom &G, const int c)
{
  const int e0 = G.normal[0] ? 1 : G.ext[0], e1 = G.normal[1] ? 1 : G.ext[1];
  const int p0 = c % e0, p1 = (c / e0) % e1, p2 = c / (e0 * e1);
  return (G.normal[0] ? G.t[0] : p0 + G.lo[0]) * G.stride[0]
       + (G.normal[1] ? G.t[1] : p1 + G.lo[1]) * G.stride[1]
       + (G.normal[2] ? G.t[2] : p2 + G.lo[2]) * G.stride[2];
}
__device__ __forceinline__ void bc_zero_block(double *x, const BCGeom &G, const int tid, const int nthreads)
{
  const int cells = G.ext[0] * G.ext[1] * G.ext[2];
  for (int c = tid; c < cells; c += nthreads) {
    const int i = c % G.ext[0], j = (c / G.ext[0]) % G.ext[1], k = c / (G.ext[0] * G.ext[1]);
    x[(i + G.lo[0]) * G.stride[0] + (j + G.lo[1]) * G.stride[1] + (k + G.lo[2]) * G.stride[2]] = 0.0;
  }
}

__device__ __forceinline__ void bc_v4_block(const DLevel &L, const int id, const blockCopy_type &B, const int tid, const int nthreads)
{
  const BCGeom G = bc_geometry(B, B.subtype, L.dim, L.jStride, L.kStride);
  const BCNormal N = bc_normal(B.subtype, L.jStride, L.kStride);
  double *x = L.vec(B.read.box, id);
  if (L.ghosts > 2) {                                    /* boundary_fv.c:299-306 */
    bc_zero_block(x, G, tid, nthreads);
    __syncthreads();
  }
  const int cols = bc_num_columns(G);
  for (int c = tid; c < cols; c += nthreads) { double *w = x + bc_column_offset(G, c); bc_v4_column(w, w, N); }
}

/* quadratic: deeper ghost layers are zeroed first (boundary_fv.c:139-145) */
__device__ __forceinline__ void bc_v2_block(const DLevel &L, const int id, const blockCopy_type &B, const int tid, const int nthreads)
{
  const BCGeom G = bc_geometry(B, B.subtype, L.dim, L.jStride, L.kStride);
  const BCNormal N = bc_normal(B.subtype, L.jStride, L.kStride);
  double *x = L.vec(B.read.box, id);
  if (L.ghosts > 1) {
    bc_zero_block(x, G, tid, nthreads);
    __syncthreads();
  }
  const int cols = bc_num_columns(G);
  for (int c = tid; c < cols; c += nthreads) { double *w = x + bc_column_offset(G, c); bc_v2_col(w, w, N.m, N.d[0], N.d[1], N.d[2]); }
}

#endif
