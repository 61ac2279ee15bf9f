/*
 * stencil_box.cuh -- the operator kernels for boxes of 4^3 .. 32^3 cells whose neighbours all live on this GPU:
 * ghost fill and operator FUSED into one launch.
 *
 * On these levels every kernel is a few microseconds of latency, and a sweep used to be two of them: the fused ghost
 * fill (exchange_boundary + apply_BCs, ghost.cu) and the sweep itself.  Here a thread block owns a TI x TJ x TK tile
 * of one box and stages x on the tile plus its 2-cell halo in shared memory ITSELF:
 *   - halo cells inside the box are plain loads;
 *   - halo cells in the box's ghost zone come from the per-tile records of the level's NO_CORNERS fill
 *     (TileTable, built in device_level.cu from the reference-identical exchange and BC lists): a cell of the
 *     neighbouring box is read from that box's interior, a boundary-condition column is extrapolated from the
 *     interior values it depends on (bc.cuh) -- straight into the staged tile.
 * The values are those the separate fill would have left in the ghost cells (same expressions, same operands), so
 * the result is bit-identical; the ghost cells in HBM are simply not needed any more (residual / apply_op still
 * write them, because callers of the reference API may look at them: residual.c:15-16 fills x in place).
 * gsrb.c:41-129, chebyshev.c:51-97, jacobi.c, residual.c:18-49, apply_op.c:18-47; arithmetic = fv4_apply_op_at and the
 * smoothers' cell updates (stencil.cuh).
 *
 * Face coefficients, rhs and Dinv are read straight from global memory at compile-time strides (the box size is a
 * template parameter), i.e. as loads at immediate offsets through L1.  Rows of the staged tile are stored as they are
 * in memory with an even pitch, so the two rows a half-warp works on -- whose active cells have opposite i-parity on a
 * red-black sweep -- fall into disjoint shared-memory banks.
 */
#ifndef HPGMG_B200_STENCIL_BOX_CUH
#define HPGMG_B200_STENCIL_BOX_CUH

#include "stencil.cuh"
#include "bc.cuh"

template <int N, int TI, int TJ, int TK>
struct BoxCfg {
  static constexpr int P = N + 4;                                  /* padded box extent (ghosts = 2), level.c:935-938 */
  static constexpr int jS = (P + 3) / 4 * 4, kS = jS * P;
  static constexpr int SW = TI + 4, SH = TJ + 4, SD = TK + 4;      /* staged tile */
  static constexpr int SCELLS = SW * SH * SD;
  static constexpr int NT = (TI / 2) * TJ * TK;                    /* one thread per i-pair */
  static constexpr int NI = N / TI, NJ = N / TJ, NK = N / TK, TILES = NI * NJ * NK;
};

template <int SW, int SH>
struct TileLoader {                                                /* p points at the cell in the staged tile */
  const double *p;
  __device__ __forceinline__ double operator()(const int di, const int dj, const int dk) const { return p[di + dj * SW + dk * SW * SH]; }
};
template <int JS, int KS>
struct BoxLoader {                                                 /* p points at the cell in a box array with compile-time strides */
  const double *p;
  __device__ __forceinline__ double operator()(const int di, const int dj, const int dk) const { return p[di + dj * JS + dk * KS]; }
};

struct BoxArgs {
  DLevel L;
  const int *low;
  const TileRange *ranges;
  const TileCopy *copies;
  const TileBC *bc;
  int x_id, rhs_id, out_id;
  int sweep;                                                       /* GSRB colour */
  int write_ghosts;                                                /* also leave the ghost values in HBM (residual, apply_op) */
  double b, h2inv, c1, c2;
  double weight;                                                   /* Jacobi: lambda of box b at lam + b * lam_bstride (cell 0,0,0) */
  const double *lam;
  size_t lam_bstride;
};

template <int OP, int N, int TI, int TJ, int TK>
__global__ void __launch_bounds__((TI / 2) * TJ * TK) stencil_box_kernel(const BoxArgs A)
{
  typedef BoxCfg<N, TI, TJ, TK> C;
  __shared__ __align__(16) double tile[C::SCELLS];
  const int tid = threadIdx.x;
  const int box = blockIdx.x / C::TILES, t = blockIdx.x - box * C::TILES;
  const int i0 = (t % C::NI) * TI, j0 = ((t / C::NI) % C::NJ) * TJ, k0 = (t / (C::NI * C::NJ)) * TK;
  const DLevel &L = A.L;
  const TileRange R = A.ranges[blockIdx.x];                        /* written at setup, not by the previous kernel: may precede the wait */
  PDL_WAIT();
  double *v = L.base + (size_t)A.x_id * (size_t)L.volume;          /* fill records are relative to the vector's start (all boxes) */
  const double *xb = L.vec(box, A.x_id);                           /* cell (0,0,0) of this box */

  /* ---- stage x: cells of the box ... */
  constexpr int ROUNDS = (C::SCELLS + C::NT - 1) / C::NT;
#pragma unroll
  for (int r = 0; r < ROUNDS; r++) {
    const int c = tid + r * C::NT;
    const int si = c % C::SW, sj = (c / C::SW) % C::SH, sk = c / (C::SW * C::SH);
    const int i = i0 + si - 2, j = j0 + sj - 2, k = k0 + sk - 2;
    if (c < C::SCELLS && (unsigned)i < (unsigned)N && (unsigned)j < (unsigned)N && (unsigned)k < (unsigned)N) tile[c] = xb[i + j * C::jS + k * C::kS];
  }
  /* ... cells of the neighbouring boxes ... */
  for (int e = tid; e < R.ncopy; e += C::NT) {
    const TileCopy c = A.copies[R.copy0 + e];
    const double val = v[c.src];
    tile[c.sidx] = val;
    if (A.write_ghosts) v[c.dst] = val;
  }
  /* ... and boundary-condition columns (apply_BCs_v4, boundary_fv.c:262-569) */
  for (int e = tid; e < R.nbc; e += C::NT) {
    const TileBC it = A.bc[R.bc0 + e];
    const BCNormal Nn = bc_normal(it.subtype, C::jS, C::kS);
    const BCNormal Ns = bc_normal(it.subtype, C::SW, C::SW * C::SH);
    const double *r = v + it.src;
    double *w = tile + it.sidx;
    if (Nn.m == 1)      bc_v4_col1(r, w, Nn.d[0], Ns.d[0]);
    else if (Nn.m == 2) bc_v4_col2(r, w, Nn.d[0], Nn.d[1], Ns.d[0], Ns.d[1]);
    else                bc_v4_col3(r, w, Nn.d[0], Nn.d[1], Nn.d[2], Ns.d[0], Ns.d[1], Ns.d[2]);
    if (A.write_ghosts) {                                           /* the same values into the box's ghost cells */
      double *g = v + it.dst;
      g[0] = w[0];
      g[-Nn.d[0]] = w[-Ns.d[0]];
      if (Nn.m >= 2) { g[-Nn.d[1]] = w[-Ns.d[1]]; g[-Nn.d[0] - Nn.d[1]] = w[-Ns.d[0] - Ns.d[1]]; }
      if (Nn.m >= 3) {
        g[-Nn.d[2]] = w[-Ns.d[2]];  g[-Nn.d[0] - Nn.d[2]] = w[-Ns.d[0] - Ns.d[2]];
        g[-Nn.d[1] - Nn.d[2]] = w[-Ns.d[1] - Ns.d[2]];  g[-Nn.d[0] - Nn.d[1] - Nn.d[2]] = w[-Ns.d[0] - Ns.d[1] - Ns.d[2]];
      }
    }
  }
  __syncthreads();

  /* ---- the operator on my i-pair ---- */
  const int p = tid % (TI / 2), jj = (tid / (TI / 2)) % TJ, kk = tid / ((TI / 2) * TJ);
  const int i = i0 + 2 * p, j = j0 + jj, k = k0 + kk;
  const int cell = i + j * C::jS + k * C::kS;
  const double *ts = tile + (2 * p + 2) + (jj + 2) * C::SW + (kk + 2) * C::SW * C::SH;
  const double *bi = L.vec(box, VECTOR_BETA_I) + cell, *bj = L.vec(box, VECTOR_BETA_J) + cell, *bk = L.vec(box, VECTOR_BETA_K) + cell;
  double2 *out = reinterpret_cast<double2 *>(L.vec(box, A.out_id) + cell);
  if constexpr (OP == OP_GSRB) {
    const int a = (j ^ k ^ gsrb_box_parity(A.low, box, A.sweep)) & 1;     /* the pair's active cell */
    const double2 rhs2 = *reinterpret_cast<const double2 *>(L.vec(box, A.rhs_id) + cell);
    const double2 dinv2 = *reinterpret_cast<const double2 *>(L.vec(box, VECTOR_DINV) + cell);
    const TileLoader<C::SW, C::SH> X = { ts + a };
    const BoxLoader<C::jS, C::kS> BI = { bi + a }, BJ = { bj + a }, BK = { bk + a };
    const double Ax = fv4_apply_op_at(X, BI, BJ, BK, A.b, A.h2inv);
    const double xnew = gsrb_update(ts[a], a ? dinv2.y : dinv2.x, a ? rhs2.y : rhs2.x, Ax);
    const double xo = ts[1 - a];                                   /* the other cell is copied (gsrb.c:65-71) */
    *out = a ? make_double2(xo, xnew) : make_double2(xnew, xo);
  } else {
    double Ax[2];
#pragma unroll
    for (int q = 0; q < 2; q++) {
      const TileLoader<C::SW, C::SH> X = { ts + q };
      const BoxLoader<C::jS, C::kS> BI = { bi + q }, BJ = { bj + q }, BK = { bk + q };
      Ax[q] = fv4_apply_op_at(X, BI, BJ, BK, A.b, A.h2inv);
    }
    if constexpr (OP == OP_APPLY) {
      *out = make_double2(Ax[0], Ax[1]);
    } else {
      const double2 rhs2 = *reinterpret_cast<const double2 *>(L.vec(box, A.rhs_id) + cell);
      if constexpr (OP == OP_RESIDUAL) {
        *out = make_double2(rhs2.x - Ax[0], rhs2.y - Ax[1]);
      } else if constexpr (OP == OP_JACOBI) {
        const double2 lam2 = *reinterpret_cast<const double2 *>(A.lam + (size_t)box * A.lam_bstride + cell);
        *out = make_double2(jacobi_update(ts[0], A.weight, lam2.x, rhs2.x, Ax[0]), jacobi_update(ts[1], A.weight, lam2.y, rhs2.y, Ax[1]));
      } else {                                                       /* OP_CHEBY */
        const double2 dinv2 = *reinterpret_cast<const double2 *>(L.vec(box, VECTOR_DINV) + cell);
        const double2 xm = *out;                                     /* x_{n-1} aliases x_{n+1} (chebyshev.c:75-80) */
        *out = make_double2(chebyshev_update(ts[0], xm.x, A.c1, A.c2, dinv2.x, rhs2.x, Ax[0]),
                            chebyshev_update(ts[1], xm.y, A.c1, A.c2, dinv2.y, rhs2.y, Ax[1]));
      }
    }
  }
}

#endif
