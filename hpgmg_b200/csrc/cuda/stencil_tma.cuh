/*
 * stencil_tma.cuh -- the operator kernels for boxes >= 32^3, Blackwell version: 2.5-D blocking with the halo
 * tiles staged in shared memory by the TMA engine.
 *
 * GSRB / Chebyshev / Jacobi / residual / apply_op on a TI x TJ column of cells marching along k (gsrb.c:41-129,
 * chebyshev.c:51-97, jacobi.c, residual.c:18-49, apply_op.c:18-47 with the macro of operators.fv4.c:87-114); the
 * arithmetic is fv4_apply_op_at, shared with every other kernel, hence the same bits.  Around the arithmetic:
 *
 *  - staging: one elected thread issues cp.async.bulk.tensor (TMA) copies of whole (TI+4) x rows tiles
 *    of x, beta_i, beta_j, beta_k PF steps ahead into ring buffers; completion is counted by mbarriers
 *    (complete_tx::bytes).  No LDGSTS / address arithmetic in the compute warps (the cp.async version
 *    spent 16 LDGSTS = 128 LSU cycles per warp and plane on it).
 *  - layout: rows are stored as they are in memory (TMA cannot split parities).  GSRB: bank conflicts of the stride-2
 *    red-black accesses are avoided by the lane mapping: a thread owns an i-pair (one active cell per sweep), even lanes work
 *    on row r, odd lanes on row r+1 of a row pair; the active cells of the two rows have opposite i-parity, so the 16 lanes of
 *    a half-warp touch 16 distinct 8-byte banks.  Residual / Chebyshev / Jacobi / apply_op: a thread owns the j-pair (i,j), (i,j+1);
 *    lanes are consecutive cells of a row (conflict-free), and the two stencils share their common operands (pure loads
 *    merged by the compiler: 85 LDS per cell pair instead of 110).
 *  - addressing: a lane keeps ONE 32-bit shared address per ring slot; every stencil operand is a load at a compile-time
 *    offset from it (LDS [R+imm]).
 *  - scheduling: block b owns the planes [P*b/G, P*(b+1)/G) of the linearised (box, tile, k) space and
 *    walks them as segments of one column each.  The launcher (smooth.cu: launch_tma) picks G = columns x
 *    equal k-chunks, so that every block is exactly one chunk and all blocks march k in step; any other G
 *    (HPGMG_B200_TMA_BLOCKS) gives an even split with partial columns -- correct, but 24 % slower on `7 8`
 *    because neighbouring tiles then fetch their common halo rows at different times.
 *  - GSRB only: Dinv = 1/Aii is formed from the face coefficients in registers away from the domain boundary
 *    (stencil.cuh) instead of being read; alternate sweeps march k downwards (REV).
 *  - residual only: the kernel also leaves max |res| in a scalar slot when the caller wants the norm next.
 */
#ifndef HPGMG_B200_STENCIL_TMA_CUH
#define HPGMG_B200_STENCIL_TMA_CUH

#include <cuda.h>
#include "stencil.cuh"

template <int TI, int TJ, int PF>
struct TmaCfg {
  static constexpr int W = TI + 4;                 /* cells i0-2 .. i0+TI+1 of a row                      */
  static constexpr int XR = TJ + 4;                /* x rows    j0-2 .. j0+TJ+1                           */
  static constexpr int BR = TJ + 2;                /* beta rows j0-1 .. j0+TJ                             */
  static constexpr int XP = 5 + PF, BP = 3 + PF, KP = 2 + PF;   /* ring depths: planes in use + PF planes in flight */
  static constexpr int NB = PF + 1;                /* mbarriers: one per step in flight + the one being waited on */
  static constexpr int NT = (TI / 2) * TJ;         /* threads: one per i-pair of cells                    */
  static constexpr int XBYTES = XR * W * 8, BBYTES = BR * W * 8;          /* bytes one TMA copy delivers  */
  static constexpr int XPB = (XBYTES + 127) / 128 * 128;                  /* slot pitch (TMA wants 128-B aligned destinations) */
  static constexpr int BPB = (BBYTES + 127) / 128 * 128;
  static constexpr int OFF_BI = XP * XPB, OFF_BJ = OFF_BI + BP * BPB, OFF_BK = OFF_BJ + BP * BPB, OFF_BAR = OFF_BK + KP * BPB;
  static constexpr size_t SMEM = (size_t)OFF_BAR + 8 * NB + 128;         /* + mbarriers + alignment slack */
};

/* ---- PTX wrappers ---------------------------------------------------------------------------------- */
__device__ __forceinline__ double lds_f64(const unsigned a)
{
  double v;
  asm volatile("ld.shared.f64 %0, [%1];" : "=d"(v) : "r"(a));
  return v;
}
__device__ __forceinline__ void mbar_init(const unsigned bar, const unsigned count)
{
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(const unsigned bar, const unsigned bytes)
{
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(const unsigned bar, const unsigned parity)
{
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "MBAR_WAIT:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra MBAR_DONE;\n"
      "bra MBAR_WAIT;\n"
      "MBAR_DONE:\n"
      "}\n" ::"r"(bar), "r"(parity) : "memory");
}
/* one (W x rows x 1 x 1) tile of the level slab viewed as [box*vector][k][j][i] */
__device__ __forceinline__ void tma_load_4d(const unsigned dst, const CUtensorMap *map, const int c0, const int c1, const int c2, const int c3, const unsigned bar)
{
  asm volatile("cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4, %5}], [%6];"
               ::"r"(dst), "l"(map), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(bar) : "memory");
}

/* shared-memory loader: a[d] is the byte address of the lane's active cell in the ring slot that holds
 * plane k + DK0 + d; an operand at (di,dj,dk) is a load at a compile-time offset from it. */
template <int W, int DK0, int NPLANES>
struct SlotLoader {
  unsigned a[NPLANES];
  __device__ __forceinline__ double operator()(const int di, const int dj, const int dk) const
  {
    return lds_f64(a[dk - DK0] + (unsigned)((dj * W + di) * 8));
  }
};

/* The same load as a PURE function of (address, token): not volatile, so the two stencil evaluations of a thread that owns
 * two cells share the operands they have in common (the compiler merges loads with identical operands: 85 instead of 110
 * per cell pair).  The token is made by a volatile asm at the top of a march step, after the step's planes have landed, so
 * a load can neither move above that point nor be merged with a load of another step. */
__device__ __forceinline__ double lds_f64_pure(const unsigned a, const unsigned tok)
{
  double v;
  asm("ld.shared.f64 %0, [%1]; // step %2" : "=d"(v) : "r"(a), "r"(tok));
  return v;
}
template <int W, int DK0, int NPLANES>
struct PureSlotLoader {
  unsigned a[NPLANES];
  unsigned tok;
  __device__ __forceinline__ double operator()(const int di, const int dj, const int dk) const
  {
    return lds_f64_pure(a[dk - DK0] + (unsigned)((dj * W + di) * 8), tok);
  }
};

/* PF: how many steps ahead the planes are requested.  MINB: resident blocks per SM the register budget is
 * sized for.  REV: march k downwards -- alternating the direction from sweep to sweep lets a sweep start
 * on the planes the previous sweep touched last, which are still in the 126 MB L2. */
template <int OP, int TI, int TJ, int PF, int MINB, bool REV>
__global__ void __launch_bounds__((TI / 2) * TJ, MINB)
stencil_tma_kernel(const StencilArgs A, const __grid_constant__ CUtensorMap map_x, const __grid_constant__ CUtensorMap map_b, const long long total_planes)
{
  typedef TmaCfg<TI, TJ, PF> C;
  extern __shared__ unsigned char smem_raw[];
  const unsigned s0 = ((unsigned)__cvta_generic_to_shared(smem_raw) + 127u) & ~127u;
  const unsigned xs = s0, bis = s0 + C::OFF_BI, bjs = s0 + C::OFF_BJ, bks = s0 + C::OFF_BK, bar0 = s0 + C::OFF_BAR;

  const int tid = threadIdx.x;
  if (tid == 0) {
#pragma unroll
    for (int q = 0; q < C::NB; q++) mbar_init(bar0 + 8 * q, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  PDL_WAIT();

  const DLevel &L = A.L;
  const int n = L.dim, jS = L.jStride, kS = L.kStride;
  const int tiles_i = n / TI, tiles = tiles_i * (n / TJ);

  /* GSRB: lane -> (row, i-pair): even lanes row 2rp, odd lanes row 2rp+1; 16 consecutive pairs per warp.
   * The uncoloured operators (JP): a thread owns the J-pair (i, j), (i, j+1) -- lanes are consecutive cells of a row, so every
   * 64-bit shared load of a warp is two conflict-free wavefronts, and the two cells share 25 of their 110 operands. */
  constexpr bool JP = (OP != OP_GSRB);
  static_assert(!JP || TI == 32, "the j-pair mapping puts one row of a tile on the lanes of a warp");
  constexpr int WPR = (TI / 2) / 16;                                /* warps per row pair */
  const int warp = tid >> 5, lane = tid & 31;
  const int r = JP ? 2 * warp : 2 * (warp / WPR) + (lane & 1);
  const int p = 16 * (warp % WPR) + (lane >> 1);
  const int ci_lane = JP ? lane : 2 * p;                            /* first (only) cell of the thread within the tile row */
  const unsigned lane_x = (unsigned)(((r + 2) * C::W + 2 + ci_lane) * 8);   /* the thread's first cell, x tile  */
  const unsigned lane_b = (unsigned)(((r + 1) * C::W + 2 + ci_lane) * 8);   /* the same in the beta tiles       */

  /* my share of the linearised (box, tile, k) space */
  const long long lo = total_planes * (long long)blockIdx.x / (long long)gridDim.x;
  const long long hi = total_planes * (long long)(blockIdx.x + 1) / (long long)gridDim.x;
  unsigned phasebits = 0;                                           /* bit q: parity of the next wait on mbarrier q */
  double vmax = 0.0;                                                /* OP_RESIDUAL: max |res| over this thread's cells */

  for (long long pos = lo; pos < hi;) {
    const int col = (int)(pos / n);
    const int k0 = (int)(pos - (long long)col * n);
    const int k1 = (int)min((long long)n, (long long)k0 + (hi - pos));
    pos += k1 - k0;
    const int box = col / tiles, tile = col - box * tiles;
    const int i0 = (tile % tiles_i) * TI, j0 = (tile / tiles_i) * TJ;
    const int g = L.ghosts;                                          /* tensor coordinates count from the padded origin */
    const int cx = box * L.nvec + A.x_id, cbi = box * L.nvec + VECTOR_BETA_I, cbj = box * L.nvec + VECTOR_BETA_J, cbk = box * L.nvec + VECTOR_BETA_K;
    const int ci = i0 - 2 + g, cjx = j0 - 2 + g, cjb = j0 - 1 + g;

    /* Step q (plane kf + q dir) reads x planes q..q+4, beta_i/j planes q..q+2 and beta_k planes q, q+1, counted
     * in marching order from the first plane each array needs; plane m of an array lives in ring slot m mod depth.
     * Prologue: everything step 0 needs on mbarrier 0, then what steps 1..PF-1 need in addition, one mbarrier each. */
    constexpr int dir = REV ? -1 : 1;
    const int kf = REV ? k1 - 1 : k0, len = k1 - k0;
    if (tid == 0) {
      mbar_expect_tx(bar0, 5 * C::XBYTES + 8 * C::BBYTES);
#pragma unroll
      for (int d = 0; d < 5; d++) tma_load_4d(xs + d * C::XPB, &map_x, ci, cjx, kf + (d - 2) * dir + g, cx, bar0);
#pragma unroll
      for (int d = 0; d < 3; d++) {
        tma_load_4d(bis + d * C::BPB, &map_b, ci, cjb, kf + (d - 1) * dir + g, cbi, bar0);
        tma_load_4d(bjs + d * C::BPB, &map_b, ci, cjb, kf + (d - 1) * dir + g, cbj, bar0);
      }
#pragma unroll
      for (int d = 0; d < 2; d++) tma_load_4d(bks + d * C::BPB, &map_b, ci, cjb, kf + (REV ? 1 - d : d) + g, cbk, bar0);
#pragma unroll
      for (int q = 1; q < PF; q++)
        if (q < len) {
          const unsigned bq = bar0 + 8 * (q % C::NB);
          mbar_expect_tx(bq, C::XBYTES + 3 * C::BBYTES);
          tma_load_4d(xs + ((q + 4) % C::XP) * C::XPB, &map_x, ci, cjx, kf + (q + 2) * dir + g, cx, bq);
          tma_load_4d(bis + ((q + 2) % C::BP) * C::BPB, &map_b, ci, cjb, kf + (q + 1) * dir + g, cbi, bq);
          tma_load_4d(bjs + ((q + 2) % C::BP) * C::BPB, &map_b, ci, cjb, kf + (q + 1) * dir + g, cbj, bq);
          tma_load_4d(bks + ((q + 1) % C::KP) * C::BPB, &map_b, ci, cjb, kf + (REV ? -q : q + 1) + g, cbk, bq);
        }
    }

    const int j = j0 + r;
    const int cell = (i0 + ci_lane) + j * jS;                      /* GSRB: pair (2p, 2p+1) of row j; JP: cells (lane, j), (lane, j+1); plane 0 */
    const double *g_rhs = (OP == OP_APPLY) ? nullptr : L.vec(box, A.rhs_id) + cell;
    /* the point-wise inverse: Dinv, or lambda of a Jacobi sweep (Dinv or the L1 row inverse, which need not be in the slab) */
    const double *g_dinv = (OP == OP_GSRB || OP == OP_CHEBY) ? L.vec(box, VECTOR_DINV) + cell
                         : (OP == OP_JACOBI) ? A.lam + (size_t)box * A.lam_bstride + cell : nullptr;
    const double *g_xm1 = (OP == OP_CHEBY) ? L.vec(box, A.xm1_id) + cell : nullptr;
    double *g_out = L.vec(box, A.out_id) + cell;
    double *c_out = nullptr;                                         /* OP_RESRES: the coarse cell under (lane, j), plane 0 of the coarse box */
    double racc = 0.0;
    if (OP == OP_RESRES) {
      const int *M = A.rmap + 4 * box;
      c_out = A.Lc.vec(M[0], A.rc_id) + (M[1] + ((i0 + ci_lane) >> 1)) + (M[2] + (j >> 1)) * A.Lc.jStride + M[3] * A.Lc.kStride;
    }
    /* which cell of the pair is updated on plane k0 of this sweep (gsrb.c:55,100); flips every plane.
     * For the uncoloured operators it only fixes the ORDER in which the lane evaluates its two cells
     * (odd lanes start with the odd cell, so that a half-warp still covers all banks). */
    int s = (OP == OP_GSRB) ? ((j ^ kf ^ A.low[3 * box] ^ A.low[3 * box + 1] ^ A.low[3 * box + 2] ^ A.sweep) & 1) : (lane & 1);

    /* Dinv from memory only where a cell of the tile is within 2 cells of the domain boundary (its stencil then
     * reaches boundary-condition ghost cells and the stored diagonal carries their contribution); elsewhere it is
     * 1/Aii of the face coefficients the stencil loads anyway (stencil.cuh) -- 8 of the sweep's 56 B/cell less */
    bool tile_inner = false;
    int gk0 = 0;
    if (OP == OP_GSRB && A.diag) {
      const int gi = A.low[3 * box] + i0, gj = A.low[3 * box + 1] + j0;
      tile_inner = gi >= 2 && gi + TI <= A.dom[0] - 2 && gj >= 2 && gj + TJ <= A.dom[1] - 2;
      gk0 = A.low[3 * box + 2];
    }
    const int gk_hi = A.dom[2] - 3;
#define PLANE_NEEDS_DINV(kk) (!(OP == OP_GSRB) || !tile_inner || gk0 + (kk) < 2 || gk0 + (kk) > gk_hi)

    /* point-wise operands (rhs, Dinv or lambda, x_{n-1}) are read one plane ahead into registers */
    double2 rhs_n = make_double2(0.0, 0.0), dinv_n = make_double2(0.0, 0.0), xm_n = make_double2(0.0, 0.0);
#define LOAD_PAIR(ptr, kk) (JP ? make_double2((ptr)[(kk) * kS], (ptr)[(kk) * kS + jS]) : *reinterpret_cast<const double2 *>((ptr) + (kk) * kS))
    if (OP != OP_APPLY) rhs_n = LOAD_PAIR(g_rhs, kf);
    if ((OP == OP_GSRB || OP == OP_CHEBY || OP == OP_JACOBI) && PLANE_NEEDS_DINV(kf)) dinv_n = LOAD_PAIR(g_dinv, kf);
    if (OP == OP_CHEBY) xm_n = LOAD_PAIR(g_xm1, kf);

    mbar_wait(bar0, phasebits & 1u);                               /* step 0's planes */
    phasebits ^= 1u;

    int sx = 0, sb = 0, sk = 0, bq = 0;                            /* ring slots of the step's first planes; the step's mbarrier */
    for (int t = 0; t < len; t++) {
      const int k = kf + t * dir;
      const bool more = (t + 1 < len);
      /* ---- request what step t+PF needs in addition: the slots right behind the step's first planes were last
       *      read in step t-1 (barrier at its end), and mbarrier (t+PF) mod NB was last waited on at the end of step t-2 ---- */
      if (tid == 0 && t + PF < len) {
        const int nx = sx == 0 ? C::XP - 1 : sx - 1;
        const int nb = sb == 0 ? C::BP - 1 : sb - 1;
        const int nk = sk == 0 ? C::KP - 1 : sk - 1;
        const int qn = bq == 0 ? C::NB - 1 : bq - 1;                 /* (t + PF) mod NB == (t - 1) mod NB */
        const unsigned bn = bar0 + 8 * qn;
        mbar_expect_tx(bn, C::XBYTES + 3 * C::BBYTES);
        tma_load_4d(xs + nx * C::XPB, &map_x, ci, cjx, k + (PF + 2) * dir + g, cx, bn);
        tma_load_4d(bis + nb * C::BPB, &map_b, ci, cjb, k + (PF + 1) * dir + g, cbi, bn);
        tma_load_4d(bjs + nb * C::BPB, &map_b, ci, cjb, k + (PF + 1) * dir + g, cbj, bn);
        tma_load_4d(bks + nk * C::BPB, &map_b, ci, cjb, k + (REV ? -PF : PF + 1) + g, cbk, bn);
      }
      const double2 rhs2 = rhs_n, dinv2 = dinv_n, xm2 = xm_n;
      if (more) {
        if (OP != OP_APPLY) rhs_n = LOAD_PAIR(g_rhs, k + dir);
        if ((OP == OP_GSRB || OP == OP_CHEBY || OP == OP_JACOBI) && PLANE_NEEDS_DINV(k + dir)) dinv_n = LOAD_PAIR(g_dinv, k + dir);
        if (OP == OP_CHEBY) xm_n = LOAD_PAIR(g_xm1, k + dir);
      }

      /* ---- slot addresses of this step's planes, indexed by plane offset (ring position r holds plane
       *      k + (r - 2) dir for x, k + (r - 1) dir for beta_i/j, and the step's two beta_k planes in marching order) ---- */
      unsigned ax[5], abi[3], abj[3], abk[2];
#pragma unroll
      for (int d = 0; d < 5; d++) { const int q = sx + d; ax[REV ? 4 - d : d] = xs + (unsigned)((q >= C::XP ? q - C::XP : q) * C::XPB) + lane_x; }
#pragma unroll
      for (int d = 0; d < 3; d++) { const int q = sb + d; const unsigned o = (unsigned)((q >= C::BP ? q - C::BP : q) * C::BPB) + lane_b; abi[REV ? 2 - d : d] = bis + o; abj[REV ? 2 - d : d] = bjs + o; }
#pragma unroll
      for (int d = 0; d < 2; d++) { const int q = sk + d; abk[REV ? 1 - d : d] = bks + (unsigned)((q >= C::KP ? q - C::KP : q) * C::BPB) + lane_b; }

      SlotLoader<C::W, -2, 5> X;
      SlotLoader<C::W, -1, 3> BI, BJ;
      SlotLoader<C::W, 0, 2> BK;
      double2 out2;
      if (OP == OP_GSRB) {
        const unsigned so = (unsigned)(8 * s);
#pragma unroll
        for (int d = 0; d < 5; d++) X.a[d] = ax[d] + so;
#pragma unroll
        for (int d = 0; d < 3; d++) { BI.a[d] = abi[d] + so; BJ.a[d] = abj[d] + so; }
#pragma unroll
        for (int d = 0; d < 2; d++) BK.a[d] = abk[d] + so;
        double aii;
        const double Ax = fv4_apply_op_at(X, BI, BJ, BK, A.b, A.h2inv, &aii);
        const double xc = X(0, 0, 0);
        const double xo = lds_f64(ax[2] + (unsigned)(8 * (1 - s)));    /* the pair's other cell: copied (gsrb.c:65-71) */
        const double dinv = PLANE_NEEDS_DINV(k) ? (s ? dinv2.y : dinv2.x) : 1.0 / aii;
        const double xnew = xc + dinv * ((s ? rhs2.y : rhs2.x) - Ax);
        out2 = s ? make_double2(xo, xnew) : make_double2(xnew, xo);
        s ^= 1;
      } else {
        unsigned tok;
        asm volatile("mov.u32 %0, %1;" : "=r"(tok) : "r"(t) : "memory");     /* this step's planes are in place from here on */
        double res[2];
#pragma unroll
        for (int c = 0; c < 2; c++) {                                  /* cell (lane, j + c) */
          const unsigned so = (unsigned)(c * C::W * 8);
          PureSlotLoader<C::W, -2, 5> PX;
          PureSlotLoader<C::W, -1, 3> PBI, PBJ;
          PureSlotLoader<C::W, 0, 2> PBK;
          PX.tok = PBI.tok = PBJ.tok = PBK.tok = tok;
#pragma unroll
          for (int d = 0; d < 5; d++) PX.a[d] = ax[d] + so;
#pragma unroll
          for (int d = 0; d < 3; d++) { PBI.a[d] = abi[d] + so; PBJ.a[d] = abj[d] + so; }
#pragma unroll
          for (int d = 0; d < 2; d++) PBK.a[d] = abk[d] + so;
          const double Ax = fv4_apply_op_at(PX, PBI, PBJ, PBK, A.b, A.h2inv);
          double v;
          if (OP == OP_APPLY) v = Ax;
          else if (OP == OP_RESIDUAL) { v = (c ? rhs2.y : rhs2.x) - Ax; const double f = fabs(v); if (f > vmax) vmax = f; }
          else if (OP == OP_RESRES) v = (c ? rhs2.y : rhs2.x) - Ax;
          else if (OP == OP_JACOBI) {                                /* jacobi.c: x_n + weight*lambda*(rhs - Ax_n), left to right */
            const double xn = PX(0, 0, 0);
            v = xn + (A.weight * (c ? dinv2.y : dinv2.x)) * ((c ? rhs2.y : rhs2.x) - Ax);
          }
          else {                                                     /* OP_CHEBY, chebyshev.c:90 */
            const double xn = PX(0, 0, 0);
            v = xn + A.c1 * (xn - (c ? xm2.y : xm2.x)) + A.c2 * (c ? dinv2.y : dinv2.x) * ((c ? rhs2.y : rhs2.x) - Ax);
          }
          res[c] = v;
        }
        out2 = make_double2(res[0], res[1]);
      }
      if (OP == OP_RESRES) {
        /* restriction.c:54-57: (f000 + f100 + f010 + f110 + f001 + f101 + f011 + f111) * 0.125, summed left to right.  This
         * lane holds (i, j) and (i, j+1) of plane k, lane+1 the cells i+1; k-chunks start on even planes and j is even. */
        const double o0 = __shfl_down_sync(0xffffffffu, out2.x, 1), o1 = __shfl_down_sync(0xffffffffu, out2.y, 1);
        if ((k & 1) == 0) racc = ((out2.x + o0) + out2.y) + o1;
        else {
          racc = (((racc + out2.x) + o0) + out2.y) + o1;
          if ((lane & 1) == 0) c_out[(k >> 1) * A.Lc.kStride] = racc * 0.125;
        }
      }
      else if (JP) { g_out[k * kS] = out2.x; g_out[k * kS + jS] = out2.y; }
      else *reinterpret_cast<double2 *>(g_out + k * kS) = out2;

      sx = sx + 1 == C::XP ? 0 : sx + 1;
      sb = sb + 1 == C::BP ? 0 : sb + 1;
      sk = sk + 1 == C::KP ? 0 : sk + 1;
      bq = bq + 1 == C::NB ? 0 : bq + 1;
      if (more) {                                                    /* the next step's planes have landed */
        mbar_wait(bar0 + 8 * bq, (phasebits >> bq) & 1u);
        phasebits ^= 1u << bq;
      }
      __syncthreads();                                               /* everyone is done with the oldest slots */
    }
#undef PLANE_NEEDS_DINV
#undef LOAD_PAIR
  }
  if (OP == OP_RESIDUAL && A.norm_slot != nullptr) {                /* norm(): misc.c:287-329, max of |res| */
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const double other = __shfl_down_sync(0xffffffffu, vmax, o);
      if (other > vmax) vmax = other;
    }
    if (lane == 0) atomic_max_nonneg(A.norm_slot, vmax);
  }
}

#endif
