/*
 * coarse.cu -- the coarse end of the multigrid cycle as ONE single-thread-block kernel.
 *
 * Levels of at most 512 cells (8^3 and coarser in the benchmark) carry no work but ~55 % of the kernel
 * launches of an F-cycle (SURVEY.md appendix C): every operator there is a few microseconds of launch
 * latency around nanoseconds of work.  This kernel runs, for a chain of such levels c..bottom that live
 * entirely on this GPU,
 *
 *   MODE_VCYCLE : MGVCycle(c)                                             (mg.c:1135-1164)
 *   MODE_FTAIL  : the coarse tail of FMGSolve (mg.c:1285-1301): zero(e_bottom); bottom solve;
 *                 for l = bottom-1 .. c: interpolation_fcycle(l <- l+1); MGVCycle(l)
 *
 * with __syncthreads() where the stream version has kernel boundaries.
 *
 * Residency.  A single-box level keeps the vectors the cycle touches (TEMP, e, R, Dinv, beta_i/j/k; on the
 * bottom level also the 8 Krylov vectors; under L1-Jacobi the level's L1 row inverse, which is not in the slab)
 * in shared memory for the duration of the kernel: 160 KB for 8^3 + 4^3 + 2^3.  They arrive and leave as bulk
 * asynchronous copies (cp.async.bulk, one per vector, issued by one thread and counted by an mbarrier).  The phase program addresses vectors by SLOT, so the same
 * operator bodies run on a level that stays in global memory (slot == vector id there).
 *
 * Speed.  A phase is latency-bound: one warp issuing the instructions of one fv4 stencil.  The resident
 * single-box levels of 8^3, 4^3 and 2^3 cells therefore get bodies specialised on the box size -- strides
 * are compile-time constants, the slab is addressed as shared memory, every stencil operand is a load at an
 * immediate offset (~190 instead of ~600 instructions per stencil) -- and a ghost fill that derives its
 * boundary-condition columns from the thread index instead of walking tables in global memory.  Every
 * other level (other sizes, several boxes, not resident) runs the generic bodies over the same tables as
 * the level-wide kernels.  All of them evaluate the same expressions (stencil.cuh, bc.cuh, bicgstab.cuh),
 * so the bits are those of the multi-launch path
 * (tests/test_gpu_parity.py::test_coarse_kernel_equals_multilaunch_path).
 */
#include <math.h>
#include "common.cuh"
#include "stencil.cuh"
#include "bc.cuh"
#include "bicgstab.cuh"

#define COARSE_MAX_LEVELS 8
#define COARSE_THREADS    512
#define COARSE_MAX_SLOTS  24
#define COARSE_SMEM_MAX   231424                    /* dynamic shared memory the kernel may ask for: 227 KB minus its static variables */

enum { MODE_VCYCLE = 0, MODE_FTAIL = 1 };

struct CoarseLevel {
  DLevel L;                                       /* as the kernel sees it: base = shared-memory copy (patched in-kernel) or the global slab;
                                                     nvec = number of slots */
  double *gbase;                                  /* the level's slab in global memory */
  const int *low;
  const FillCopy *xch[2];                         /* [0] NO_CORNERS, [1] BOX: one record per ghost cell copied   */
  const FillBC *bc[2];                            /*                          one record per BC column            */
  int n_xch[2], n_bc[2];
  const blockCopy_type *restr, *interp;           /* local transfer lists */
  int n_restr, n_interp;
  int restr_cells, interp_cells;                  /* cells of the largest entry of each list */
  double h2inv;
  double c1[6], c2[6];                            /* Chebyshev coefficients of this level */
  double jw;                                      /* Jacobi weight (jacobi.c): 2/3 with lambda = Dinv, 1 with the L1 row inverse */
  const double *l1;                               /* L1-Jacobi: the level's L1 row inverse in global memory ([box][volume]) */
  int s_lam;                                      /* slot of lambda; -1: read it from l1.  == nslots on a resident level under L1-Jacobi:
                                                     the resident copy of l1, right after the slots */
  int smem_offset;                                /* >=0: resident, doubles from the start of the pool */
  int nslots;
  int fast;                                       /* 8, 4, 2: resident single box of that size, specialised bodies; 0: generic */
  int s_dinv, s_bi, s_bj, s_bk;                   /* slots of the operator data */
  unsigned char slot_id[COARSE_MAX_SLOTS];        /* slot -> vector id */
  unsigned char slot_io[COARSE_MAX_SLOTS];        /* bit 0: load at entry, bit 1: store at exit */
};

/* phase clocks of the last profiled launch (hpgmg_b200_coarse_profile): SM cycles per category */
enum { CP_LOAD = 0, CP_FILL, CP_STENCIL, CP_RESTRICT, CP_ZERO, CP_INTERP, CP_BOTTOM, CP_STORE, CP_TOTAL, CP_N };
__device__ long long g_coarse_prof[CP_N];
__shared__ long long s_prof[CP_N + 1];
#define CPROF(cat) do { if (s_prof_on && threadIdx.x == 0) { const long long t_ = clock64(); s_prof[cat] += t_ - s_prof[CP_N]; s_prof[CP_N] = t_; } } while (0)
__shared__ int s_prof_on;

/* The cycle is handed to the kernel as a PROGRAM of phases (built on the host by the same recursion the stream
 * version runs, p_vcycle / p_ftail below) and executed by one loop with one switch, so that every operator body
 * exists once in the binary.  Vector operands are slots of the phase's level. */
enum { PH_FILL = 0, PH_STENCIL, PH_RESTRICT_ZERO, PH_ZERO, PH_INTERP3, PH_INTERP5, PH_BOTTOM };
struct Phase { unsigned char op, lv, a, b, c, d, e, f; };
#define COARSE_MAX_PHASES 384

struct CoarseArgs {
  int nlevels, mode, smoother, profile, nphases;
  int e_slot_bottom, R_slot_bottom;
  BottomIds bottom_ids;
  double a, b, rtol;
  double *krylov;
  CoarseLevel lv[COARSE_MAX_LEVELS];
  Phase prog[COARSE_MAX_PHASES];
};

/* ---- box geometry known at compile time (level.c:935-938) ------------------------------------------ */
template <int N>
struct Geo {
  static constexpr int P = N + 4;                                  /* padded extent, ghosts = 2 */
  static constexpr int jS = (P + 3) / 4 * 4, kS = jS * P, VOL = kS * P;
  static constexpr int ORG = 2 * (1 + jS + kS);
};
template <int JS, int KS>
struct FixedLoader {                                               /* p points at cell ijk of an array with compile-time strides */
  const double *p;
  __device__ __forceinline__ double operator()(const int di, const int dj, const int dk) const { return p[di + dj * JS + dk * KS]; }
};

/* ---- generic bodies: any level, through the flat tables of the level-wide kernels ------------------ */
/* exchange_boundary + apply_BCs_v4 (or v2) for one shape: copies and BC columns are independent of each other
 * (FillBC::src), so this is a single phase */
__device__ static void c_fill_ghosts(const CoarseLevel &V, const int slot, const bool box_shape, const bool force_v2)
{
  const DLevel &L = V.L;
  double *v = L.base + (size_t)slot * (size_t)L.volume;
  const int w = box_shape ? 1 : 0;
  const bool v2 = force_v2 || L.dim < 4;
  const int ncopies = V.n_xch[w], work = ncopies + V.n_bc[w];
  for (int e = threadIdx.x; e < work; e += blockDim.x) {
    if (e < ncopies) {
      const FillCopy c = V.xch[w][e];
      v[c.dst] = v[c.src];
    } else {
      const FillBC it = V.bc[w][e - ncopies];
      const BCNormal N = bc_normal(it.subtype, L.jStride, L.kStride);
      if (v2) bc_v2_col_zero_rest(v + it.src, v + it.dst, N.m, N.d[0], N.d[1], N.d[2]);
      else    bc_v4_column(v + it.src, v + it.dst, N);
    }
  }
}

/* one sweep / residual over every cell of every box.  mode: 0 GSRB sweep s, 1 Chebyshev sweep s, 2 residual, 3 Jacobi sweep.
 * GSRB on even boxes: a thread owns an i-pair (exactly one active cell per pair, so no lane idles). */
__device__ static void c_stencil(const CoarseLevel &V, const int mode, const int src, const int dst, const int rhs_slot, const int s, const double b)
{
  const DLevel &L = V.L;
  const int n = L.dim, jS = L.jStride, kS = L.kStride;
  if (mode == 0 && (n & 1) == 0) {
    const int hn = n >> 1, per_box = hn * n * n, total = per_box * L.nboxes;
    for (int q = threadIdx.x; q < total; q += blockDim.x) {
      const int box = q / per_box, c = q - box * per_box;
      const int p = c % hn, j = (c / hn) % n, k = c / (hn * n);
      const int ijk = 2 * p + j * jS + k * kS;
      const double *x = L.vec(box, src) + ijk;
      const double *rhs = L.vec(box, rhs_slot) + ijk;
      double *out = L.vec(box, dst) + ijk;
      const int color000 = (V.low[3 * box] ^ V.low[3 * box + 1] ^ V.low[3 * box + 2] ^ s) & 1;
      const int a = (j ^ k ^ color000) & 1;
      const double Ax = fv4_apply_op(x + a, L.vec(box, V.s_bi) + ijk + a, L.vec(box, V.s_bj) + ijk + a, L.vec(box, V.s_bk) + ijk + a, jS, kS, b, V.h2inv);
      const double xnew = x[a] + L.vec(box, V.s_dinv)[ijk + a] * (rhs[a] - Ax);
      out[1 - a] = x[1 - a];
      out[a] = xnew;
    }
    return;
  }
  const int cells = n * n * n, total = cells * L.nboxes;
  for (int q = threadIdx.x; q < total; q += blockDim.x) {
    const int box = q / cells, c = q - box * cells;
    const int i = c % n, j = (c / n) % n, k = c / (n * n);
    const int ijk = i + j * jS + k * kS;
    const double *x = L.vec(box, src) + ijk;
    double *out = L.vec(box, dst) + ijk;
    if (mode == 0) {
      const int color000 = (V.low[3 * box] ^ V.low[3 * box + 1] ^ V.low[3 * box + 2] ^ s) & 1;
      if ((i ^ j ^ k ^ color000) & 1) { out[0] = x[0]; continue; }
    }
    const double Ax = fv4_apply_op(x, L.vec(box, V.s_bi) + ijk, L.vec(box, V.s_bj) + ijk, L.vec(box, V.s_bk) + ijk, jS, kS, b, V.h2inv);
    const double rhs = L.vec(box, rhs_slot)[ijk];
    if (mode == 2) { out[0] = rhs - Ax; continue; }
    if (mode == 3) {                                                /* jacobi.c: x_n + weight*lambda*(rhs - Ax_n) */
      const double lam = V.s_lam >= 0 ? L.vec(box, V.s_lam)[ijk] : V.l1[(size_t)box * L.volume + L.origin + ijk];
      out[0] = x[0] + (V.jw * lam) * (rhs - Ax);
      continue;
    }
    const double dinv = L.vec(box, V.s_dinv)[ijk];
    if (mode == 0) out[0] = x[0] + dinv * (rhs - Ax);
    else { const double xn = x[0]; out[0] = xn + V.c1[s] * (xn - out[0]) + V.c2[s] * dinv * (rhs - Ax); }
  }
}

__device__ static void c_zero(const DLevel &L, const int slot)
{
  const int m = L.dim + 2 * L.ghosts, cells = m * m * m, total = cells * L.nboxes;
  for (int q = threadIdx.x; q < total; q += blockDim.x) {
    const int box = q / cells, c = q - box * cells;
    const int i = c % m - L.ghosts, j = (c / m) % m - L.ghosts, k = c / (m * m) - L.ghosts;
    L.vec(box, slot)[i + j * L.jStride + k * L.kStride] = 0.0;
  }
}

/* restriction.c:54-57 over the local list of the fine level, all entries spread over the whole block */
__device__ static void c_restrict_cell(const DLevel &Lc, const int slot_c, const DLevel &Lf, const int slot_f, const blockCopy_type *blocks, const int n, const int entry_cells)
{
  const int rj = Lf.jStride, rk = Lf.kStride;
  for (int w = threadIdx.x; w < n * entry_cells; w += blockDim.x) {
    const int e = w / entry_cells, c = w - e * entry_cells;
    const blockCopy_type &B = blocks[e];
    const int di = B.dim.i, dj = B.dim.j;
    if (c >= di * dj * B.dim.k) continue;
    const int i = c % di, j = (c / di) % dj, k = c / (di * dj);
    const double *r = Lf.vec(B.read.box, slot_f) + (B.read.i + 2 * i) + (B.read.j + 2 * j) * rj + (B.read.k + 2 * k) * rk;
    Lc.vec(B.write.box, slot_c)[(B.write.i + i) + (B.write.j + j) * Lc.jStride + (B.write.k + k) * Lc.kStride] =
        (r[0] + r[1] + r[rj] + r[1 + rj] + r[rk] + r[1 + rk] + r[rj + rk] + r[1 + rj + rk]) * 0.125;
  }
}

__device__ __forceinline__ void c_pro3(const double cm, const double c0, const double cp, double &lo, double &hi)
{
  const double c1 = 1.0 / 8.0;
  lo = (c0 + c1 * (cm - cp));
  hi = (c0 - c1 * (cm - cp));
}
__device__ __forceinline__ void c_pro5(const double cmm, const double cm, const double c0, const double cp, const double cpp, double &lo, double &hi)
{
  const double c2 = -3.0 / 128.0, c1 = 22.0 / 128.0;
  lo = (c0 + c1 * (cm - cp) + c2 * (cmm - cpp));
  hi = (c0 - c1 * (cm - cp) - c2 * (cmm - cpp));
}

/* interpolation_v2.c:112-172 (W=3) / interpolation_v4.c:149-238 (W=5) over the coarse level's local list: one thread per
 * coarse cell; i-pass and j-pass plane by plane, then the k-pass (the order of interpolation_kernel, transfer.cu) */
template <int W>
__device__ static void c_interpolate(const DLevel &Lf, const int slot_f, const double prescale, const DLevel &Lc, const int slot_c, const blockCopy_type *blocks, const int n, const int entry_cells)
{
  constexpr int R = W / 2;
  const int rj = Lc.jStride, rk = Lc.kStride, wj = Lf.jStride, wk = Lf.kStride;
  for (int wi = threadIdx.x; wi < n * entry_cells; wi += blockDim.x) {
    const int e = wi / entry_cells, c = wi - e * entry_cells;
    const blockCopy_type &B = blocks[e];
    const int di = B.dim.i, dj = B.dim.j;
    if (c >= di * dj * B.dim.k) continue;
    const int ii = c % di, jj = (c / di) % dj, kk = c / (di * dj);
    const double *r = Lc.vec(B.read.box, slot_c) + (ii + B.read.i) + (jj + B.read.j) * rj + (kk + B.read.k) * rk;
    double fj[2][2][W];
#pragma unroll
    for (int K = 0; K < W; K++) {
      double fi[2][W];
#pragma unroll
      for (int J = 0; J < W; J++) {
        const double *p = r + (J - R) * rj + (K - R) * rk;
        if constexpr (W == 3) c_pro3(p[-1], p[0], p[1], fi[0][J], fi[1][J]);
        else                  c_pro5(p[-2], p[-1], p[0], p[1], p[2], fi[0][J], fi[1][J]);
      }
#pragma unroll
      for (int I = 0; I < 2; I++) {
        if constexpr (W == 3) c_pro3(fi[I][0], fi[I][1], fi[I][2], fj[I][0][K], fj[I][1][K]);
        else                  c_pro5(fi[I][0], fi[I][1], fi[I][2], fi[I][3], fi[I][W - 1], fj[I][0][K], fj[I][1][K]);
      }
    }
    double *w = Lf.vec(B.write.box, slot_f) + (2 * ii + B.write.i) + (2 * jj + B.write.j) * wj + (2 * kk + B.write.k) * wk;
#pragma unroll
    for (int J = 0; J < 2; J++)
#pragma unroll
    for (int I = 0; I < 2; I++) {
      double lo, hi;
      if constexpr (W == 3) c_pro3(fj[I][J][0], fj[I][J][1], fj[I][J][2], lo, hi);
      else                  c_pro5(fj[I][J][0], fj[I][J][1], fj[I][J][2], fj[I][J][3], fj[I][J][W - 1], lo, hi);
      double *w0 = w + I + J * wj;
      w0[0] = prescale * w0[0] + lo;
      w0[wk] = prescale * w0[wk] + hi;
    }
  }
}

/* ---- bodies specialised on the box size: resident single-box levels -------------------------------- */
/* Ghost fill of ONE box whose six faces are all domain boundary (homogeneous Dirichlet): no copies, and the BC
 * columns follow from the thread index: 6 N^2 face columns, 12 N edge columns, 8 corner columns (BOX shape only).
 * v points at cell (0,0,0).  Same column bodies as everywhere else (bc.cuh), normal axes in ascending order.  The
 * strides of a column are DATA (selected, not branched on), so the lanes of a warp that work on different faces or
 * edges still run one instruction stream: branching per face/edge cost 4 serialised 16-point extrapolations per warp. */
template <int N>
__device__ static void c_fill_fast(double *v, const bool box_shape, const bool force_v2)
{
  typedef Geo<N> G;
  constexpr int NF = 6 * N * N, NE = 12 * N;
  const bool v2 = force_v2 || N < 4;
  const int work = NF + NE + (box_shape ? 8 : 0);
  for (int t = threadIdx.x; t < work; t += blockDim.x) {
    if (t < NF) {
      const int f = t / (N * N), c = t - f * (N * N), p = c % N, q = c / N;
      const int axis = f >> 1, hi = f & 1;
      const int S0 = axis == 0 ? 1 : (axis == 1 ? G::jS : G::kS);
      const int T0 = axis == 0 ? G::jS : 1, T1 = axis == 2 ? G::jS : G::kS;      /* the two tangential strides */
      double *w = v + (hi ? N : -1) * S0 + p * T0 + q * T1;
      const int d0 = hi ? -S0 : S0;
      if (v2) bc_v2_col_zero_rest(w, w, 1, d0, 0, 0);
      else    bc_v4_col1(w, w, d0);
    } else if (t < NF + NE) {
      const int e = (t - NF) / N, p = (t - NF) - e * N;
      const int pair = e >> 2, hi0 = e & 1, hi1 = (e >> 1) & 1;                 /* normal axes (0,1), (0,2), (1,2) */
      const int S0 = pair == 2 ? G::jS : 1, S1 = pair == 0 ? G::jS : G::kS;
      const int T = pair == 0 ? G::kS : (pair == 1 ? G::jS : 1);
      double *w = v + (hi0 ? N : -1) * S0 + (hi1 ? N : -1) * S1 + p * T;
      const int d0 = hi0 ? -S0 : S0, d1 = hi1 ? -S1 : S1;
      if (v2) bc_v2_col_zero_rest(w, w, 2, d0, d1, 0);
      else    bc_v4_col2(w, w, d0, d1);
    } else {
      const int c = t - NF - NE;
      const int h0 = c & 1, h1 = (c >> 1) & 1, h2 = (c >> 2) & 1;
      double *w = v + (h0 ? N : -1) + (h1 ? N : -1) * G::jS + (h2 ? N : -1) * G::kS;
      const int d0 = h0 ? -1 : 1, d1 = h1 ? -G::jS : G::jS, d2 = h2 ? -G::kS : G::kS;
      if (v2) bc_v2_col_zero_rest(w, w, 3, d0, d1, d2);
      else    bc_v4_col3(w, w, d0, d1, d2);
    }
  }
}

/* one sweep / residual of ONE box of N^3 cells whose low corner is the domain's; `base` points at cell (0,0,0) of slot 0,
 * strides Geo<N>.  GSRB: one thread per i-pair = per updated cell; Chebyshev / Jacobi / residual: one thread per cell.
 * Resident levels only: lambda of a Jacobi sweep is always in a slot there. */
template <int N>
__device__ static void c_stencil_fast(const CoarseLevel &V, double *base, const int mode, const int src, const int dst, const int rhs_slot, const int s, const double b)
{
  typedef Geo<N> G;
  constexpr int LG = N == 8 ? 3 : (N == 4 ? 2 : 1);
  const double *x = base + src * G::VOL, *bi = base + V.s_bi * G::VOL, *bj = base + V.s_bj * G::VOL, *bk = base + V.s_bk * G::VOL;
  const double *rhs = base + rhs_slot * G::VOL, *dinv = base + V.s_dinv * G::VOL, *lam = base + V.s_lam * G::VOL;
  double *out = base + dst * G::VOL;
  const double h2inv = V.h2inv;
  const int work = mode == 0 ? N * N * N / 2 : N * N * N;
  for (int q = threadIdx.x; q < work; q += blockDim.x) {
    int i, j, k;
    if (mode == 0) {
      int p;
      if (N == 8) {
        /* a warp = 4 pairs x 4 rows x 2 planes: with jStride 12 and kStride 144 the 16 lanes of a plane fall into 16 distinct
         * 8-byte banks and the two planes (opposite colour) into the same 16 again: 2 wavefronts per 64-bit load, the minimum */
        p = q & 3;  j = ((q >> 2) & 3) | (((q >> 5) & 1) << 2);  k = ((q >> 4) & 1) | (((q >> 6) & 3) << 1);
      } else {
        p = q & (N / 2 - 1);  j = (q >> (LG - 1)) & (N - 1);  k = q >> (2 * LG - 1);
      }
      i = 2 * p + ((j ^ k ^ s) & 1);                                /* the pair's active cell (gsrb.c:55,100); box low = 0,0,0 */
    } else {
      i = q & (N - 1);  j = (q >> LG) & (N - 1);  k = q >> (2 * LG);
    }
    const int ijk = i + j * G::jS + k * G::kS;
    const FixedLoader<G::jS, G::kS> X = { x + ijk }, BI = { bi + ijk }, BJ = { bj + ijk }, BK = { bk + ijk };
    const double Ax = fv4_apply_op_at(X, BI, BJ, BK, b, h2inv);
    if (mode == 0) {
      const double xnew = x[ijk] + dinv[ijk] * (rhs[ijk] - Ax);
      out[ijk ^ 1] = x[ijk ^ 1];                                    /* the pair's other cell is copied (gsrb.c:65-71); strides are even */
      out[ijk] = xnew;
    } else if (mode == 2) {
      out[ijk] = rhs[ijk] - Ax;
    } else if (mode == 3) {
      out[ijk] = x[ijk] + (V.jw * lam[ijk]) * (rhs[ijk] - Ax);     /* jacobi.c */
    } else {
      const double xn = x[ijk];
      out[ijk] = xn + V.c1[s] * (xn - out[ijk]) + V.c2[s] * dinv[ijk] * (rhs[ijk] - Ax);     /* x_{n-1} aliases x_{n+1} (chebyshev.c:75-80) */
    }
  }
}

__device__ static void c_bottom_solve(const CoarseArgs &A, double *prod, double *red)
{
  const CoarseLevel &V = A.lv[A.nlevels - 1];
  BottomArgs B;
  B.L = V.L;  B.bc = V.bc[0];  B.nbc = V.n_bc[0];
  B.x_id = A.e_slot_bottom;  B.R_id = A.R_slot_bottom;  B.ids = A.bottom_ids;
  B.a = A.a;  B.b = A.b;  B.h2inv = V.h2inv;  B.rtol = A.rtol;  B.iters = A.krylov;
  bicgstab_solve(B, prod, red);
}

/* ---- bulk asynchronous copies between the global slabs and the resident copies ---------------------- */
__device__ __forceinline__ void bulk_load(double *smem_dst, const double *gmem_src, const unsigned bytes, const unsigned bar)
{
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"((unsigned)__cvta_generic_to_shared(smem_dst)), "l"(gmem_src), "r"(bytes), "r"(bar) : "memory");
}
__device__ __forceinline__ void bulk_store(double *gmem_dst, const double *smem_src, const unsigned bytes)
{
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gmem_dst), "r"((unsigned)__cvta_generic_to_shared(smem_src)), "r"(bytes) : "memory");
}

__global__ void __launch_bounds__(COARSE_THREADS, 1) coarse_cycle_kernel(const __grid_constant__ CoarseArgs Ain)
{
  extern __shared__ __align__(128) double dyn[];
  __shared__ __align__(8) unsigned long long s_bar;
  CoarseArgs &A = *reinterpret_cast<CoarseArgs *>(dyn);
  constexpr int ARGS_DOUBLES = (int)((sizeof(CoarseArgs) + 127) / 128) * 16;
  double *prod = dyn + ARGS_DOUBLES;
  double *red = prod + BOTTOM_MAX_CELLS + 1;
  double *pool = red + 34 + ((16 - (BOTTOM_MAX_CELLS + 1 + 34) % 16) % 16);        /* a multiple of 128 bytes from dyn: bulk copies need 16 */
  const unsigned bar = (unsigned)__cvta_generic_to_shared(&s_bar);
  if (threadIdx.x == 0) {
    s_prof_on = Ain.profile;
    for (int c = 0; c < CP_N; c++) s_prof[c] = 0;
    s_prof[CP_N] = clock64();  s_prof[CP_TOTAL] = -s_prof[CP_N];
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  {                                                                /* stage the arguments (kernel parameters, not memory: before the wait) */
    const int *src = reinterpret_cast<const int *>(&Ain);
    int *dst = reinterpret_cast<int *>(dyn);
    for (int w = threadIdx.x; w < (int)(sizeof(CoarseArgs) / sizeof(int)); w += blockDim.x) dst[w] = src[w];
  }
  __syncthreads();
  PDL_WAIT();
  if (threadIdx.x == 0) {                                          /* request the resident vectors: one bulk copy each */
    unsigned total = 0;
    for (int l = 0; l < Ain.nlevels; l++) {
      const CoarseLevel &G = Ain.lv[l];
      if (G.smem_offset < 0) continue;
      A.lv[l].L.base = pool + G.smem_offset;
      for (int sl = 0; sl < G.nslots; sl++) if (G.slot_io[sl] & 1) total += (unsigned)G.L.volume * 8u;
      if (G.s_lam == G.nslots) total += (unsigned)G.L.volume * 8u;
    }
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(total) : "memory");
    for (int l = 0; l < Ain.nlevels; l++) {
      const CoarseLevel &G = Ain.lv[l];
      if (G.smem_offset < 0) continue;
      for (int sl = 0; sl < G.nslots; sl++)
        if (G.slot_io[sl] & 1) bulk_load(pool + G.smem_offset + (size_t)sl * G.L.volume, G.gbase + (size_t)G.slot_id[sl] * G.L.volume, (unsigned)G.L.volume * 8u, bar);
      if (G.s_lam == G.nslots) bulk_load(pool + G.smem_offset + (size_t)G.nslots * G.L.volume, G.l1, (unsigned)G.L.volume * 8u, bar);     /* read-only */
    }
  }
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "COARSE_WAIT:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], 0;\n"
      "@p bra COARSE_DONE;\n"
      "bra COARSE_WAIT;\n"
      "COARSE_DONE:\n"
      "}\n" ::"r"(bar) : "memory");
  __syncthreads();
  CPROF(CP_LOAD);

#pragma unroll 1
  for (int ph = 0; ph < A.nphases; ph++) {
    const Phase P = A.prog[ph];
    const CoarseLevel &V = A.lv[P.lv];
    double *fb = pool + V.smem_offset;                              /* shared-memory address space stays visible to the compiler on the fast paths */
    switch (P.op) {
      case PH_FILL:
        if (V.fast == 8)      c_fill_fast<8>(fb + Geo<8>::ORG + P.a * Geo<8>::VOL, P.b != 0, P.c != 0);
        else if (V.fast == 4) c_fill_fast<4>(fb + Geo<4>::ORG + P.a * Geo<4>::VOL, P.b != 0, P.c != 0);
        else if (V.fast == 2) c_fill_fast<2>(fb + Geo<2>::ORG + P.a * Geo<2>::VOL, P.b != 0, P.c != 0);
        else                  c_fill_ghosts(V, P.a, P.b != 0, P.c != 0);
        __syncthreads();
        CPROF(CP_FILL);
        break;
      case PH_STENCIL:
        if (V.fast == 8)      c_stencil_fast<8>(V, fb + Geo<8>::ORG, P.a, P.b, P.c, P.d, P.e, A.b);
        else if (V.fast == 4) c_stencil_fast<4>(V, fb + Geo<4>::ORG, P.a, P.b, P.c, P.d, P.e, A.b);
        else if (V.fast == 2) c_stencil_fast<2>(V, fb + Geo<2>::ORG, P.a, P.b, P.c, P.d, P.e, A.b);
        else                  c_stencil(V, P.a, P.b, P.c, P.d, P.e, A.b);
        __syncthreads();
        CPROF(CP_STENCIL);
        break;
      case PH_RESTRICT_ZERO:                                        /* restriction(l+1, R <- l, TEMP) and zero_vector(l+1, e): independent */
        c_restrict_cell(A.lv[P.lv + 1].L, P.a, V.L, P.b, V.restr, V.n_restr, V.restr_cells);
        c_zero(A.lv[P.lv + 1].L, P.c);
        __syncthreads();
        CPROF(CP_RESTRICT);
        break;
      case PH_ZERO:
        c_zero(V.L, P.a);
        __syncthreads();
        CPROF(CP_ZERO);
        break;
      case PH_INTERP3:
        c_interpolate<3>(V.L, P.a, 1.0, A.lv[P.lv + 1].L, P.b, A.lv[P.lv + 1].interp, A.lv[P.lv + 1].n_interp, A.lv[P.lv + 1].interp_cells);
        __syncthreads();
        CPROF(CP_INTERP);
        break;
      case PH_INTERP5:
        c_interpolate<5>(V.L, P.a, 0.0, A.lv[P.lv + 1].L, P.b, A.lv[P.lv + 1].interp, A.lv[P.lv + 1].n_interp, A.lv[P.lv + 1].interp_cells);
        __syncthreads();
        CPROF(CP_INTERP);
        break;
      default:
        c_bottom_solve(A, prod, red);
        __syncthreads();
        CPROF(CP_BOTTOM);
        break;
    }
  }

  /* write the vectors the cycle produced back (TEMP, e, R; the operator data is read-only) */
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");      /* this thread's generic-proxy writes -> visible to the bulk-copy engine */
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int l = 0; l < Ain.nlevels; l++) {
      const CoarseLevel &G = Ain.lv[l];
      if (G.smem_offset < 0) continue;
      for (int sl = 0; sl < G.nslots; sl++)
        if (G.slot_io[sl] & 2) bulk_store(G.gbase + (size_t)G.slot_id[sl] * G.L.volume, pool + G.smem_offset + (size_t)sl * G.L.volume, (unsigned)G.L.volume * 8u);
    }
    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
    asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
  }
  __syncthreads();
  CPROF(CP_STORE);
  if (s_prof_on && threadIdx.x == 0) { s_prof[CP_TOTAL] += clock64(); for (int c = 0; c < CP_N; c++) g_coarse_prof[c] = s_prof[c]; }
}

/* ---- host side ------------------------------------------------------------------------------------ */
static int coarse_program_length(int nlevels, int ftail);
static int g_coarse_enabled = -1;
static int g_coarse_smem = 1;
static int g_coarse_fast = 1;
static int g_coarse_profile = 0;
/* cycles per phase category of the next/last coarse kernel launch: load, fill, stencil, restrict, zero, interp, bottom, store, total */
extern "C" void hpgmg_b200_coarse_profile(int on, long long *out9)
{
  g_coarse_profile = on;
  if (out9) {
    CUDA_CHECK(cudaStreamSynchronize(g_stream));
    CUDA_CHECK(cudaMemcpyFromSymbol(out9, g_coarse_prof, sizeof(long long) * CP_N));
  }
}
/* single-block cycles pay off up to 8^3 (one cell per thread, latency-bound); 16^3 is faster as separate launches */
static long g_coarse_max_cells = 512;
extern "C" void hpgmg_b200_coarse_levels_in_smem(int on) { if ((on ? 1 : 0) != g_coarse_smem) hpgmg_graph_drop_all(NULL); g_coarse_smem = on ? 1 : 0; }
extern "C" void hpgmg_b200_use_coarse_kernel(int on) { if ((on ? 1 : 0) != g_coarse_enabled) hpgmg_graph_drop_all(NULL); g_coarse_enabled = on ? 1 : 0; }

static int level_is_coarse_eligible(const level_type *level, int is_top, int is_bottom)
{
  if (level->num_my_boxes != level->boxes_in.i * level->boxes_in.j * level->boxes_in.k) return 0;   /* every box of the level is mine */
  if (level->boundary_condition.type != BC_DIRICHLET || level->must_subtract_mean == 1) return 0;
  if (HPGMG_DEV(level)->fill_nvec != level->numVectors) return 0;
  if (level->numVectors > COARSE_MAX_SLOTS || level->box_ghosts != 2) return 0;
  if ((long)level->dim.i * level->dim.j * level->dim.k > g_coarse_max_cells) return 0;
  for (int s = 0; s < STENCIL_MAX_SHAPES; s++)
    if (level->exchange_ghosts[s].num_sends || level->exchange_ghosts[s].num_recvs) return 0;
  /* transfers BETWEEN chain levels must be local; those across the top of the chain run outside the kernel */
  if (!is_bottom && (level->restriction[RESTRICT_CELL].num_sends || level->interpolation.num_recvs)) return 0;
  if (!is_top && (level->restriction[RESTRICT_CELL].num_recvs || level->interpolation.num_sends)) return 0;
  return 1;
}

/* Can levels `from`..bottom of this hierarchy run in the single-block kernel?  (all of them small,
 * entirely local to this rank, Dirichlet, and a single-box bottom the BiCGStab body can solve) */
extern "C" int hpgmg_coarse_chain_eligible(mg_type *MG, int from)
{
  if (g_coarse_enabled < 0) {
    const char *e = getenv("HPGMG_B200_NO_COARSE_KERNEL");
    g_coarse_enabled = (e && atoi(e)) ? 0 : 1;
    const char *m = getenv("HPGMG_B200_COARSE_MAX_CELLS");
    if (m && atol(m) > 0) g_coarse_max_cells = atol(m) > COARSE_MAX_CELLS ? COARSE_MAX_CELLS : atol(m);
    const char *f = getenv("HPGMG_B200_COARSE_FAST");               /* 0: generic bodies on every level (A/B parity check) */
    if (f) g_coarse_fast = atoi(f);
  }
  if (!g_coarse_enabled) return 0;
#ifdef VECTOR_ALPHA
  return 0;                                        /* Helmholtz build: the global-memory kernels carry the a*alpha*x term */
#endif
  const int bottom = MG->num_levels - 1;
  if (from > bottom || bottom - from + 1 > COARSE_MAX_LEVELS) return 0;
  if (coarse_program_length(bottom - from + 1, 1) > COARSE_MAX_PHASES) return 0;
  for (int l = from; l <= bottom; l++) if (!level_is_coarse_eligible(MG->levels[l], l == from, l == bottom)) return 0;
  const level_type *B = MG->levels[bottom];
  if (B->num_my_boxes != 1 || B->boxes_in.i != 1 || B->box_dim > BOTTOM_MAX_DIM || B->box_dim < 2) return 0;
  if (B->numVectors < VECTORS_RESERVED + 8) return 0;
  return 1;
}

/* ---- the phase program: the recursion of the stream version, recorded instead of executed ---- */
struct Slots { int temp, e, R; };                                   /* per level: slots of the cycle's vectors */
static void p_add(CoarseArgs &A, int op, int lv, int a = 0, int b = 0, int c = 0, int d = 0, int e = 0)
{
  if (A.nphases >= COARSE_MAX_PHASES) { fprintf(stderr, "hpgmg_b200: coarse-cycle program too long\n"); exit(1); }
  Phase P = { (unsigned char)op, (unsigned char)lv, (unsigned char)a, (unsigned char)b, (unsigned char)c, (unsigned char)d, (unsigned char)e, 0 };
  A.prog[A.nphases++] = P;
}
static void p_smooth(CoarseArgs &A, const Slots *S, int l)                  /* smooth(): gsrb.c:24-132 / chebyshev.c:8-100 / jacobi.c */
{
  const int mode = A.smoother == HPGMG_SMOOTHER_CHEBY ? 1 : (A.smoother == HPGMG_SMOOTHER_JACOBI || A.smoother == HPGMG_SMOOTHER_L1JACOBI) ? 3 : 0;
  for (int s = 0; s < 6; s++) {
    const int src = (s & 1) ? S[l].temp : S[l].e, dst = (s & 1) ? S[l].e : S[l].temp;
    p_add(A, PH_FILL, l, src, 0, 0);
    p_add(A, PH_STENCIL, l, mode, src, dst, S[l].R, s);
  }
}
static void p_vcycle(CoarseArgs &A, const Slots *S, int c)                  /* MGVCycle: mg.c:1135-1164 */
{
  const int bottom = A.nlevels - 1;
  for (int l = c; l < bottom; l++) {
    p_smooth(A, S, l);
    p_add(A, PH_FILL, l, S[l].e, 0, 0);                                    /* residual(): exchange + BC on x */
    p_add(A, PH_STENCIL, l, 2, S[l].e, S[l].temp, S[l].R, 0);
    p_add(A, PH_RESTRICT_ZERO, l, S[l + 1].R, S[l].temp, S[l + 1].e);      /* restriction(l+1,R <- l,TEMP); zero_vector(l+1,e) */
  }
  p_add(A, PH_BOTTOM, bottom);
  for (int l = bottom - 1; l >= c; l--) {
    p_add(A, PH_FILL, l + 1, S[l + 1].e, 1, 1);                            /* interpolation_v2: exchange(BOX) + apply_BCs_v2 on the coarse level */
    p_add(A, PH_INTERP3, l, S[l].e, S[l + 1].e);
    p_smooth(A, S, l);
  }
}
static int coarse_program_length(int nlevels, int ftail)
{
  int v = 0, total = 0;                                                     /* phases of MGVCycle(c): 29 per non-bottom level + 1 */
  for (int c = nlevels - 1; c >= 0; c--) {
    v = 29 * (nlevels - 1 - c) + 1;
    if (ftail && c < nlevels - 1) total += 2 + v;
  }
  return ftail ? total + 2 : v;
}

extern "C" void hpgmg_coarse_cycle(mg_type *MG, int from, int mode_ftail, int zero_bottom, int e_id, int R_id, double a, double b)
{
  static CoarseArgs A;                        /* ~6 KB: passed by value as a __grid_constant__ parameter */
  const int bottom = MG->num_levels - 1;
  memset(&A, 0, sizeof(A));
  A.nlevels = bottom - from + 1;
  A.mode = mode_ftail ? MODE_FTAIL : MODE_VCYCLE;
  A.smoother = hpgmg_rt_smoother();
  A.profile = g_coarse_profile;
  A.a = a;  A.b = b;  A.rtol = MG_DEFAULT_BOTTOM_NORM;
  A.krylov = hpgmg_rt_scalar_slots() + HPGMG_SLOT_KRYLOV;
  Slots S[COARSE_MAX_LEVELS];
  /* residency: from the bottom up while the slots fit in the 227 KB of one SM */
  constexpr size_t ARGS_DOUBLES = ((sizeof(CoarseArgs) + 127) / 128) * 16;
  constexpr size_t FIXED_DOUBLES = ARGS_DOUBLES + BOTTOM_MAX_CELLS + 1 + 34 + 16;
  const size_t budget = COARSE_SMEM_MAX - FIXED_DOUBLES * sizeof(double) - 128;
  size_t used = 0;
  bool stop = false;
  for (int l = bottom; l >= from; l--) {
    level_type *level = MG->levels[l];
    hpgmg_device_level *D = HPGMG_DEV(level);
    CoarseLevel &V = A.lv[l - from];
    V.L = D->L;  V.gbase = D->L.base;  V.low = D->low;
    const int shapes[2] = { STENCIL_SHAPE_NO_CORNERS, STENCIL_SHAPE_BOX };
    for (int w = 0; w < 2; w++) {
      V.xch[w] = D->fill[shapes[w]].copies;  V.n_xch[w] = D->fill[shapes[w]].ncopies;
      V.bc[w] = D->fill[shapes[w]].bc;       V.n_bc[w] = D->fill[shapes[w]].nbc;
    }
    V.restr = D->restriction[RESTRICT_CELL][1].blocks;           V.n_restr = D->restriction[RESTRICT_CELL][1].n;
    V.interp = D->interpolation[1].blocks;                       V.n_interp = D->interpolation[1].n;
    const communicator_type *Cr = &level->restriction[RESTRICT_CELL], *Ci = &level->interpolation;
    for (int e = 0; e < Cr->num_blocks[1]; e++) { const int c = Cr->blocks[1][e].dim.i * Cr->blocks[1][e].dim.j * Cr->blocks[1][e].dim.k; if (c > V.restr_cells) V.restr_cells = c; }
    for (int e = 0; e < Ci->num_blocks[1]; e++) { const int c = Ci->blocks[1][e].dim.i * Ci->blocks[1][e].dim.j * Ci->blocks[1][e].dim.k; if (c > V.interp_cells) V.interp_cells = c; }
    V.h2inv = 1.0 / (level->h * level->h);
    /* Chebyshev coefficients exactly as chebyshev.c:22-40 */
    double beta = 1.000 * level->dominant_eigenvalue_of_DinvA, alpha = 0.125000 * beta;
    double theta = 0.5 * (beta + alpha), delta = 0.5 * (beta - alpha), sigma = theta / delta, rho_n = 1 / sigma;
    V.c1[0] = 0.0;  V.c2[0] = 1 / theta;
    for (int s = 1; s < 6; s++) { double rho_nm1 = rho_n; rho_n = 1.0 / (2.0 * sigma - rho_nm1); V.c1[s] = rho_n * rho_nm1; V.c2[s] = rho_n * 2.0 / delta; }
    const bool l1jacobi = A.smoother == HPGMG_SMOOTHER_L1JACOBI;
    V.jw = l1jacobi ? 1.0 : 2.0 / 3.0;                               /* jacobi.c */
    V.l1 = l1jacobi ? hpgmg_l1inv_array(level) : NULL;

    /* slots: the vectors a cycle touches; identity (slot == vector id) when the level stays in global memory */
    int ids[COARSE_MAX_SLOTS], io[COARSE_MAX_SLOTS], n = 0;
    auto add = [&](int id, int flags) { for (int q = 0; q < n; q++) if (ids[q] == id) { io[q] |= flags; return q; } ids[n] = id; io[n] = flags; return n++; };
    const int s_temp = add(VECTOR_TEMP, 3), s_e = add(e_id, 3), s_R = add(R_id, 3);
    const int s_dinv = add(VECTOR_DINV, 1), s_bi = add(VECTOR_BETA_I, 1), s_bj = add(VECTOR_BETA_J, 1), s_bk = add(VECTOR_BETA_K, 1);
    int kry[8] = { 0 };
    if (l == bottom) for (int q = 0; q < 8; q++) kry[q] = add(VECTORS_RESERVED + q, 0);     /* scratch of the solver: every one is written before it is read */
    const size_t doubles = (size_t)(n + (l1jacobi ? 1 : 0)) * V.L.volume;     /* + the resident copy of the L1 row inverse */
    const box_type *box0 = &level->my_boxes[0];
    const bool single = V.L.nboxes == 1 && box0->low.i == 0 && box0->low.j == 0 && box0->low.k == 0;
    V.smem_offset = -1;
    if (g_coarse_smem && !stop && single && (used + doubles) * sizeof(double) <= budget && ((uintptr_t)V.gbase % 16) == 0 && (V.L.volume % 2) == 0) {
      V.smem_offset = (int)used;
      used += (doubles + 15) / 16 * 16;
      V.nslots = n;  V.L.nvec = n;
      for (int q = 0; q < n; q++) { V.slot_id[q] = (unsigned char)ids[q]; V.slot_io[q] = (unsigned char)io[q]; }
      V.s_dinv = s_dinv;  V.s_bi = s_bi;  V.s_bj = s_bj;  V.s_bk = s_bk;
      V.s_lam = l1jacobi ? n : s_dinv;
      S[l - from].temp = s_temp;  S[l - from].e = s_e;  S[l - from].R = s_R;
      if (l == bottom) {
        BottomIds I = { kry[0], kry[1], kry[2], kry[3], kry[4], kry[5], kry[6], kry[7], s_dinv, s_temp, s_bi, s_bj, s_bk };
        A.bottom_ids = I;
      }
      const int nb = V.L.dim;
      V.fast = (g_coarse_fast && (nb == 8 || nb == 4 || nb == 2) && V.L.jStride == ((nb + 4 + 3) / 4) * 4 && V.L.kStride == V.L.jStride * (nb + 4)) ? nb : 0;
    } else {
      stop = true;                                                    /* keep the resident set contiguous from the bottom */
      V.nslots = 0;
      V.s_dinv = VECTOR_DINV;  V.s_bi = VECTOR_BETA_I;  V.s_bj = VECTOR_BETA_J;  V.s_bk = VECTOR_BETA_K;
      V.s_lam = l1jacobi ? -1 : VECTOR_DINV;
      S[l - from].temp = VECTOR_TEMP;  S[l - from].e = e_id;  S[l - from].R = R_id;
      if (l == bottom) A.bottom_ids = bottom_ids_identity();
      V.fast = 0;
    }
  }
  A.e_slot_bottom = S[bottom - from].e;  A.R_slot_bottom = S[bottom - from].R;
  A.nphases = 0;
  if (A.mode == MODE_VCYCLE) p_vcycle(A, S, 0);
  else {                                                                    /* MODE_FTAIL: mg.c:1285-1301 restricted to the chain */
    const int cb = A.nlevels - 1;
    if (zero_bottom) p_add(A, PH_ZERO, cb, S[cb].e);                        /* mg.c:1285: only if the bottom is not the solve level */
    p_add(A, PH_BOTTOM, cb);
    for (int l = cb - 1; l >= 0; l--) {
      p_add(A, PH_FILL, l + 1, S[l + 1].e, 1, 0);                           /* interpolation_v4: exchange(BOX) + apply_BCs_v4 */
      p_add(A, PH_INTERP5, l, S[l].e, S[l + 1].e);
      p_vcycle(A, S, l);
    }
  }
  const size_t smem = FIXED_DOUBLES * sizeof(double) + 128 + used * sizeof(double);
  static bool configured = false;
  if (!configured) {
    CUDA_CHECK(cudaFuncSetAttribute(coarse_cycle_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, COARSE_SMEM_MAX));
    configured = true;
  }
  if (hpgmg_ablate(4)) return;
  LAUNCH(coarse_cycle_kernel, 1, COARSE_THREADS, smem, A);
}
