/*
 * smooth.cu -- the operator-applying kernels: GSRB, Chebyshev, weighted Jacobi and L1-Jacobi smoothers, residual,
 * apply_op and the black-box diagonal rebuild.  Entry points mirror the reference one for one:
 *   smooth            operators/gsrb.c:24-132 (GSRB_OOP + GSRB_STRIDE2) | operators/chebyshev.c:8-100 |
 *                     operators/jacobi.c (USE_JACOBI: w = 2/3, lambda = D^-1; USE_L1JACOBI: w = 1, lambda = L1 row inverse)
 *   residual          operators/residual.c:9-51
 *   apply_op          operators/apply_op.c:9-50
 *   rebuild_operator  operators.fv4.c:145-173, rebuild_operator_blackbox operators/rebuild.c:47-208
 *
 * Launch geometry: a grid of (i-tiles, j-tiles, box*k-tiles) thread blocks per level; every box of
 * a level has the same shape so one launch covers all boxes this GPU owns.
 */
#include <math.h>
#include "common.cuh"
#include "stencil.cuh"

enum { OP_APPLY = 0, OP_RESIDUAL = 1, OP_GSRB = 2, OP_CHEBY = 3, OP_REBUILD = 4,
       OP_RESRES = 5,     /* residual fused with the cell restriction that follows it in MGVCycle (k-marching kernel only) */
       OP_JACOBI = 6 };   /* one Jacobi sweep: x + (weight*lambda)*(rhs - A x) */

/* The Helmholtz build (-DUSE_HELMHOLTZ, as in the reference: operators.fv4.c:56-85): A x = a*alpha*x - b*h2inv*(...).  The
 * reference subtracts (b*h2inv)*(...) from a*alpha*x; fv4_apply_op returns (-b*h2inv)*(...), the exact negation, and
 * p - q == p + (-q) in IEEE arithmetic, so the sum below has the reference's bits.  In that build every operator goes
 * through the two global-memory kernels of this file (no TMA / fused-box / single-block paths). */
#ifdef VECTOR_ALPHA
#define HELMHOLTZ_TERM(a, alpha, x) (a) * (alpha) * (x) +
#define VECTOR_ALPHA_OR_0 VECTOR_ALPHA
#else
#define HELMHOLTZ_TERM(a, alpha, x)
#define VECTOR_ALPHA_OR_0 0
#endif

struct StencilArgs {
  DLevel L;
  const int *low;          /* [nboxes][3] */
  int x_id, rhs_id, out_id, xm1_id;
  double a, b, h2inv;
  double c1, c2;           /* Chebyshev */
  double weight;           /* Jacobi: 2/3 (lambda = Dinv) or 1 (lambda = L1 row inverse) */
  const double *lam;       /* Jacobi: lambda of box b, cell (0,0,0), at lam + b * lam_bstride */
  size_t lam_bstride;
  int sweep;               /* GSRB sweep number s (colour) */
  int reverse;             /* march k downwards (TMA kernel only; same result) */
  int diag;                /* TMA GSRB kernel: form Dinv = 1/Aii in registers from the face coefficients wherever the stencil
                              stays clear of the boundary-condition ghost cells (the stored Dinv holds exactly that there) */
  int dom[3];              /* level dimensions in cells */
  double *norm_slot;       /* TMA residual kernel: also leave max |res| here (the norm the caller wants next), or NULL */
  /* OP_RESRES: the residual is not stored; its restriction goes to vector rc_id of the coarse level Lc.  rmap[4 box] =
   * { coarse box, coarse cell of the box's cell (0,0,0): i, j, k } */
  DLevel Lc;
  const int *rmap;
  int rc_id;
};

/* generic one-thread-per-cell kernel (any box size) ------------------------------------------- */
template <int OP>
__global__ void __launch_bounds__(256) stencil_generic_kernel(const StencilArgs A)
{
  PDL_WAIT();
  const DLevel &L = A.L;
  const int n = L.dim;
  const int ktiles = (n + blockDim.z - 1) / blockDim.z;
  const int box = blockIdx.z / ktiles;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  const int j = blockIdx.y * blockDim.y + threadIdx.y;
  const int k = (blockIdx.z % ktiles) * blockDim.z + threadIdx.z;
  if (i >= n || j >= n || k >= n) return;
  const int jS = L.jStride, kS = L.kStride;
  const int ijk = i + j * jS + k * kS;
  const double *__restrict__ x  = L.vec(box, A.x_id) + ijk;
  const double *__restrict__ bi = L.vec(box, VECTOR_BETA_I) + ijk;
  const double *__restrict__ bj = L.vec(box, VECTOR_BETA_J) + ijk;
  const double *__restrict__ bk = L.vec(box, VECTOR_BETA_K) + ijk;

  if (OP == OP_GSRB) {
    double *__restrict__ out = L.vec(box, A.out_id) + ijk;
    const int color000 = (A.low[3 * box] ^ A.low[3 * box + 1] ^ A.low[3 * box + 2] ^ A.sweep) & 1;
    if (((i ^ j ^ k ^ color000) & 1) == 0) {
      const double Ax = HELMHOLTZ_TERM(A.a, L.vec(box, VECTOR_ALPHA_OR_0)[ijk], x[0]) fv4_apply_op(x, bi, bj, bk, jS, kS, A.b, A.h2inv);
      const double dinv = L.vec(box, VECTOR_DINV)[ijk];
      const double rhs = L.vec(box, A.rhs_id)[ijk];
      out[0] = x[0] + dinv * (rhs - Ax);
    } else {
      out[0] = x[0];
    }
    return;
  }
  const double Ax = HELMHOLTZ_TERM(A.a, L.vec(box, VECTOR_ALPHA_OR_0)[ijk], x[0]) fv4_apply_op(x, bi, bj, bk, jS, kS, A.b, A.h2inv);
  if (OP == OP_APPLY) {
    L.vec(box, A.out_id)[ijk] = Ax;
  } else if (OP == OP_RESIDUAL) {
    L.vec(box, A.out_id)[ijk] = L.vec(box, A.rhs_id)[ijk] - Ax;
  } else if (OP == OP_CHEBY) {
    const double xn = x[0];
    const double xm1 = L.vec(box, A.xm1_id)[ijk];
    const double dinv = L.vec(box, VECTOR_DINV)[ijk];
    const double rhs = L.vec(box, A.rhs_id)[ijk];
    L.vec(box, A.out_id)[ijk] = xn + A.c1 * (xn - xm1) + A.c2 * dinv * (rhs - Ax);
  } else if (OP == OP_JACOBI) {                          /* jacobi.c: x_n + weight*lambda*(rhs - Ax_n), left to right */
    const double lam = A.lam[(size_t)box * A.lam_bstride + ijk];
    const double rhs = L.vec(box, A.rhs_id)[ijk];
    L.vec(box, A.out_id)[ijk] = x[0] + (A.weight * lam) * (rhs - Ax);
  } else if (OP == OP_REBUILD) {
    /* rebuild.c:127-133: x is a 0/1 colouring; Aii += x*Ax, sumAbsAij += |(1-x)*Ax| */
    double *Aii = L.vec(box, A.out_id) + ijk;
    double *sumAbs = L.vec(box, A.rhs_id) + ijk;
    Aii[0] += (x[0]) * Ax;
    sumAbs[0] += fabs((1.0 - x[0]) * Ax);
  }
}

#include "stencil_tma.cuh"
#include "stencil_box.cuh"
#include <vector>

/* switches kept for A/B parity checks (tests/test_gpu_parity.py::test_kernel_variants_give_the_same_bits); read once */
static int g_force_generic = -1, g_tma = 1, g_tma_blocks = 0, g_zigzag = 1, g_diag = 1, g_pair_kernel = 1, g_tma_minplanes = 4, g_box_fused_max = 16;

static void stencil_env(void)
{
  if (g_force_generic >= 0) return;
  const char *e = getenv("HPGMG_B200_GENERIC_STENCIL");    /* every level through the one-thread-per-cell kernel */
  g_force_generic = (e && atoi(e)) ? 1 : 0;
  if ((e = getenv("HPGMG_B200_TMA")) != NULL) g_tma = atoi(e);                 /* 0: boxes >= 32^3 through the pair kernel */
  if ((e = getenv("HPGMG_B200_TMA_BLOCKS")) != NULL) g_tma_blocks = atoi(e);   /* uneven split of the plane space */
  if ((e = getenv("HPGMG_B200_ZIGZAG")) != NULL) g_zigzag = atoi(e);           /* 0: every sweep marches k upwards */
  if ((e = getenv("HPGMG_B200_DIAG")) != NULL) g_diag = atoi(e);               /* 0: Dinv always read from memory */
  if ((e = getenv("HPGMG_B200_PAIR_KERNEL")) != NULL) g_pair_kernel = atoi(e); /* 0: small boxes through the generic kernel */
  if ((e = getenv("HPGMG_B200_TMA_MINPLANES")) != NULL && atoi(e) > 0) g_tma_minplanes = atoi(e);   /* shortest k-chunk a block may get */
  if ((e = getenv("HPGMG_B200_BOX_FUSED_MAX")) != NULL) g_box_fused_max = atoi(e);   /* largest box the fill-fused kernels take (0: none, 32: also the TMA kernel's smallest size) */
}

/* ---- TMA descriptors: the level slab [box*vector][k][j][i] as a rank-4 tensor, one (W x rows) tile per copy ---- */
typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *, const cuuint32_t *,
                                  const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn tensor_map_encoder(void)
{
  static EncodeTiledFn fn = NULL;
  if (!fn) {
    void *p = NULL;
    cudaDriverEntryPointQueryResult q;
    CUDA_CHECK(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q));
    if (q != cudaDriverEntryPointSuccess || !p) { fprintf(stderr, "hpgmg_b200: cuTensorMapEncodeTiled is not available from this driver\n"); exit(1); }
    fn = (EncodeTiledFn)p;
  }
  return fn;
}

struct TileMaps {
  const double *base;  int nboxes, nvec, dim, w, xr, br;
  CUtensorMap x, b;
};
static std::vector<TileMaps *> g_tile_maps;

static const TileMaps *tile_maps(const DLevel &L, const int w, const int xr, const int br)
{
  for (size_t t = 0; t < g_tile_maps.size(); t++) {
    const TileMaps *M = g_tile_maps[t];
    if (M->base == L.base && M->nboxes == L.nboxes && M->nvec == L.nvec && M->dim == L.dim && M->w == w && M->xr == xr && M->br == br) return M;
  }
  TileMaps *M = NULL;
  if (posix_memalign((void **)&M, 64, sizeof(TileMaps)) != 0) { fprintf(stderr, "hpgmg_b200: out of memory\n"); exit(1); }
  M->base = L.base;  M->nboxes = L.nboxes;  M->nvec = L.nvec;  M->dim = L.dim;  M->w = w;  M->xr = xr;  M->br = br;
  const cuuint64_t ext = (cuuint64_t)(L.dim + 2 * L.ghosts);
  const cuuint64_t gdim[4] = { (cuuint64_t)L.jStride, ext, ext, (cuuint64_t)L.nboxes * (cuuint64_t)L.nvec };
  const cuuint64_t gstride[3] = { (cuuint64_t)L.jStride * 8, (cuuint64_t)L.kStride * 8, (cuuint64_t)L.volume * 8 };
  const cuuint32_t estride[4] = { 1, 1, 1, 1 };
  for (int which = 0; which < 2; which++) {
    const cuuint32_t box[4] = { (cuuint32_t)w, (cuuint32_t)(which ? br : xr), 1, 1 };
    const CUresult rc = tensor_map_encoder()(which ? &M->b : &M->x, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 4, (void *)L.base, gdim, gstride, box, estride,
                                             CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (rc != CUDA_SUCCESS) { fprintf(stderr, "hpgmg_b200: cuTensorMapEncodeTiled failed (%d) for dim %d jStride %d\n", (int)rc, L.dim, L.jStride); exit(1); }
  }
  g_tile_maps.push_back(M);
  return M;
}

static bool g_norm_fused = false;          /* did the last residual launch also produce the norm? */

/* equal k-chunks per column of the marching kernel: as many as fit the resident slots, at least g_tma_minplanes planes each */
static long long tma_chunks(const long long columns, const int n, const int minb)
{
  const long long slots = (long long)minb * hpgmg_rt_sm_count();
  long long chunks = slots / columns;
  if (chunks > n / g_tma_minplanes) chunks = n / g_tma_minplanes;
  if (chunks < 1) chunks = 1;
  while (n % chunks) chunks--;
  return chunks;
}

template <int OP, int TI, int TJ, int PF, int MINB>
static void launch_tma(const StencilArgs &A)
{
  typedef TmaCfg<TI, TJ, PF> C;
  static bool configured = false;
  if (!configured) {
    CUDA_CHECK(cudaFuncSetAttribute(stencil_tma_kernel<OP, TI, TJ, PF, MINB, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)C::SMEM));
    if (OP == OP_GSRB) CUDA_CHECK(cudaFuncSetAttribute(stencil_tma_kernel<OP, TI, TJ, PF, MINB, (OP == OP_GSRB)>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)C::SMEM));
    configured = true;
  }
  const TileMaps *M = tile_maps(A.L, C::W, C::XR, C::BR);
  const int n = A.L.dim;
  const long long total = (long long)A.L.nboxes * (n / TI) * (n / TJ) * n;
  /* Grid: whole columns (or equal k-chunks of columns) per block, so that all blocks march k in step:
   * tiles that are neighbours in j then fetch their common halo rows at the same time and the second
   * fetch hits L2 (measured on `7 8`: 256 blocks = one column each 189 us; 296 blocks with an even but
   * unaligned split of the plane space 234 us).  Chunks only while the grid still fits the resident
   * slots (MINB blocks per SM) and keeps >= 4 planes per block (measured on `7 8`: 16 planes 5.97 ms, 8 planes 5.78, 4 planes 5.74). */
  const long long columns = total / n;
  const long long chunks = tma_chunks(columns, n, MINB);
  long long blocks = g_tma_blocks > 0 ? g_tma_blocks : columns * chunks;
  if (OP == OP_RESIDUAL && A.norm_slot) g_norm_fused = true;
  if (A.reverse && OP == OP_GSRB) LAUNCH((stencil_tma_kernel<OP, TI, TJ, PF, MINB, (OP == OP_GSRB)>), dim3((unsigned)blocks), dim3(C::NT), C::SMEM, A, M->x, M->b, total);
  else                            LAUNCH((stencil_tma_kernel<OP, TI, TJ, PF, MINB, false>), dim3((unsigned)blocks), dim3(C::NT), C::SMEM, A, M->x, M->b, total);
}

/* Small even boxes (<= 32^3): one thread per i-PAIR of cells, straight from global memory through L1.
 * On a GSRB sweep exactly one cell of the pair is active, so every lane evaluates one stencil (the
 * per-cell kernel above idles half of each warp); results leave as 16-byte stores. */
template <int OP>
__global__ void __launch_bounds__(256) stencil_pair_kernel(const StencilArgs A)
{
  PDL_WAIT();
  const DLevel &L = A.L;
  const int n = L.dim, hn = n >> 1;
  const int ktiles = (n + blockDim.z - 1) / blockDim.z;
  const int box = blockIdx.z / ktiles;
  const int p = blockIdx.x * blockDim.x + threadIdx.x;
  const int j = blockIdx.y * blockDim.y + threadIdx.y;
  const int k = (blockIdx.z % ktiles) * blockDim.z + threadIdx.z;
  if (p >= hn || j >= n || k >= n) return;
  const int jS = L.jStride, kS = L.kStride;
  const int ijk = 2 * p + j * jS + k * kS;
  const double *__restrict__ x  = L.vec(box, A.x_id) + ijk;
  const double *__restrict__ bi = L.vec(box, VECTOR_BETA_I) + ijk;
  const double *__restrict__ bj = L.vec(box, VECTOR_BETA_J) + ijk;
  const double *__restrict__ bk = L.vec(box, VECTOR_BETA_K) + ijk;
  double2 *out = reinterpret_cast<double2 *>(L.vec(box, A.out_id) + ijk);
  if (OP == OP_GSRB) {
    const int color000 = (A.low[3 * box] ^ A.low[3 * box + 1] ^ A.low[3 * box + 2] ^ A.sweep) & 1;
    const int a = (j ^ k ^ color000) & 1;                     /* the active cell of the pair */
    const double2 rhs2 = *reinterpret_cast<const double2 *>(L.vec(box, A.rhs_id) + ijk);
    const double2 dinv2 = *reinterpret_cast<const double2 *>(L.vec(box, VECTOR_DINV) + ijk);
    const double Ax = HELMHOLTZ_TERM(A.a, L.vec(box, VECTOR_ALPHA_OR_0)[ijk + a], x[a]) fv4_apply_op(x + a, bi + a, bj + a, bk + a, jS, kS, A.b, A.h2inv);
    const double xnew = x[a] + (a ? dinv2.y : dinv2.x) * ((a ? rhs2.y : rhs2.x) - Ax);
    const double xo = x[1 - a];
    *out = a ? make_double2(xo, xnew) : make_double2(xnew, xo);
    return;
  }
  const double Ax0 = HELMHOLTZ_TERM(A.a, L.vec(box, VECTOR_ALPHA_OR_0)[ijk], x[0]) fv4_apply_op(x, bi, bj, bk, jS, kS, A.b, A.h2inv);
  const double Ax1 = HELMHOLTZ_TERM(A.a, L.vec(box, VECTOR_ALPHA_OR_0)[ijk + 1], x[1]) fv4_apply_op(x + 1, bi + 1, bj + 1, bk + 1, jS, kS, A.b, A.h2inv);
  if (OP == OP_APPLY) { *out = make_double2(Ax0, Ax1); return; }
  const double2 rhs2 = *reinterpret_cast<const double2 *>(L.vec(box, A.rhs_id) + ijk);
  if (OP == OP_RESIDUAL) { *out = make_double2(rhs2.x - Ax0, rhs2.y - Ax1); return; }
  if (OP == OP_JACOBI) {
    const double2 lam2 = *reinterpret_cast<const double2 *>(A.lam + (size_t)box * A.lam_bstride + ijk);
    *out = make_double2(x[0] + (A.weight * lam2.x) * (rhs2.x - Ax0), x[1] + (A.weight * lam2.y) * (rhs2.y - Ax1));
    return;
  }
  const double2 dinv2 = *reinterpret_cast<const double2 *>(L.vec(box, VECTOR_DINV) + ijk);   /* OP_CHEBY */
  const double2 xm = *reinterpret_cast<const double2 *>(L.vec(box, A.xm1_id) + ijk);
  *out = make_double2(x[0] + A.c1 * (x[0] - xm.x) + A.c2 * dinv2.x * (rhs2.x - Ax0),
                      x[1] + A.c1 * (x[1] - xm.y) + A.c2 * dinv2.y * (rhs2.y - Ax1));
}

template <int OP>
static void launch_stencil(level_type *level, StencilArgs &A)
{
  const DLevel &L = dl_of(level);
  if (L.nboxes == 0) return;
  A.L = L;
  A.low = HPGMG_DEV(level)->low;
  A.h2inv = 1.0 / (level->h * level->h);
  A.dom[0] = level->dim.i;  A.dom[1] = level->dim.j;  A.dom[2] = level->dim.k;
  /* the identity behind `diag` needs the 4^3-colour black-box diagonal (rebuild_operator, operators.fv4.c:145-173:
   * no two cells of a colour within one stencil) and Dirichlet ghost cells that only cells within 2 of the
   * boundary can see */
  A.diag = (OP == OP_GSRB && g_diag && HPGMG_DEV(level)->dinv_is_unit_diagonal && level->boundary_condition.type == BC_DIRICHLET && level->dim.i >= 8 && level->dim.j >= 8 && level->dim.k >= 8) ? 1 : 0;
  const int n = L.dim;
  stencil_env();
  if (OP != OP_REBUILD && hpgmg_ablate(n < 64 ? 8 : (OP == OP_RESIDUAL ? 32 : 64))) return;
#ifdef VECTOR_ALPHA
  A.diag = 0;                                                                     /* the diagonal carries a*alpha */
#endif
  if (OP != OP_REBUILD && !g_force_generic) {
#ifndef VECTOR_ALPHA
    if (n % 32 == 0 && g_tma) { launch_tma<OP, 32, 8, 1, 4>(A); return; }       /* boxes of 32^3 .. 256^3 */
#endif
    if ((n & 1) == 0 && n >= 4 && g_pair_kernel) {
      const int hn = n / 2;
      dim3 block(hn >= 16 ? 16 : hn, n >= 8 ? 8 : n, hn >= 16 ? 2 : (n >= 8 ? 256 / (hn * 8) : 256 / (hn * n)));
      if ((int)block.z > n) block.z = n;
      const int ktiles = (n + block.z - 1) / block.z;
      dim3 grid((hn + block.x - 1) / block.x, (n + block.y - 1) / block.y, ktiles * L.nboxes);
      LAUNCH(stencil_pair_kernel<OP>, grid, block, 0, A);
      return;
    }
  }
  dim3 block(n >= 32 ? 32 : (n >= 16 ? 16 : 8), n >= 32 ? 4 : 4, n >= 32 ? 2 : 4);
  const int ktiles = (n + block.z - 1) / block.z;
  dim3 grid((n + block.x - 1) / block.x, (n + block.y - 1) / block.y, ktiles * L.nboxes);
  LAUNCH(stencil_generic_kernel<OP>, grid, block, 0, A);
}

/* ------------------------------------------------------------------------------------------ */
void hpgmg_fill_ghosts(level_type *level, int id, int shape, int bc_version);   /* ghost.cu */
static void fill_ghosts(level_type *level, int id)
{
  hpgmg_fill_ghosts(level, id, STENCIL_SHAPE_NO_CORNERS, 4);    /* exchange_boundary + apply_BCs, fused */
}

/* ---- ghost fill + operator in one launch (stencil_box.cuh) where the level allows it ---------------- */
template <int OP, int N, int TI, int TJ, int TK>
static void launch_box(level_type *level, const StencilArgs &S, const int write_ghosts)
{
  hpgmg_device_level *D = HPGMG_DEV(level);
  const TileTable &T = D->tile_fill;
  BoxArgs A;
  memset(&A, 0, sizeof(A));
  A.L = D->L;  A.low = D->low;  A.ranges = T.ranges;  A.copies = T.copies;  A.bc = T.bc;
  A.x_id = S.x_id;  A.rhs_id = S.rhs_id;  A.out_id = S.out_id;  A.sweep = S.sweep;  A.write_ghosts = write_ghosts;
  A.b = S.b;  A.h2inv = 1.0 / (level->h * level->h);  A.c1 = S.c1;  A.c2 = S.c2;
  A.weight = S.weight;  A.lam = S.lam;  A.lam_bstride = S.lam_bstride;
  typedef BoxCfg<N, TI, TJ, TK> C;
  LAUNCH((stencil_box_kernel<OP, N, TI, TJ, TK>), D->L.nboxes * C::TILES, C::NT, 0, A);
}

/* 1 if the operator was enqueued as a fill-fused box kernel (then no separate ghost fill is needed) */
template <int OP>
static int try_launch_box(level_type *level, const StencilArgs &S, const int write_ghosts)
{
  stencil_env();
  hpgmg_device_level *D = HPGMG_DEV(level);
  const TileTable &T = D->tile_fill;
  const int n = level->box_dim;
#ifdef VECTOR_ALPHA
  return 0;
#endif
  if (g_force_generic || n > g_box_fused_max || T.ntiles == 0 || level->num_my_boxes == 0) return 0;
  if (D->fill_nvec != level->numVectors || level->box_ghosts != 2 || level->box_jStride != ((n + 4 + 3) / 4) * 4) return 0;
  if (hpgmg_ablate(n < 64 ? 8 : 64)) return 1;
  switch (n) {
    case 4:  launch_box<OP, 4, 4, 4, 4>(level, S, write_ghosts); return 1;
    case 8:  launch_box<OP, 8, 8, 8, 4>(level, S, write_ghosts); return 1;
    case 16: launch_box<OP, 16, 16, 8, 4>(level, S, write_ghosts); return 1;
    case 32: launch_box<OP, 32, 16, 8, 4>(level, S, write_ghosts); return 1;
    default: return 0;
  }
}

/* exchange_boundary + apply_BCs on x, then the operator: one fused launch on small boxes, fill kernel + operator kernel otherwise */
template <int OP>
static void fill_and_stencil(level_type *level, StencilArgs &A, const int write_ghosts)
{
  if (try_launch_box<OP>(level, A, write_ghosts)) return;
  fill_ghosts(level, A.x_id);
  launch_stencil<OP>(level, A);
}

extern "C" int stencil_get_radius(void) { return 2; }
extern "C" int stencil_get_shape(void) { return STENCIL_SHAPE_NO_CORNERS; }

extern "C" void apply_op(level_type *level, int Ax_id, int x_id, double a, double b)
{
  ProfileScope prof_(&level->timers.apply_op);
  hpgmg_note_vector_written(level, Ax_id);
  StencilArgs A = {};
  A.x_id = x_id;  A.out_id = Ax_id;  A.a = a;  A.b = b;
  fill_and_stencil<OP_APPLY>(level, A, 1);
}

extern "C" void residual(level_type *level, int res_id, int x_id, int rhs_id, double a, double b)
{
  ProfileScope prof_(&level->timers.residual);
  hpgmg_note_vector_written(level, res_id);
  StencilArgs A = {};
  A.x_id = x_id;  A.rhs_id = rhs_id;  A.out_id = res_id;  A.a = a;  A.b = b;
  fill_and_stencil<OP_RESIDUAL>(level, A, 1);
}

/* residual() followed by restriction(level_c, rc_id <- level, res_id, RESTRICT_CELL), as MGVCycle runs them (mg.c:1150-1151).
 * Where the level runs the k-marching kernel and every box restricts into a box on this GPU, the residual kernel sums the
 * 2x2x2 children itself (restriction.c:54-57, same order) and writes the coarse cells: the residual is neither written nor
 * re-read (16 of its 48 B/cell) and the restriction launch disappears.  res_id then keeps its old contents -- MGVCycle
 * overwrites it in the post-smooth. */
static int *restriction_map(level_type *level, level_type *level_c)
{
  hpgmg_device_level *D = HPGMG_DEV(level);
  if (D->restrict_map_state != 0) return D->restrict_map_state > 0 ? D->restrict_map : NULL;
  if (g_capturing) return NULL;                          /* built by MGBuild (hpgmg_restriction_map_prepare); never inside a recording */
  D->restrict_map_state = -1;
  const communicator_type *Cf = &level->restriction[RESTRICT_CELL], *Cc = &level_c->restriction[RESTRICT_CELL];
  const int nb = level->num_my_boxes, half = level->box_dim / 2;
  if (nb == 0 || Cf->num_sends || Cf->num_recvs || Cc->num_sends || Cc->num_recvs || (level->box_dim & 3)) return NULL;
  std::vector<int> map((size_t)4 * nb, -1);
  std::vector<long> covered((size_t)nb, 0);
  for (int e = 0; e < Cf->num_blocks[1]; e++) {
    const blockCopy_type &B = Cf->blocks[1][e];
    if (B.read.box < 0 || B.read.box >= nb || B.write.box < 0 || (B.read.i & 1) || (B.read.j & 1) || (B.read.k & 1)) return NULL;
    const int m[4] = { B.write.box, B.write.i - B.read.i / 2, B.write.j - B.read.j / 2, B.write.k - B.read.k / 2 };
    int *M = &map[(size_t)4 * B.read.box];
    if (M[0] < 0) { M[0] = m[0]; M[1] = m[1]; M[2] = m[2]; M[3] = m[3]; }
    else if (M[0] != m[0] || M[1] != m[1] || M[2] != m[2] || M[3] != m[3]) return NULL;
    covered[B.read.box] += (long)B.dim.i * B.dim.j * B.dim.k;
  }
  for (int b = 0; b < nb; b++) if (covered[b] != (long)half * half * half) return NULL;
  CUDA_CHECK(cudaMalloc(&D->restrict_map, map.size() * sizeof(int)));
  CUDA_CHECK(cudaMemcpyAsync(D->restrict_map, map.data(), map.size() * sizeof(int), cudaMemcpyHostToDevice, g_stream));
  CUDA_CHECK(cudaStreamSynchronize(g_stream));
  D->restrict_map_state = 1;
  return D->restrict_map;
}
extern "C" void hpgmg_restriction_map_prepare(level_type *level, level_type *level_c)
{
  if (hpgmg_rt_layout_only() || !HPGMG_DEV(level) || !HPGMG_DEV(level_c)) return;
  restriction_map(level, level_c);
}
extern "C" void hpgmg_residual_then_restriction(level_type *level_c, int rc_id, level_type *level, int res_id, int x_id, int rhs_id, double a, double b)
{
  static int fuse = -1;
  if (fuse < 0) { const char *e = getenv("HPGMG_B200_FUSE_RESTRICT"); fuse = e ? atoi(e) : 1; }
  stencil_env();
  const int n = level->box_dim;
  const int *rmap = NULL;
#ifndef VECTOR_ALPHA
  if (fuse && !hpgmg_rt_profile() && !g_force_generic && g_tma && n % 32 == 0 && level->num_my_boxes > 0 && level_c->num_my_boxes > 0 && !hpgmg_ablate(32))
    rmap = restriction_map(level, level_c);
  /* the fused kernel pairs planes 2m, 2m+1 inside a block: k-chunks must be even (and not split by HPGMG_B200_TMA_BLOCKS) */
  if (rmap && (g_tma_blocks > 0 || ((n / tma_chunks((long long)level->num_my_boxes * (n / 32) * (n / 8), n, 4)) & 1))) rmap = NULL;
#endif
  if (!rmap) {
    residual(level, res_id, x_id, rhs_id, a, b);
    restriction(level_c, rc_id, level, res_id, RESTRICT_CELL);
    return;
  }
  hpgmg_note_vector_written(level_c, rc_id);
  fill_ghosts(level, x_id);
  StencilArgs A = {};
  A.x_id = x_id;  A.rhs_id = rhs_id;  A.out_id = res_id;  A.a = a;  A.b = b;
  A.L = dl_of(level);  A.low = HPGMG_DEV(level)->low;  A.h2inv = 1.0 / (level->h * level->h);
  A.dom[0] = level->dim.i;  A.dom[1] = level->dim.j;  A.dom[2] = level->dim.k;
  A.Lc = dl_of(level_c);  A.rmap = rmap;  A.rc_id = rc_id;
  launch_tma<OP_RESRES, 32, 8, 1, 4>(A);
}

/* residual() followed by norm() of the result (mg.c:1316-1322, 1259-1262), the max taken inside the residual kernel
 * where that kernel is the TMA one: saves re-reading the residual (8 B/cell and a launch).  max is order-free. */
extern "C" void hpgmg_residual_norm_async(level_type *level, int res_id, int x_id, int rhs_id, double a, double b, int slot)
{
  static int fuse = -1;
  if (fuse < 0) { const char *e = getenv("HPGMG_B200_FUSE_NORM"); fuse = e ? atoi(e) : 1; }
  if (!fuse || hpgmg_rt_profile()) { residual(level, res_id, x_id, rhs_id, a, b); hpgmg_norm_async(level, res_id, slot); return; }
  double *s = hpgmg_rt_scalar_slots() + slot;
  CUDA_CHECK(cudaMemsetAsync(s, 0, sizeof(double), g_stream));
  StencilArgs A = {};
  A.x_id = x_id;  A.rhs_id = rhs_id;  A.out_id = res_id;  A.a = a;  A.b = b;  A.norm_slot = s;
  g_norm_fused = false;
  fill_and_stencil<OP_RESIDUAL>(level, A, 1);
  if (g_norm_fused) hpgmg_comm_allreduce_slot_max(level, slot);     /* MPI_Allreduce(MAX), misc.c:324; no-op on one rank */
  else hpgmg_norm_async(level, res_id, slot);
}

static void smooth_gsrb(level_type *level, int x_id, int rhs_id, double a, double b)
{
  for (int s = 0; s < 6; s++) {                      /* NUM_SMOOTHS=3 -> RBRBRB (operators.fv4.c:177-180) */
    const int src = (s & 1) == 0 ? x_id : VECTOR_TEMP;
    const int dst = (s & 1) == 0 ? VECTOR_TEMP : x_id;
    StencilArgs A = {};
    A.x_id = src;  A.rhs_id = rhs_id;  A.out_id = dst;  A.a = a;  A.b = b;  A.sweep = s;
    A.reverse = g_zigzag ? (s & 1) : 0;
    fill_and_stencil<OP_GSRB>(level, A, 0);
  }
}

/* one GSRB sweep kernel alone (no ghost fill) */
extern "C" void hpgmg_b200_gsrb_sweep(level_type *level, int src_id, int dst_id, int rhs_id, double a, double b, int s)
{
  StencilArgs A = {};
  A.x_id = src_id;  A.rhs_id = rhs_id;  A.out_id = dst_id;  A.a = a;  A.b = b;  A.sweep = s;
  launch_stencil<OP_GSRB>(level, A);
}

/* Chebyshev coefficients exactly as chebyshev.c:22-40 (degree 6, operators.fv4.c:184) */
static void chebyshev_coefficients(const level_type *level, double c1[6], double c2[6])
{
  double beta = 1.000 * level->dominant_eigenvalue_of_DinvA;
  double alpha = 0.125000 * beta;
  double theta = 0.5 * (beta + alpha);
  double delta = 0.5 * (beta - alpha);
  double sigma = theta / delta;
  double rho_n = 1 / sigma;
  c1[0] = 0.0;
  c2[0] = 1 / theta;
  for (int s = 1; s < 6; s++) {
    double rho_nm1 = rho_n;
    rho_n = 1.0 / (2.0 * sigma - rho_nm1);
    c1[s] = rho_n * rho_nm1;
    c2[s] = rho_n * 2.0 / delta;
  }
}

static void chebyshev_sweep(level_type *level, int src, int dst, int rhs_id, double a, double b, const double c1, const double c2, const int with_fill)
{
  StencilArgs A = {};
  A.x_id = src;  A.xm1_id = dst;  A.rhs_id = rhs_id;  A.out_id = dst;  A.a = a;  A.b = b;     /* x_{n-1} aliases x_{n+1} (chebyshev.c:75-80) */
  A.c1 = c1;  A.c2 = c2;
  if (with_fill) fill_and_stencil<OP_CHEBY>(level, A, 0);
  else launch_stencil<OP_CHEBY>(level, A);
}

static void smooth_chebyshev(level_type *level, int x_id, int rhs_id, double a, double b)
{
  if (level->dominant_eigenvalue_of_DinvA <= 0.0 && level->my_rank == 0) fprintf(stderr, "dominant_eigenvalue_of_DinvA <= 0.0 !\n");
  double c1[6], c2[6];
  chebyshev_coefficients(level, c1, c2);
  for (int s = 0; s < 6; s++) {
    const int src = (s & 1) == 0 ? x_id : VECTOR_TEMP;
    const int dst = (s & 1) == 0 ? VECTOR_TEMP : x_id;
    chebyshev_sweep(level, src, dst, rhs_id, a, b, c1[s], c2[s], 1);
  }
}

/* The L1 row inverse of a level in the default build (rebuild_operator_blackbox stores it only while L1-Jacobi is selected).
 * The reference fixes its smoother at compile time, so it always has the vector; here a level built for another smoother
 * cannot be smoothed with L1-Jacobi: recomputing the array here would overwrite VECTOR_TEMP and VECTOR_E, which hold live
 * data in the middle of a cycle. */
extern "C" double *hpgmg_l1inv_array(level_type *level)
{
  double *p = HPGMG_DEV(level)->l1inv;
  if (!p && level->num_my_boxes > 0) {
    fprintf(stderr, "hpgmg_b200: the level of h=%e has no L1 row inverse: L1-Jacobi was not the selected smoother when its operator was "
                    "built. Select HPGMG_SMOOTHER_L1JACOBI (hpgmg_b200_set_smoother) before rebuild_operator / MGBuild.\n", level->h);
    fflush(stderr);
    exit(1);
  }
  return p;
}

extern "C" void hpgmg_download_l1inv(level_type *level, int box, double *host)
{
#ifdef VECTOR_L1INV
  hpgmg_download_box_vector(level, box, VECTOR_L1INV, host);
#else
  const double *p = hpgmg_l1inv_array(level);
  hpgmg_rt_copy_d2h(host, p + (size_t)box * level->box_volume, (size_t)level->box_volume * sizeof(double));
  hpgmg_rt_sync();
#endif
}

/* weight and lambda of the selected Jacobi variant (jacobi.c): USE_JACOBI 2/3 and Dinv, USE_L1JACOBI 1 and the L1 row inverse */
static void jacobi_operands(level_type *level, StencilArgs &A)
{
  const DLevel &L = dl_of(level);
  if (hpgmg_rt_smoother() == HPGMG_SMOOTHER_L1JACOBI) {
    A.weight = 1.0;
#ifdef VECTOR_L1INV
    A.lam = L.vec(0, VECTOR_L1INV);  A.lam_bstride = (size_t)L.nvec * L.volume;
#else
    A.lam = hpgmg_l1inv_array(level) + L.origin;  A.lam_bstride = (size_t)L.volume;
#endif
  } else {
    A.weight = 2.0 / 3.0;
    A.lam = L.vec(0, VECTOR_DINV);  A.lam_bstride = (size_t)L.nvec * L.volume;
  }
}

static void smooth_jacobi(level_type *level, int x_id, int rhs_id, double a, double b)
{
  StencilArgs J = {};
  jacobi_operands(level, J);
  for (int s = 0; s < 6; s++) {                      /* NUM_SMOOTHS=6 (operators.fv4.c:176-195); x -> TEMP -> x like GSRB */
    StencilArgs A = J;
    A.x_id = (s & 1) == 0 ? x_id : VECTOR_TEMP;
    A.out_id = (s & 1) == 0 ? VECTOR_TEMP : x_id;
    A.rhs_id = rhs_id;  A.a = a;  A.b = b;
    fill_and_stencil<OP_JACOBI>(level, A, 0);
  }
}

static int is_jacobi(const int smoother) { return smoother == HPGMG_SMOOTHER_JACOBI || smoother == HPGMG_SMOOTHER_L1JACOBI; }

/* one sweep kernel of the current smoother alone (no ghost fill): what bench.py times for the roofline line */
extern "C" void hpgmg_b200_smoother_sweep(level_type *level, int src_id, int dst_id, int rhs_id, double a, double b, int s)
{
  if (hpgmg_rt_smoother() == HPGMG_SMOOTHER_CHEBY) {
    double c1[6], c2[6];
    chebyshev_coefficients(level, c1, c2);
    chebyshev_sweep(level, src_id, dst_id, rhs_id, a, b, c1[s % 6], c2[s % 6], 0);
  } else if (is_jacobi(hpgmg_rt_smoother())) {
    StencilArgs A = {};
    jacobi_operands(level, A);
    A.x_id = src_id;  A.rhs_id = rhs_id;  A.out_id = dst_id;  A.a = a;  A.b = b;
    launch_stencil<OP_JACOBI>(level, A);
  } else hpgmg_b200_gsrb_sweep(level, src_id, dst_id, rhs_id, a, b, s);
}

extern "C" void smooth(level_type *level, int x_id, int rhs_id, double a, double b)
{
  ProfileScope prof_(&level->timers.smooth);
  hpgmg_note_vector_written(level, x_id);
  if (hpgmg_rt_smoother() == HPGMG_SMOOTHER_CHEBY) smooth_chebyshev(level, x_id, rhs_id, a, b);
  else if (is_jacobi(hpgmg_rt_smoother())) smooth_jacobi(level, x_id, rhs_id, a, b);
  else smooth_gsrb(level, x_id, rhs_id, a, b);
}

/* ------------------------------------------------------------------------------------------ */
/* D^-1 and the Gershgorin bound on lambda_max(D^-1 A) from the operator alone (rebuild.c:47-208) */
__global__ void rebuild_finish_kernel(const DLevel L, const int *low, int Aii_id, int sum_id, double a, double b, double h2inv, double *eig_slot, double *l1inv)
{
  PDL_WAIT();
  const int n = L.dim;
  const int cells = n * n * n;
  double local = 0.0;                                  /* all Di are > 0 for this operator */
  for (int box = blockIdx.y; box < L.nboxes; box += gridDim.y) {
    for (int c = blockIdx.x * blockDim.x + threadIdx.x; c < cells; c += gridDim.x * blockDim.x) {
      const int i = c % n, j = (c / n) % n, k = c / (n * n);
      const int ijk = i + j * L.jStride + k * L.kStride;
      double *Aii = L.vec(box, Aii_id) + ijk;
      double *sumAbs = L.vec(box, sum_id) + ijk;
      if (Aii[0] == 0.0) {
        printf("Aii[%d,%d,%d]==0.0 !!!\n", i + low[3 * box], j + low[3 * box + 1], k + low[3 * box + 2]);
        Aii[0] = a + b * h2inv;
      }
      const double Di = (Aii[0] + sumAbs[0]) / Aii[0];
      if (Di > local) local = Di;
      if (Aii[0] >= 1.5 * sumAbs[0]) sumAbs[0] = 1.0 / (Aii[0]);
      else                           sumAbs[0] = 1.0 / (Aii[0] + 0.5 * sumAbs[0]);
      if (l1inv) l1inv[(size_t)box * L.volume + L.origin + ijk] = sumAbs[0];    /* the L1-Jacobi lambda, kept (default build) */
      Aii[0] = 1.0 / Aii[0];
    }
  }
  atomic_max_nonneg(eig_slot, local);
}

extern "C" void rebuild_operator_blackbox(level_type *level, double a, double b, int colors_in_each_dim)
{
  if (level->dim.i < colors_in_each_dim) colors_in_each_dim = level->dim.i;
  if (level->dim.j < colors_in_each_dim) colors_in_each_dim = level->dim.j;
  if (level->dim.k < colors_in_each_dim) colors_in_each_dim = level->dim.k;
  const int chatty = level->my_rank == 0 && hpgmg_rt_verbose();
  if (chatty) {
    fprintf(stdout, "  calculating D^{-1} exactly for level h=%e using %3d colors...  ", level->h, colors_in_each_dim * colors_in_each_dim * colors_in_each_dim);
    fflush(stdout);
  }
#ifdef VECTOR_L1INV
  const int x_id = VECTOR_TEMP, Aii_id = VECTOR_DINV, sum_id = VECTOR_L1INV;      /* rebuild.c:77-81 */
#else
  const int x_id = VECTOR_TEMP, Aii_id = VECTOR_DINV, sum_id = VECTOR_E;
#endif
  zero_vector(level, Aii_id);
  zero_vector(level, sum_id);
  for (int kc = 0; kc < colors_in_each_dim; kc++)
  for (int jc = 0; jc < colors_in_each_dim; jc++)
  for (int ic = 0; ic < colors_in_each_dim; ic++) {
    color_vector(level, x_id, colors_in_each_dim, ic, jc, kc);
    fill_ghosts(level, x_id);
    StencilArgs A = {};
    A.x_id = x_id;  A.rhs_id = sum_id;  A.out_id = Aii_id;  A.a = a;  A.b = b;
    launch_stencil<OP_REBUILD>(level, A);
  }
  double *slot = hpgmg_rt_scalar_slots() + HPGMG_SLOT_SCRATCH;
  CUDA_CHECK(cudaMemsetAsync(slot, 0, sizeof(double), g_stream));
  const DLevel &L = dl_of(level);
  double *l1inv = NULL;
#ifndef VECTOR_L1INV
  /* the default vector map has no room for the L1 row inverse: an array of the level, made when L1-Jacobi is selected
   * and refreshed by every later rebuild */
  hpgmg_device_level *D = HPGMG_DEV(level);
  if (!D->l1inv && L.nboxes > 0 && hpgmg_rt_smoother() == HPGMG_SMOOTHER_L1JACOBI)
    D->l1inv = (double *)hpgmg_rt_alloc_zero((size_t)L.nboxes * L.volume * sizeof(double));
  l1inv = D->l1inv;
#endif
  if (L.nboxes > 0) {
    const int cells = L.dim * L.dim * L.dim;
    dim3 grid((cells + 255) / 256 > 1024 ? 1024 : (cells + 255) / 256, L.nboxes);
    LAUNCH(rebuild_finish_kernel, grid, 256, 0, L, HPGMG_DEV(level)->low, Aii_id, sum_id, a, b, 1.0 / (level->h * level->h), slot, l1inv);
  }
  double eig = 0.0;
  hpgmg_rt_read_scalars(&eig, HPGMG_SLOT_SCRATCH, 1);
  if (L.nboxes == 0) eig = -1e9;
  eig = hpgmg_comm_allreduce_max_world(level, eig);    /* MPI_Allreduce(MAX) on MPI_COMM_WORLD (rebuild.c:195) */
  if (chatty) fprintf(stdout, "done\n");
  if (chatty && hpgmg_rt_smoother() == HPGMG_SMOOTHER_CHEBY) { fprintf(stdout, "  estimating  lambda_max... <%1.15e\n", eig); fflush(stdout); }
  level->dominant_eigenvalue_of_DinvA = eig;
  HPGMG_DEV(level)->dinv_is_unit_diagonal = (colors_in_each_dim >= 4) ? 1 : 0;
  hpgmg_graph_drop_all(NULL);                          /* recorded solves carry the old eigenvalue / diagonal shortcut by value */
}

extern "C" void rebuild_operator(level_type *level, level_type *fromLevel, double a, double b)
{
  if (fromLevel != NULL) {
#ifdef VECTOR_ALPHA
    restriction(level, VECTOR_ALPHA, fromLevel, VECTOR_ALPHA, RESTRICT_CELL);
#endif
    restriction(level, VECTOR_BETA_I, fromLevel, VECTOR_BETA_I, RESTRICT_FACE_I);
    restriction(level, VECTOR_BETA_J, fromLevel, VECTOR_BETA_J, RESTRICT_FACE_J);
    restriction(level, VECTOR_BETA_K, fromLevel, VECTOR_BETA_K, RESTRICT_FACE_K);
  }
  extrapolate_betas(level);
#ifdef VECTOR_ALPHA
  exchange_boundary(level, VECTOR_ALPHA, STENCIL_SHAPE_BOX);
#endif
  exchange_boundary(level, VECTOR_BETA_I, STENCIL_SHAPE_BOX);
  exchange_boundary(level, VECTOR_BETA_J, STENCIL_SHAPE_BOX);
  exchange_boundary(level, VECTOR_BETA_K, STENCIL_SHAPE_BOX);
  rebuild_operator_blackbox(level, a, b, 4);
  exchange_boundary(level, VECTOR_DINV, STENCIL_SHAPE_BOX);
}
