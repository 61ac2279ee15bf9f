/*
 * stencil_fv2.cuh -- the k-marching kernel of the 7-point fv2 operator (built with -DHPGMG_FV2 only; included by smooth.cu).
 *
 * Boxes of 32^3 and up.  A thread block is a 32 x 8 tile of (i, j) columns; every thread owns one column and marches k over
 * its block's chunk of planes.  The three x values of the column the star needs (planes k-1, k, k+1) and the face
 * coefficient beta_k of plane k+1 (the next cell's beta_k(k)) stay in registers, so each plane costs one new x, one rhs-side
 * value and the four in-plane x neighbours and the i+1 / j+1 betas, which neighbouring lanes of the same warp or tile have just
 * loaded: those come from L1, and HBM sees each array once -- 56 B per cell for GSRB and Jacobi, 64 for Chebyshev, 48 for
 * the residual, 40 for apply_op.  The Helmholtz build (-DUSE_HELMHOLTZ) also reads alpha at the cells that evaluate the stencil,
 * 8 B more per cell for every operator.  Staging is by plain loads: the halo is one cell deep, which L1 serves without shared
 * memory and without the barriers a TMA pipeline would need (DESIGN.md section 4).
 *
 * The arithmetic is op_apply_at and the smoother updates of stencil.cuh over loaders that read the register window, so the
 * results are bit-identical to the generic and pair kernels.
 */
#ifndef HPGMG_B200_STENCIL_FV2_CUH
#define HPGMG_B200_STENCIL_FV2_CUH

#define FV2_TI 32
#define FV2_TJ 8

/* x at (di,dj,dk) from the column's cell: dk = +-1 and the cell itself from registers, the in-plane neighbours from memory */
struct Fv2WindowX {
  const double *__restrict__ p;     /* cell (i, j, k) */
  int jS;
  double xd, xc, xu;
  __device__ __forceinline__ double operator()(const int di, const int dj, const int dk) const
  {
    if (dk < 0) return xd;
    if (dk > 0) return xu;
    if (di == 0 && dj == 0) return xc;
    return p[di + dj * jS];
  }
};
/* beta_k: planes k and k+1 of the column, both in registers */
struct Fv2WindowBK {
  double b0, b1;
  __device__ __forceinline__ double operator()(const int, const int, const int dk) const { return dk > 0 ? b1 : b0; }
};

template <int OP>
__global__ void __launch_bounds__(FV2_TI * FV2_TJ, 4) stencil_fv2_march_kernel(const StencilArgs A, const int chunks)
{
  PDL_WAIT();
  const DLevel &L = A.L;
  const int n = L.dim, jS = L.jStride, kS = L.kStride;
  const int planes = n / chunks;
  const int box = blockIdx.z / chunks, k0 = (blockIdx.z % chunks) * planes;
  const int i = blockIdx.x * FV2_TI + threadIdx.x, j = blockIdx.y * FV2_TJ + threadIdx.y;
  const int ij = i + j * jS;
  const double *__restrict__ x = L.vec(box, A.x_id) + ij;
  const double *__restrict__ bi = L.vec(box, VECTOR_BETA_I) + ij;
  const double *__restrict__ bj = L.vec(box, VECTOR_BETA_J) + ij;
  const double *__restrict__ bk = L.vec(box, VECTOR_BETA_K) + ij;
  double *__restrict__ out = L.vec(box, A.out_id) + ij;
  const double *__restrict__ rhs = L.vec(box, A.rhs_id) + ij;
  const double *__restrict__ dinv = L.vec(box, VECTOR_DINV) + ij;
  const double *__restrict__ xm1 = L.vec(box, A.xm1_id) + ij;
  const double *__restrict__ lam = A.lam ? A.lam + (size_t)box * A.lam_bstride + ij : nullptr;
#ifdef VECTOR_ALPHA
  const double *__restrict__ alpha = L.vec(box, VECTOR_ALPHA) + ij;
#endif
  const int color = (OP == OP_GSRB) ? ((i ^ j ^ gsrb_box_parity(A.low, box, A.sweep)) & 1) : 0;

  Fv2WindowX X = { x + k0 * kS, jS, x[(k0 - 1) * kS], x[k0 * kS], 0.0 };
  Fv2WindowBK BK = { 0.0, bk[k0 * kS] };
#pragma unroll 1
  for (int k = k0; k < k0 + planes; k++) {
    const int o = k * kS;
    X.p = x + o;
    X.xu = x[o + kS];
    BK.b0 = BK.b1;
    BK.b1 = bk[o + kS];
    const GlobalLoader BI = { bi + o, jS, kS }, BJ = { bj + o, jS, kS };
    if (OP == OP_GSRB && ((k ^ color) & 1) != 0) {
      out[o] = X.xc;                                               /* not this sweep's colour */
    } else {
      const double Ax = HELMHOLTZ_TERM(A.a, alpha[o], X.xc) op_apply_at(X, BI, BJ, BK, A.b, A.h2inv);
      if (OP == OP_APPLY)         out[o] = Ax;
      else if (OP == OP_RESIDUAL) out[o] = rhs[o] - Ax;
      else if (OP == OP_GSRB)     out[o] = gsrb_update(X.xc, dinv[o], rhs[o], Ax);
      else if (OP == OP_CHEBY)    out[o] = chebyshev_update(X.xc, xm1[o], A.c1, A.c2, dinv[o], rhs[o], Ax);
      else if (OP == OP_JACOBI)   out[o] = jacobi_update(X.xc, A.weight, lam[o], rhs[o], Ax);
    }
    X.xd = X.xc;
    X.xc = X.xu;
  }
}

/* one launch over every box of the level: (i tiles, j tiles, box x k-chunks); equal k-chunks, as many as fill the resident
 * slots (tma_chunks, smooth.cu) */
template <int OP>
static void launch_fv2_march(const StencilArgs &A)
{
  const int n = A.L.dim;
  const long long columns = (long long)A.L.nboxes * (n / FV2_TI) * (n / FV2_TJ);
  const int chunks = (int)tma_chunks(columns, n, 4);
  LAUNCH(stencil_fv2_march_kernel<OP>, dim3(n / FV2_TI, n / FV2_TJ, A.L.nboxes * chunks), dim3(FV2_TI, FV2_TJ), 0, A, chunks);
}

#endif
