/*
 * blas1.cu -- element-wise vector operations and reductions over a level.
 * Restates operators/misc.c: zero_vector :6-44 (zeroes ghost zones too), init_vector :48-87,
 * add_vectors :94-124, mul_vectors :131-161, invert_vector :168-197, scale_vector :204-233,
 * dot :239-282, norm :287-329 (MAX norm), mean :336-380, shift_vector :386-415, error :420-425,
 * color_vector :441-471, random_vector :478-504.  Interior cells only unless noted.
 *
 * Reductions: norm is a max, hence order-free: block partials go through an atomicMax on the bit
 * pattern.  dot/mean are sums, whose value depends on the order: they are accumulated exactly as
 * the single-threaded reference does -- k,j,i inside each compute tile (level->my_blocks), then
 * tile by tile -- by one thread per tile followed by one thread over the tile partials.  They are
 * only used on the coarsest grid inside the benchmark, where a level is a single small tile.
 */
#include <math.h>
#include "common.cuh"

enum { B_ZERO = 0, B_INIT, B_SCALE, B_ADD, B_MUL, B_INVERT, B_SHIFT, B_COLOR, B_RANDOM };

struct BlasArgs {
  DLevel L;
  const int *low;
  int c, a, b;
  double sa, sb;
  int colors, ic, jc, kc;
};

template <int OP>
__global__ void __launch_bounds__(256) blas1_kernel(const BlasArgs A)
{
  PDL_WAIT();
  const DLevel &L = A.L;
  const int g = (OP == B_ZERO || OP == B_INIT) ? L.ghosts : 0;      /* these two cover the ghost zones */
  const int n = L.dim + 2 * g;
  const int cells = n * n * n;
  const int box = blockIdx.y;
  if ((OP == B_ZERO || OP == B_SCALE || OP == B_ADD) && (n & 1) == 0) {            /* the hot ones: 16-byte i-pairs */
    const int hn = n / 2, pairs = hn * n * n;
    for (int cidx = blockIdx.x * blockDim.x + threadIdx.x; cidx < pairs; cidx += gridDim.x * blockDim.x) {
      const int i = 2 * (cidx % hn) - g, j = (cidx / hn) % n - g, k = cidx / (hn * n) - g;
      const int ijk = i + j * L.jStride + k * L.kStride;
      double2 *c = reinterpret_cast<double2 *>(L.vec(box, A.c) + ijk);
      if (OP == B_ZERO) *c = make_double2(0.0, 0.0);
      else if (OP == B_SCALE) {
        const double2 a = *reinterpret_cast<const double2 *>(L.vec(box, A.a) + ijk);
        *c = make_double2(A.sa * a.x, A.sa * a.y);
      } else {
        const double2 a = *reinterpret_cast<const double2 *>(L.vec(box, A.a) + ijk), b = *reinterpret_cast<const double2 *>(L.vec(box, A.b) + ijk);
        *c = make_double2(A.sa * a.x + A.sb * b.x, A.sa * a.y + A.sb * b.y);
      }
    }
    return;
  }
  for (int cidx = blockIdx.x * blockDim.x + threadIdx.x; cidx < cells; cidx += gridDim.x * blockDim.x) {
    const int i = cidx % n - g, j = (cidx / n) % n - g, k = cidx / (n * n) - g;
    const int ijk = i + j * L.jStride + k * L.kStride;
    double *c = L.vec(box, A.c) + ijk;
    if (OP == B_ZERO) c[0] = 0.0;
    else if (OP == B_INIT) {
      const int ghostZone = (i < 0) || (j < 0) || (k < 0) || (i >= L.dim) || (j >= L.dim) || (k >= L.dim);
      c[0] = ghostZone ? 0.0 : A.sa;
    }
    else if (OP == B_SCALE)  c[0] = A.sa * L.vec(box, A.a)[ijk];
    else if (OP == B_ADD)    c[0] = A.sa * L.vec(box, A.a)[ijk] + A.sb * L.vec(box, A.b)[ijk];
    else if (OP == B_MUL)    c[0] = A.sa * L.vec(box, A.a)[ijk] * L.vec(box, A.b)[ijk];
    else if (OP == B_INVERT) c[0] = A.sa / L.vec(box, A.a)[ijk];
    else if (OP == B_SHIFT)  c[0] = L.vec(box, A.a)[ijk] + A.sa;
    else if (OP == B_COLOR) {
      const double si = ((i + A.low[3 * box + 0] + A.ic) % A.colors) == 0 ? 1.0 : 0.0;
      const double sj = ((j + A.low[3 * box + 1] + A.jc) % A.colors) == 0 ? 1.0 : 0.0;
      const double sk = ((k + A.low[3 * box + 2] + A.kc) % A.colors) == 0 ? 1.0 : 0.0;
      c[0] = si * sj * sk;
    }
    else if (OP == B_RANDOM) c[0] = -1.000 + 2.0 * (i ^ j ^ k ^ 0x1);
  }
}

template <int OP>
static void launch_blas1(level_type *level, BlasArgs &A)
{
  if (hpgmg_ablate(128)) return;
  hpgmg_note_vector_written(level, A.c);
  const DLevel &L = dl_of(level);
  if (L.nboxes == 0) return;
  A.L = L;
  A.low = HPGMG_DEV(level)->low;
  const int g = (OP == B_ZERO || OP == B_INIT) ? L.ghosts : 0;
  const int n = L.dim + 2 * g;
  const int cells = n * n * n;
  int bx = (cells + 255) / 256;
  if (bx > 2048) bx = 2048;
  LAUNCH(blas1_kernel<OP>, dim3(bx, L.nboxes), 256, 0, A);
}

/* The 16-byte pairs of B_ZERO start at ghost cell -g of a row; create_vectors aligns cell 0, so with an odd number of ghost
 * layers (fv2) they are misaligned: there the whole box is zeroed as init_vector(0.0) does it, one double at a time. */
extern "C" void zero_vector(level_type *level, int id_a)
{
  BlasArgs A = {}; ProfileScope prof_(&level->timers.blas1); A.c = id_a;
  if (level->box_ghosts & 1) launch_blas1<B_INIT>(level, A);
  else                       launch_blas1<B_ZERO>(level, A);
}
extern "C" void init_vector(level_type *level, int id_a, double scalar)
{ BlasArgs A = {}; ProfileScope prof_(&level->timers.blas1); A.c = id_a; A.sa = scalar; launch_blas1<B_INIT>(level, A); }
extern "C" void scale_vector(level_type *level, int id_c, double scale_a, int id_a)
{ BlasArgs A = {}; ProfileScope prof_(&level->timers.blas1); A.c = id_c; A.a = id_a; A.sa = scale_a; launch_blas1<B_SCALE>(level, A); }
extern "C" void add_vectors(level_type *level, int id_c, double scale_a, int id_a, double scale_b, int id_b)
{ BlasArgs A = {}; ProfileScope prof_(&level->timers.blas1); A.c = id_c; A.a = id_a; A.b = id_b; A.sa = scale_a; A.sb = scale_b; launch_blas1<B_ADD>(level, A); }
extern "C" void mul_vectors(level_type *level, int id_c, double scale, int id_a, int id_b)
{ BlasArgs A = {}; ProfileScope prof_(&level->timers.blas1); A.c = id_c; A.a = id_a; A.b = id_b; A.sa = scale; launch_blas1<B_MUL>(level, A); }
extern "C" void invert_vector(level_type *level, int id_c, double scale_a, int id_a)
{ BlasArgs A = {}; ProfileScope prof_(&level->timers.blas1); A.c = id_c; A.a = id_a; A.sa = scale_a; launch_blas1<B_INVERT>(level, A); }
extern "C" void shift_vector(level_type *level, int id_c, int id_a, double shift_a)
{ BlasArgs A = {}; ProfileScope prof_(&level->timers.blas1); A.c = id_c; A.a = id_a; A.sa = shift_a; launch_blas1<B_SHIFT>(level, A); }
extern "C" void color_vector(level_type *level, int id_a, int colors_in_each_dim, int icolor, int jcolor, int kcolor)
{ BlasArgs A = {}; ProfileScope prof_(&level->timers.blas1); A.c = id_a; A.colors = colors_in_each_dim; A.ic = icolor; A.jc = jcolor; A.kc = kcolor; launch_blas1<B_COLOR>(level, A); }
extern "C" void random_vector(level_type *level, int id_a)
{ BlasArgs A = {}; ProfileScope prof_(&level->timers.blas1); A.c = id_a; launch_blas1<B_RANDOM>(level, A); }

/* ---- max norm ---------------------------------------------------------------------------------- */
__global__ void __launch_bounds__(256) norm_kernel(const DLevel L, const int id, double *__restrict__ slot)
{
  PDL_WAIT();
  const int n = L.dim, box = blockIdx.y;
  const double *__restrict__ v = L.vec(box, id);
  double m = 0.0;
  if ((n & 1) == 0) {                                   /* rows start 16-byte aligned: read i-pairs */
    const int hn = n / 2, pairs = hn * n * n;
    for (int c = blockIdx.x * blockDim.x + threadIdx.x; c < pairs; c += gridDim.x * blockDim.x) {
      const int p = c % hn, j = (c / hn) % n, k = c / (hn * n);
      const double2 q = *reinterpret_cast<const double2 *>(v + 2 * p + j * L.jStride + k * L.kStride);
      const double f0 = fabs(q.x), f1 = fabs(q.y);
      if (f0 > m) m = f0;
      if (f1 > m) m = f1;
    }
  } else {
    const int cells = n * n * n;
    for (int c = blockIdx.x * blockDim.x + threadIdx.x; c < cells; c += gridDim.x * blockDim.x) {
      const int i = c % n, j = (c / n) % n, k = c / (n * n);
      const double f = fabs(v[i + j * L.jStride + k * L.kStride]);
      if (f > m) m = f;
    }
  }
  /* warp shuffle max, then one atomic per block */
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const double other = __shfl_down_sync(0xffffffffu, m, o);
    if (other > m) m = other;
  }
  __shared__ double wmax[8];
  if ((threadIdx.x & 31) == 0) wmax[threadIdx.x >> 5] = m;
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < (int)(blockDim.x >> 5); w++) if (wmax[w] > m) m = wmax[w];
    atomic_max_nonneg(slot, m);
  }
}

/* c = 1.0 * a together with max |a| (FMGSolve / MGSolve begin with norm(F); R = F: mg.c:1259-1262): one pass over F */
__global__ void __launch_bounds__(256) copy_norm_kernel(const DLevel L, const int id_c, const int id_a, double *__restrict__ slot)
{
  PDL_WAIT();
  const int n = L.dim, box = blockIdx.y;
  const double *__restrict__ v = L.vec(box, id_a);
  double *__restrict__ c = L.vec(box, id_c);
  double m = 0.0;
  const int hn = n / 2, pairs = hn * n * n;                /* even n only: rows start 16-byte aligned */
  for (int q = blockIdx.x * blockDim.x + threadIdx.x; q < pairs; q += gridDim.x * blockDim.x) {
    const int p = q % hn, j = (q / hn) % n, k = q / (hn * n);
    const int ijk = 2 * p + j * L.jStride + k * L.kStride;
    const double2 a = *reinterpret_cast<const double2 *>(v + ijk);
    *reinterpret_cast<double2 *>(c + ijk) = make_double2(1.0 * a.x, 1.0 * a.y);
    const double f0 = fabs(a.x), f1 = fabs(a.y);
    if (f0 > m) m = f0;
    if (f1 > m) m = f1;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const double other = __shfl_down_sync(0xffffffffu, m, o);
    if (other > m) m = other;
  }
  __shared__ double wmax[8];
  if ((threadIdx.x & 31) == 0) wmax[threadIdx.x >> 5] = m;
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < (int)(blockDim.x >> 5); w++) if (wmax[w] > m) m = wmax[w];
    atomic_max_nonneg(slot, m);
  }
}

/* ---- dense <-> padded: the cells of every box in a contiguous array without ghosts, in one of two layouts ---- */
/* Where the cells of box `box` lie in the dense array, in 16-byte i-pairs: box_start() is the pair of cell (0,0,0) of the box,
 * pair() the offset of pair p of row j of plane k from there (q: the same pair counted inside the box, p fastest). */
struct BoxMajorDense {               /* [box][k][j][i], box after box: the end-to-end solve's staging buffers */
  __device__ __forceinline__ double2 *box_start(double *dense, const DLevel &L, int box) const
  { const int n = L.dim; return reinterpret_cast<double2 *>(dense + (size_t)box * n * n * n); }
  __device__ __forceinline__ int pair(int q, int, int, int) const { return q; }
};
struct GridDense {                   /* [k][j][i] over the level's whole domain: a box's cells start at its low corner */
  const int *low;                    /* device [nboxes][3] (hpgmg_device_level::low); low.i is even since the box size is */
  size_t hjS, hkS;                   /* row and plane strides of the domain, in pairs: dim.i / 2 and dim.i * dim.j / 2 */
  __device__ __forceinline__ double2 *box_start(double *dense, const DLevel &, int box) const
  { const int *lo = low + 3 * box; return reinterpret_cast<double2 *>(dense) + ((size_t)lo[2] * hkS + (size_t)lo[1] * hjS + lo[0] / 2); }
  __device__ __forceinline__ size_t pair(int, int p, int j, int k) const { return (size_t)p + (size_t)j * hjS + (size_t)k * hkS; }
};

/* MODE 0: box vector <- dense.  MODE 1: dense <- box vector.  MODE 2: F <- dense, R <- 1.0*dense, max|dense| (the first step of
 * FMGSolve, mg.c:1259-1269, fused with the unpack of the right-hand side) */
template <int MODE, class Dense>
__global__ void __launch_bounds__(256) dense_kernel(const DLevel L, const int id, const int id2, double *__restrict__ dense, double *__restrict__ slot, const Dense lay)
{
  PDL_WAIT();
  const int n = L.dim, box = blockIdx.y;
  const int hn = n / 2, pairs = hn * n * n;                /* even n only */
  double *__restrict__ v = L.vec(box, id);
  double *__restrict__ v2 = (MODE == 2) ? L.vec(box, id2) : nullptr;
  double2 *__restrict__ d = lay.box_start(dense, L, box);
  double m = 0.0;
  for (int q = blockIdx.x * blockDim.x + threadIdx.x; q < pairs; q += gridDim.x * blockDim.x) {
    const int p = q % hn, j = (q / hn) % n, k = q / (hn * n);
    const int ijk = 2 * p + j * L.jStride + k * L.kStride;
    double2 *__restrict__ dq = d + lay.pair(q, p, j, k);
    if constexpr (MODE == 1) { *dq = *reinterpret_cast<const double2 *>(v + ijk); }
    else {
    const double2 a = *dq;
    *reinterpret_cast<double2 *>(v + ijk) = a;
    if constexpr (MODE == 2) {
      *reinterpret_cast<double2 *>(v2 + ijk) = make_double2(1.0 * a.x, 1.0 * a.y);
      const double f0 = fabs(a.x), f1 = fabs(a.y);
      if (f0 > m) m = f0;
      if (f1 > m) m = f1;
    }
    }
  }
  if constexpr (MODE == 2) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const double other = __shfl_down_sync(0xffffffffu, m, o);
    if (other > m) m = other;
  }
  __shared__ double wmax[8];
  if ((threadIdx.x & 31) == 0) wmax[threadIdx.x >> 5] = m;
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < (int)(blockDim.x >> 5); w++) if (wmax[w] > m) m = wmax[w];
    atomic_max_nonneg(slot, m);
  }
  }
}
template <int MODE, class Dense>
static void launch_dense(level_type *level, int id, int id2, double *dense, double *slot, const Dense &lay)
{
  const DLevel &L = dl_of(level);
  if (L.nboxes == 0) return;
  if (L.dim & 1) { fprintf(stderr, "hpgmg_b200: dense pack/unpack needs an even box size\n"); exit(1); }
  const int pairs = (L.dim / 2) * L.dim * L.dim;
  int bx = (pairs + 1023) / 1024;
  if (bx > 592) bx = 592;
  LAUNCH((dense_kernel<MODE, Dense>), dim3(bx, L.nboxes), 256, 0, L, id, id2, dense, slot, lay);
}
static GridDense grid_of(const level_type *level)
{
  GridDense g;
  g.low = HPGMG_DEV(level)->low;
  g.hjS = (size_t)level->dim.i / 2;
  g.hkS = (size_t)level->dim.i * level->dim.j / 2;
  return g;
}
template <class Dense>
static void unpack_copy_norm(level_type *level, int id_f, int id_r, const double *dense, int slot, const Dense &lay)
{
  hpgmg_note_vector_written(level, id_f);  hpgmg_note_vector_written(level, id_r);
  double *s = hpgmg_rt_scalar_slots() + slot;
  CUDA_CHECK(cudaMemsetAsync(s, 0, sizeof(double), g_stream));
  g_launches++;
  launch_dense<2>(level, id_f, id_r, const_cast<double *>(dense), s, lay);
  hpgmg_comm_allreduce_slot_max(level, slot);
}
extern "C" void hpgmg_unpack_async(level_type *level, int id, const double *dense)
{ hpgmg_note_vector_written(level, id); launch_dense<0>(level, id, id, const_cast<double *>(dense), NULL, BoxMajorDense()); }
extern "C" void hpgmg_pack_async(level_type *level, int id, double *dense) { launch_dense<1>(level, id, id, dense, NULL, BoxMajorDense()); }
extern "C" void hpgmg_unpack_copy_norm_async(level_type *level, int id_f, int id_r, const double *dense, int slot)
{ unpack_copy_norm(level, id_f, id_r, dense, slot, BoxMajorDense()); }
extern "C" void hpgmg_grid_unpack_copy_norm_async(level_type *level, int id_f, int id_r, const double *grid, int slot)
{ unpack_copy_norm(level, id_f, id_r, grid, slot, grid_of(level)); }
extern "C" void hpgmg_grid_pack_async(level_type *level, int id, double *grid) { launch_dense<1>(level, id, id, grid, NULL, grid_of(level)); }

extern "C" void hpgmg_norm_async(level_type *level, int id_a, int slot);
/* norm(level, id_a) into `slot` and scale_vector(level, id_c, 1.0, id_a) */
extern "C" void hpgmg_copy_norm_async(level_type *level, int id_c, int id_a, int slot)
{
  const DLevel &L = dl_of(level);
  static int fuse = -1;
  if (fuse < 0) { const char *e = getenv("HPGMG_B200_FUSE_NORM"); fuse = e ? atoi(e) : 1; }
  if (!fuse || hpgmg_rt_profile() || (L.dim & 1) || hpgmg_ablate(128)) { hpgmg_norm_async(level, id_a, slot); scale_vector(level, id_c, 1.0, id_a); return; }
  double *s = hpgmg_rt_scalar_slots() + slot;
  CUDA_CHECK(cudaMemsetAsync(s, 0, sizeof(double), g_stream));
  g_launches++;
  if (L.nboxes > 0) {
    const int pairs = (L.dim / 2) * L.dim * L.dim;
    int bx = (pairs + 1023) / 1024;
    if (bx > 592) bx = 592;
    LAUNCH(copy_norm_kernel, dim3(bx, L.nboxes), 256, 0, L, id_c, id_a, s);
  }
  hpgmg_comm_allreduce_slot_max(level, slot);
}

extern "C" void hpgmg_norm_async(level_type *level, int id_a, int slot)
{
  ProfileScope prof_(&level->timers.blas1);
  double *s = hpgmg_rt_scalar_slots() + slot;
  CUDA_CHECK(cudaMemsetAsync(s, 0, sizeof(double), g_stream));
  g_launches++;
  const DLevel &L = dl_of(level);
  if (L.nboxes > 0) {
    const int cells = L.dim * L.dim * L.dim;
    int bx = (cells + 2047) / 2048;
    if (bx > 592) bx = 592;
    LAUNCH(norm_kernel, dim3(bx, L.nboxes), 256, 0, L, id_a, s);
  }
  hpgmg_comm_allreduce_slot_max(level, slot);           /* MPI_Allreduce(MAX), misc.c:324; no-op on one rank */
}

extern "C" double hpgmg_level_norm(level_type *level, int id_a)
{
  hpgmg_norm_async(level, id_a, HPGMG_SLOT_SCRATCH + 1);
  double v = 0.0;
  hpgmg_rt_read_scalars(&v, HPGMG_SLOT_SCRATCH + 1, 1);
  return v;
}

/* ---- ordered sums ------------------------------------------------------------------------------ */
/* mode 0: sum a*b ; mode 1: sum a */
__global__ void tile_sum_kernel(const DLevel L, const int id_a, const int id_b, const blockCopy_type *__restrict__ tiles, const int ntiles,
                                double *__restrict__ partials, const int mode)
{
  PDL_WAIT();
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= ntiles) return;
  const blockCopy_type B = tiles[t];
  const double *__restrict__ a = L.vec(B.read.box, id_a);
  const double *__restrict__ b = L.vec(B.read.box, id_b);
  double s = 0.0;
  for (int k = B.read.k; k < B.read.k + B.dim.k; k++)
  for (int j = B.read.j; j < B.read.j + B.dim.j; j++)
  for (int i = B.read.i; i < B.read.i + B.dim.i; i++) {
    const int ijk = i + j * L.jStride + k * L.kStride;
    if (mode == 0) s += a[ijk] * b[ijk];
    else           s += a[ijk];
  }
  partials[t] = s;
}
__global__ void ordered_total_kernel(const double *__restrict__ partials, const int n, double *__restrict__ slot)
{
  PDL_WAIT();
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    double s = 0.0;
    for (int t = 0; t < n; t++) s += partials[t];
    *slot = s;
  }
}

static double ordered_sum(level_type *level, int id_a, int id_b, int mode)
{
  ProfileScope prof_(&level->timers.blas1);
  const int slot = HPGMG_SLOT_SCRATCH + 2;
  double *s = hpgmg_rt_scalar_slots() + slot;
  hpgmg_device_level *D = HPGMG_DEV(level);
  CUDA_CHECK(cudaMemsetAsync(s, 0, sizeof(double), g_stream));
  if (D->ntiles > 0) {
    LAUNCH(tile_sum_kernel, (D->ntiles + 63) / 64, 64, 0, D->L, id_a, id_b, D->tiles, D->ntiles, D->tile_partials, mode);
    LAUNCH(ordered_total_kernel, 1, 32, 0, D->tile_partials, D->ntiles, s);
  }
  double v = 0.0;
  hpgmg_rt_read_scalars(&v, slot, 1);
  return hpgmg_comm_allreduce_sum(level, v);             /* MPI_Allreduce(SUM), misc.c:276,373 */
}

extern "C" double dot(level_type *level, int id_a, int id_b) { return ordered_sum(level, id_a, id_b, 0); }

extern "C" double mean(level_type *level, int id_a)
{
  const double sum_level = ordered_sum(level, id_a, id_a, 1);
  const double ncells_level = (double)level->dim.i * (double)level->dim.j * (double)level->dim.k;
  return sum_level / ncells_level;
}

extern "C" double error(level_type *level, int id_a, int id_b)
{
  add_vectors(level, VECTOR_TEMP, 1.0, id_a, -1.0, id_b);
  return hpgmg_level_norm(level, VECTOR_TEMP);
}
