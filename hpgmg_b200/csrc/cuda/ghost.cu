/*
 * ghost.cu -- everything that fills ghost cells: the intra-GPU part of exchange_boundary, the
 * homogeneous-Dirichlet boundary conditions (linear / quadratic / quartic extrapolation of cell
 * averages) and the extrapolation of the face coefficients.
 *
 *   exchange_boundary   operators/exchange_boundary.c:12-117 + CopyBlock operators/blockCopy.c:6-105
 *   apply_BCs_v1/v2/v4  operators/boundary_fv.c:6-90 / 101-250 / 262-569 (apply_BCs = v4, operators.fv4.c:51; v2 in the fv2 build)
 *   extrapolate_betas   operators/boundary_fv.c:573-681
 *
 * The kernels walk the device copies of the SAME block lists the reference walks (level.c:367-465,
 * 498-922): one thread block per list entry.  A BC entry's `subtype` is the normal to the DOMAIN
 * (0..26 = 13+di+3dj+9dk); ghost cells along each normal axis are produced by a 1-D extrapolation
 * from the 4 (v4) interior cells along that axis, applied axis by axis in i, j, k order -- the
 * order the reference's face / edge (16-point) / corner (64-point) code uses -- so results are
 * bit-identical.
 */
#include <string.h>
#include "common.cuh"
#include "stencil.cuh"
#include "p2p.cuh"

/* ---- copy lists ------------------------------------------------------------------------------ */
__global__ void __launch_bounds__(128) copy_blocks_kernel(const DLevel L, const int id, const blockCopy_type *__restrict__ blocks)
{
  PDL_WAIT();
  const blockCopy_type B = blocks[blockIdx.x];
  const double *__restrict__ rd;
  double *__restrict__ wr;
  int rj, rk, wj, wk;
  if (B.read.box >= 0) { rd = L.vec(B.read.box, id); rj = L.jStride; rk = L.kStride; }
  else                 { rd = B.read.ptr;            rj = B.read.jStride; rk = B.read.kStride; }
  if (B.write.box >= 0) { wr = L.vec(B.write.box, id); wj = L.jStride; wk = L.kStride; }
  else                  { wr = B.write.ptr;            wj = B.write.jStride; wk = B.write.kStride; }
  rd += B.read.i + B.read.j * rj + B.read.k * rk;
  wr += B.write.i + B.write.j * wj + B.write.k * wk;
  const int di = B.dim.i, dj = B.dim.j, cells = di * dj * B.dim.k;
  for (int c = threadIdx.x; c < cells; c += blockDim.x) {
    const int i = c % di, j = (c / di) % dj, k = c / (di * dj);
    wr[i + j * wj + k * wk] = rd[i + j * rj + k * rk];
  }
}

void hpgmg_run_copy_list(const DLevel &L, int id, const DList &list)
{
  if (list.n <= 0) return;
  LAUNCH(copy_blocks_kernel, list.n, 128, 0, L, id, list.blocks);
}

void hpgmg_fill_ghosts(level_type *level, int id, int shape, int bc_version);

extern "C" void exchange_boundary(level_type *level, int id, int shape)
{
  if (shape >= STENCIL_MAX_SHAPES) shape = STENCIL_SHAPE_BOX;
  hpgmg_device_level *D = HPGMG_DEV(level);
  communicator_type *C = &level->exchange_ghosts[shape];
  const bool remote = level->num_ranks > 1 && (C->num_sends > 0 || C->num_recvs > 0);
  if (remote) {
    const blockCopy_type *pack, *unpack;
    int npack, nunpack;
    P2PPlan *plan;
    if (D->fill_nvec == level->numVectors && level->box_ghosts == STENCIL_RADIUS && hpgmg_comm_p2p_lookup(level, shape, &pack, &npack, &unpack, &nunpack, &plan)) {
      hpgmg_fill_ghosts(level, id, shape, 0);                              /* peer stores over NVLink, no BCs */
      return;
    }
    hpgmg_run_copy_list(D->L, id, D->exchange[shape][0]);                 /* pack   */
    hpgmg_comm_exchange(level, C, 0);                                      /* ncclSend / ncclRecv */
    hpgmg_run_copy_list(D->L, id, D->exchange[shape][1]);                 /* local  */
    hpgmg_comm_exchange_wait(level, C);
    hpgmg_run_copy_list(D->L, id, D->exchange[shape][2]);                 /* unpack */
  } else {
    hpgmg_run_copy_list(D->L, id, D->exchange[shape][1]);
  }
}

/* ---- boundary conditions (device bodies in bc.cuh) ---------------------------------------------- */
#include "bc.cuh"
#include "p2p.cuh"

__global__ void __launch_bounds__(128) bc_v4_kernel(const DLevel L, const int id, const blockCopy_type *__restrict__ blocks)
{
  PDL_WAIT();
  const blockCopy_type B = blocks[blockIdx.x];
  bc_v4_block(L, id, B, threadIdx.x, blockDim.x);
}
__global__ void __launch_bounds__(128) bc_v2_kernel(const DLevel L, const int id, const blockCopy_type *__restrict__ blocks)
{
  PDL_WAIT();
  const blockCopy_type B = blocks[blockIdx.x];
  bc_v2_block(L, id, B, threadIdx.x, blockDim.x);
}

/* linear: every ghost cell of a block mirrors (with sign) the cell one step along the inverted
 * normal (boundary_fv.c:6-90).  With two ghost layers a deeper ghost reads a shallower one, possibly
 * of ANOTHER block, so the result depends on the order: the whole list is walked by one thread in
 * list order with k,j,i ascending inside a block -- the reference run on one thread.  The path only
 * runs for box_dim<2: the 1^3 bottom of an fv2 hierarchy (the radius-2 fv4 stencil never produces one). */
__global__ void bc_v1_kernel(const DLevel L, const int id, const blockCopy_type *__restrict__ blocks, const int nblocks)
{
  PDL_WAIT();
  if (blockIdx.x != 0 || threadIdx.x != 0) return;
  for (int e = 0; e < nblocks; e++) {
    const blockCopy_type B = blocks[e];
    const BCGeom G = bc_geometry(B, B.subtype, L.dim, L.jStride, L.kStride);
    double *x = L.vec(B.read.box, id);
    int m = 0;
    for (int a = 0; a < 3; a++) m += G.normal[a] ? 1 : 0;
    const double scale = (m == 2) ? 1.0 : -1.0;           /* faces -1, edges +1, corners -1 */
    const int stride = -G.normal[0] - G.normal[1] * L.jStride - G.normal[2] * L.kStride;
    const int cells = G.ext[0] * G.ext[1] * G.ext[2];
    for (int c = 0; c < cells; c++) {
      const int i = c % G.ext[0], j = (c / G.ext[0]) % G.ext[1], k = c / (G.ext[0] * G.ext[1]);
      const int ijk = (i + G.lo[0]) + (j + G.lo[1]) * L.jStride + (k + G.lo[2]) * L.kStride;
      x[ijk] = scale * x[ijk + stride];
    }
  }
}

/* ---- fused ghost fill: exchange_boundary + apply_BCs in ONE kernel ------------------------------- */
/* Thread blocks of a fill, in dispatch order:
 *   [0, npack)                 one pack-list entry each: box cells -> LL slots in the neighbour GPU's
 *                              memory (NVLink stores, p2p.cuh); never waits;              [multi-GPU]
 *   [npack, +fill blocks)      256 work items each: an item is either one ghost cell copied from the
 *                              neighbouring box on this GPU, or one BC column, which reads its interior
 *                              values straight from the box that owns them (FillBC::src), so copies
 *                              and BCs are independent of each other;
 *   [.., +nunpack)             one unpack-list entry each: poll my LL slots until the neighbour's data of
 *                              this exchange has arrived, write the ghost cells;          [multi-GPU]
 *   [.., +late blocks)         the BC columns that read those ghost cells: they wait on an in-kernel
 *                              counter until every unpack block has finished.              [multi-GPU]
 * Blocks are dispatched in index order, so a waiting block never keeps the block it waits for off the
 * machine.  version: 4 quartic, 2 quadratic (also zeroes the deeper ghost layer of a 2-layer level, like the reference).
 * The tables exist for levels of STENCIL_RADIUS ghost layers: 2 (fv4) or 1 (fv2). */
#include "fill.cuh"

struct FillArgs {
  DLevel L;
  int id, version;
  const blockCopy_type *pack, *unpack;
  int npack, nfill_blocks, nunpack, nlate_blocks;
  /* fill blocks, in this order: pair copies, single copies (FILL_BATCH x 256 items each), pair columns, single columns (256 each) */
  int nc2_blocks, nc1_blocks, nb2_blocks;
  P2PPlan *plan;
  const FillCopy *copies2;  int ncopies2;        /* two doubles per item (FillTable, common.cuh) */
  const FillCopy *copies1;  int ncopies1;
  const FillBC *bc2;        int nbc2;            /* columns i and i+1 */
  const FillBC *bc1;        int nbc1;
  const FillBC *late;       int nlate;
};

/* columns i and i+1 of a face (one normal axis) or edge (two) whose normal has no i component: the same extrapolation on
 * the two halves of 16-byte operands (all strides are even, r and w 16-byte aligned) */
__device__ __forceinline__ void bc_v4_col1_x2(const double *r, double *w, const int d0)
{
  const double2 x1 = *reinterpret_cast<const double2 *>(r + d0), x2 = *reinterpret_cast<const double2 *>(r + 2 * d0);
  const double2 x3 = *reinterpret_cast<const double2 *>(r + 3 * d0), x4 = *reinterpret_cast<const double2 *>(r + 4 * d0);
  double2 n, f;
  quartic_pair(x1.x, x2.x, x3.x, x4.x, n.x, f.x);
  quartic_pair(x1.y, x2.y, x3.y, x4.y, n.y, f.y);
  *reinterpret_cast<double2 *>(w) = n;
  *reinterpret_cast<double2 *>(w - d0) = f;
}
__device__ __forceinline__ void bc_v4_col2_x2(const double *r, double *w, const int d0, const int d1)
{
  double2 n[4], f[4];
#pragma unroll
  for (int J = 0; J < 4; J++) {
    const double *o = r + (J + 1) * d1;
    const double2 x1 = *reinterpret_cast<const double2 *>(o + d0), x2 = *reinterpret_cast<const double2 *>(o + 2 * d0);
    const double2 x3 = *reinterpret_cast<const double2 *>(o + 3 * d0), x4 = *reinterpret_cast<const double2 *>(o + 4 * d0);
    quartic_pair(x1.x, x2.x, x3.x, x4.x, n[J].x, f[J].x);
    quartic_pair(x1.y, x2.y, x3.y, x4.y, n[J].y, f[J].y);
  }
  double2 nn, nf, fn, ff;
  quartic_pair(n[0].x, n[1].x, n[2].x, n[3].x, nn.x, nf.x);
  quartic_pair(n[0].y, n[1].y, n[2].y, n[3].y, nn.y, nf.y);
  quartic_pair(f[0].x, f[1].x, f[2].x, f[3].x, fn.x, ff.x);
  quartic_pair(f[0].y, f[1].y, f[2].y, f[3].y, fn.y, ff.y);
  *reinterpret_cast<double2 *>(w) = nn;
  *reinterpret_cast<double2 *>(w - d1) = nf;
  *reinterpret_cast<double2 *>(w - d0) = fn;
  *reinterpret_cast<double2 *>(w - d0 - d1) = ff;
}

/* fill block fb: copies in batches (records, then sources, then stores: FILL_BATCH independent loads in flight
 * per thread -- the copies are latency-, not bandwidth-bound), then one BC column per thread */
#define FILL_BATCH 4
__device__ __forceinline__ void fill_block(const FillArgs &A, int fb)
{
  const DLevel &L = A.L;
  double *v = L.base + (size_t)A.id * (size_t)L.volume;
  if (fb < A.nc2_blocks) {                                          /* ---- copies, two doubles per item ---- */
    const int t0 = fb * (256 * FILL_BATCH) + threadIdx.x;
    FillCopy c[FILL_BATCH];
    double2 val[FILL_BATCH];
#pragma unroll
    for (int n = 0; n < FILL_BATCH; n++) { const int t = t0 + n * 256; c[n] = (t < A.ncopies2) ? A.copies2[t] : FillCopy{ -1, -1 }; }
#pragma unroll
    for (int n = 0; n < FILL_BATCH; n++) if (c[n].src >= 0) val[n] = *reinterpret_cast<const double2 *>(v + c[n].src);
#pragma unroll
    for (int n = 0; n < FILL_BATCH; n++) if (c[n].src >= 0) *reinterpret_cast<double2 *>(v + c[n].dst) = val[n];
  } else if ((fb -= A.nc2_blocks) < A.nc1_blocks) {                 /* ---- copies, one double per item ---- */
    const int t0 = fb * (256 * FILL_BATCH) + threadIdx.x;
    FillCopy c[FILL_BATCH];
    double val[FILL_BATCH];
#pragma unroll
    for (int n = 0; n < FILL_BATCH; n++) { const int t = t0 + n * 256; c[n] = (t < A.ncopies1) ? A.copies1[t] : FillCopy{ -1, -1 }; }
#pragma unroll
    for (int n = 0; n < FILL_BATCH; n++) if (c[n].src >= 0) val[n] = v[c[n].src];
#pragma unroll
    for (int n = 0; n < FILL_BATCH; n++) if (c[n].src >= 0) v[c[n].dst] = val[n];
  } else if ((fb -= A.nc1_blocks) < A.nb2_blocks) {                 /* ---- BC columns i, i+1 ---- */
    const int t = fb * 256 + threadIdx.x;
    if (t < A.nbc2) {
      const FillBC it = A.bc2[t];
      const BCNormal N = bc_normal(it.subtype, L.jStride, L.kStride);
      if (A.version == 4) {
        if (N.m == 1) bc_v4_col1_x2(v + it.src, v + it.dst, N.d[0]);
        else          bc_v4_col2_x2(v + it.src, v + it.dst, N.d[0], N.d[1]);
      } else {
        bc_v2_fill_col(v + it.src, v + it.dst, N.m, N.d[0], N.d[1], N.d[2]);
        bc_v2_fill_col(v + it.src + 1, v + it.dst + 1, N.m, N.d[0], N.d[1], N.d[2]);
      }
    }
  } else {                                                           /* ---- single BC columns ---- */
    fb -= A.nb2_blocks;
    fill_items(L, A.id, fb * 256 + threadIdx.x, (const FillCopy *)nullptr, 0, A.bc1, A.nbc1, A.version);
  }
}

__global__ void __launch_bounds__(256, 4) fill_ghosts_kernel(const FillArgs A)
{
  PDL_WAIT();
  const DLevel &L = A.L;
  int b = blockIdx.x;
  if (b >= A.npack && b < A.npack + A.nfill_blocks && A.plan == nullptr) {            /* single-GPU fast path */
    fill_block(A, b - A.npack);
    return;
  }
  P2PPlan *plan = A.plan;
  const unsigned long long epoch = *(volatile unsigned long long *)&plan->epoch;      /* bumped only after every block is done */
  const unsigned flag = (unsigned)(epoch + 1);
  const int parity = (int)(epoch & 1);
  if (b < A.npack) {                                                                   /* ---- pack ---- */
    const blockCopy_type B = A.pack[b];
    const int n = B.subtype;
    uint4 *slots = plan->ll_remote[n] + (size_t)parity * plan->send_size[n];
    const double *__restrict__ rd = L.vec(B.read.box, A.id) + B.read.i + B.read.j * L.jStride + B.read.k * L.kStride;
    const int di = B.dim.i, dj = B.dim.j, cells = di * dj * B.dim.k;
    const int w0 = B.write.i + B.write.j * B.write.jStride + B.write.k * B.write.kStride;
    for (int c = threadIdx.x; c < cells; c += blockDim.x) {
      const int i = c % di, j = (c / di) % dj, k = c / (di * dj);
      ll_store(slots + w0 + i + j * B.write.jStride + k * B.write.kStride, rd[i + j * L.jStride + k * L.kStride], flag);
    }
  } else if ((b -= A.npack) < A.nfill_blocks) {                                        /* ---- GPU-local copies + BCs ---- */
    fill_block(A, b);
  } else if ((b -= A.nfill_blocks) < A.nunpack) {                                      /* ---- unpack ---- */
    const blockCopy_type B = A.unpack[b];
    const int n = B.subtype;
    const uint4 *slots = plan->ll_local[n] + (size_t)parity * plan->recv_size[n];
    double *__restrict__ wr = L.vec(B.write.box, A.id) + B.write.i + B.write.j * L.jStride + B.write.k * L.kStride;
    const int di = B.dim.i, dj = B.dim.j, cells = di * dj * B.dim.k;
    const int r0 = B.read.i + B.read.j * B.read.jStride + B.read.k * B.read.kStride;
    for (int c = threadIdx.x; c < cells; c += blockDim.x) {
      const int i = c % di, j = (c / di) % dj, k = c / (di * dj);
      wr[i + j * L.jStride + k * L.kStride] = ll_load(slots + r0 + i + j * B.read.jStride + k * B.read.kStride, flag);
    }
    __syncthreads();
    if (threadIdx.x == 0) { __threadfence(); atomicAdd(&plan->unpack_done, 1u); }
  } else {                                                                             /* ---- BC columns behind unpacked cells ---- */
    b -= A.nunpack;
    if (threadIdx.x == 0) {
      while (*(volatile unsigned int *)&plan->unpack_done < (unsigned)A.nunpack) { }
      __threadfence();
    }
    __syncthreads();
    fill_items(L, A.id, b * blockDim.x + threadIdx.x, (const FillCopy *)nullptr, 0, A.late, A.nlate, A.version);
  }
  __syncthreads();
  if (threadIdx.x == 0 && atomicAdd(&plan->done, 1u) == gridDim.x - 1u) {              /* last block: re-arm, advance */
    plan->done = 0;
    plan->unpack_done = 0;
    __threadfence();
    *(volatile unsigned long long *)&plan->epoch = epoch + 1;
  }
}

/* exchange_boundary(level,id,shape) followed by apply_BCs_v4 (bc_version 4; v2 below 4^3 like
 * boundary_fv.c:269), apply_BCs_v2 (bc_version 2), or nothing (bc_version 0).  Identical results to the
 * separate list-walking kernels. */
void hpgmg_fill_ghosts(level_type *level, int id, int shape, int bc_version)
{
  ProfileScope prof_(&level->timers.ghostZone_total);
  if (hpgmg_ablate(level->box_dim >= 64 ? 1 : 2)) return;
  hpgmg_device_level *D = HPGMG_DEV(level);
  const FillTable &T = D->fill[shape];
  const bool dirichlet = level->boundary_condition.type == BC_DIRICHLET && bc_version != 0;
  int version = bc_version;
  if (version == 4 && level->box_dim < 4) version = 2;
  communicator_type *C = &level->exchange_ghosts[shape];
  const bool remote = level->num_ranks > 1 && (C->num_sends > 0 || C->num_recvs > 0);
  /* v4 needs 2 ghost layers: on a 1-layer level the list path's apply_BCs_v4 refuses it as the reference does */
  const bool have_tables = D->fill_nvec == level->numVectors && level->box_ghosts == STENCIL_RADIUS && !(version == 2 && level->box_dim < 2) &&
                           !(version == 4 && level->box_ghosts < 2);
  const blockCopy_type *pack = NULL, *unpack = NULL;
  int npack = 0, nunpack = 0;
  P2PPlan *plan = NULL;
  const int p2p = (remote && have_tables) ? hpgmg_comm_p2p_lookup(level, shape, &pack, &npack, &unpack, &nunpack, &plan) : 0;
  if (!have_tables || (remote && !p2p)) {                /* unusual geometry, or no peer mapping: the list kernels (+ NCCL) */
    exchange_boundary(level, id, shape);
    if (bc_version == 4) apply_BCs_v4(level, id, shape); else if (bc_version == 2) apply_BCs_v2(level, id, shape);
    return;
  }
  FillArgs A;
  memset(&A, 0, sizeof(A));
  A.L = D->L;  A.id = id;  A.version = version;
  A.copies2 = T.copies2;  A.ncopies2 = T.ncopies2;
  A.copies1 = T.copies1;  A.ncopies1 = T.ncopies1;
  A.bc2 = T.bc2;          A.nbc2 = dirichlet ? T.nbc2 : 0;
  A.bc1 = T.bc1;          A.nbc1 = dirichlet ? T.nbc1 : 0;
  if (level->box_dim >= 64 && hpgmg_ablate(256)) A.ncopies2 = A.ncopies1 = 0;
  if (level->box_dim >= 64 && hpgmg_ablate(512)) A.nbc2 = A.nbc1 = 0;
  A.nc2_blocks = (A.ncopies2 + 256 * FILL_BATCH - 1) / (256 * FILL_BATCH);
  A.nc1_blocks = (A.ncopies1 + 256 * FILL_BATCH - 1) / (256 * FILL_BATCH);
  A.nb2_blocks = (A.nbc2 + 255) / 256;
  A.nfill_blocks = A.nc2_blocks + A.nc1_blocks + A.nb2_blocks + (A.nbc1 + 255) / 256;
  if (remote) {
    A.pack = pack;  A.npack = npack;  A.unpack = unpack;  A.nunpack = nunpack;  A.plan = plan;
    A.late = T.late;  A.nlate = dirichlet ? T.nlate : 0;
    A.nlate_blocks = (A.nlate + 255) / 256;
  }
  const int blocks = A.npack + A.nfill_blocks + A.nunpack + A.nlate_blocks;
  if (blocks > 0) LAUNCH(fill_ghosts_kernel, blocks, 256, 0, A);
}

extern "C" void apply_BCs_v1(level_type *level, int x_id, int shape)
{
  if (shape >= STENCIL_MAX_SHAPES) shape = STENCIL_SHAPE_BOX;
  if (level->boundary_condition.type == BC_PERIODIC) return;
  const DList &list = HPGMG_DEV(level)->bc[shape];
  if (list.n > 0) LAUNCH(bc_v1_kernel, 1, 32, 0, dl_of(level), x_id, list.blocks, list.n);
}

extern "C" void apply_BCs_v2(level_type *level, int x_id, int shape)
{
  ProfileScope prof_(&level->timers.boundary_conditions);
  if (shape >= STENCIL_MAX_SHAPES) shape = STENCIL_SHAPE_BOX;
  if (level->boundary_condition.type == BC_PERIODIC) return;
  if (level->box_dim < 2) { apply_BCs_v1(level, x_id, shape); return; }
  const DList &list = HPGMG_DEV(level)->bc[shape];
  if (list.n > 0) LAUNCH(bc_v2_kernel, list.n, 128, 0, dl_of(level), x_id, list.blocks);
}

extern "C" void apply_BCs_v4(level_type *level, int x_id, int shape)
{
  ProfileScope prof_(&level->timers.boundary_conditions);
  if (shape >= STENCIL_MAX_SHAPES) shape = STENCIL_SHAPE_BOX;
  if (level->boundary_condition.type == BC_PERIODIC) return;
  if (level->box_ghosts < 2) { fprintf(stderr, "called quartic BC's with only 1 ghost zone!!!\n"); exit(0); }
  if (level->box_dim < 4) { apply_BCs_v2(level, x_id, shape); return; }
  const DList &list = HPGMG_DEV(level)->bc[shape];
  if (list.n > 0) LAUNCH(bc_v4_kernel, list.n, 128, 0, dl_of(level), x_id, list.blocks);
}

#ifdef HPGMG_FV2
extern "C" void apply_BCs(level_type *level, int x_id, int shape) { apply_BCs_v2(level, x_id, shape); }
#else
extern "C" void apply_BCs(level_type *level, int x_id, int shape) { apply_BCs_v4(level, x_id, shape); }
#endif

/* ---- face coefficients beyond the domain ------------------------------------------------------- */
/* boundary_fv.c:573-681.  Uses the BOX-shape BC list only to know which ghost regions lie outside
 * the domain; the extrapolation direction is the BOX-relative normal of the region, and beta_d is
 * not extrapolated along d.  Each list entry is processed by ONE thread in the reference's loop
 * order (k, j, i ascending): the second ghost layer reads the first, so the order is part of the
 * result.  Setup only (untimed in the reference). */
__global__ void extrapolate_betas_kernel(const DLevel L, const blockCopy_type *__restrict__ blocks, const int n)
{
  PDL_WAIT();
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n) return;
  const blockCopy_type B = blocks[e];
  const int ilo = B.read.i, jlo = B.read.j, klo = B.read.k;
  int subtype = 13;
  if (ilo < 0) subtype -= 1;
  if (jlo < 0) subtype -= 3;
  if (klo < 0) subtype -= 9;
  if (ilo >= L.dim) subtype += 1;
  if (jlo >= L.dim) subtype += 3;
  if (klo >= L.dim) subtype += 9;
  const int normal = 26 - subtype;
  const int di = (normal % 3) - 1, dj = ((normal % 9) / 3) - 1, dk = (normal / 9) - 1;
  const int jS = L.jStride, kS = L.kStride;
  double *beta_i = L.vec(B.read.box, VECTOR_BETA_I);
  double *beta_j = L.vec(B.read.box, VECTOR_BETA_J);
  double *beta_k = L.vec(B.read.box, VECTOR_BETA_K);
  const int bi = dj * jS + dk * kS;
  const int bj = di + dk * kS;
  const int bk = di + dj * jS;
  const bool do_i = (subtype != 14) && (subtype != 12);
  const bool do_j = (subtype != 16) && (subtype != 10);
  const bool do_k = (subtype != 22) && (subtype != 4);
  for (int k = 0; k < B.dim.k; k++)
  for (int j = 0; j < B.dim.j; j++)
  for (int i = 0; i < B.dim.i; i++) {
    const int ijk = (i + ilo) + (j + jlo) * jS + (k + klo) * kS;
    if (L.dim >= 5) {
      if (do_i) beta_i[ijk] = 5.0 * beta_i[ijk + bi] - 10.0 * beta_i[ijk + 2 * bi] + 10.0 * beta_i[ijk + 3 * bi] - 5.0 * beta_i[ijk + 4 * bi] + beta_i[ijk + 5 * bi];
      if (do_j) beta_j[ijk] = 5.0 * beta_j[ijk + bj] - 10.0 * beta_j[ijk + 2 * bj] + 10.0 * beta_j[ijk + 3 * bj] - 5.0 * beta_j[ijk + 4 * bj] + beta_j[ijk + 5 * bj];
      if (do_k) beta_k[ijk] = 5.0 * beta_k[ijk + bk] - 10.0 * beta_k[ijk + 2 * bk] + 10.0 * beta_k[ijk + 3 * bk] - 5.0 * beta_k[ijk + 4 * bk] + beta_k[ijk + 5 * bk];
    } else if (L.dim >= 4) {
      if (do_i) beta_i[ijk] = 4.0 * beta_i[ijk + bi] - 6.0 * beta_i[ijk + 2 * bi] + 4.0 * beta_i[ijk + 3 * bi] - beta_i[ijk + 4 * bi];
      if (do_j) beta_j[ijk] = 4.0 * beta_j[ijk + bj] - 6.0 * beta_j[ijk + 2 * bj] + 4.0 * beta_j[ijk + 3 * bj] - beta_j[ijk + 4 * bj];
      if (do_k) beta_k[ijk] = 4.0 * beta_k[ijk + bk] - 6.0 * beta_k[ijk + 2 * bk] + 4.0 * beta_k[ijk + 3 * bk] - beta_k[ijk + 4 * bk];
    } else if (L.dim >= 2) {
      if (do_i) beta_i[ijk] = 2.0 * beta_i[ijk + bi] - beta_i[ijk + 2 * bi];
      if (do_j) beta_j[ijk] = 2.0 * beta_j[ijk + bj] - beta_j[ijk + 2 * bj];
      if (do_k) beta_k[ijk] = 2.0 * beta_k[ijk + bk] - beta_k[ijk + 2 * bk];
    }
  }
}

extern "C" void extrapolate_betas(level_type *level)
{
  if (level->boundary_condition.type == BC_PERIODIC) return;
  const DList &list = HPGMG_DEV(level)->bc[STENCIL_SHAPE_BOX];
  if (list.n > 0) LAUNCH(extrapolate_betas_kernel, (list.n + 63) / 64, 64, 0, dl_of(level), list.blocks, list.n);
}
