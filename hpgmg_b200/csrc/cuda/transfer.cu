/*
 * transfer.cu -- inter-level transfer operators.
 *
 *   restriction        operators/restriction.c:6-94 (block kernel), :104-212 (driver)
 *   interpolation_v2   operators/interpolation_v2.c:8-199, :210-320   (V-cycle prolongation, +=)
 *   interpolation_v4   operators/interpolation_v4.c:8-265, :276-386   (F-cycle prolongation)
 *
 * The kernels walk the device copies of the lists MGBuild produced (mg.c:181-831): one thread
 * block per list entry; [0] writes into send buffers, [1] is rank-local, [2] unpacks receives.
 * All arithmetic keeps the reference's association order (bit-exact contract).
 */
#include "common.cuh"

void hpgmg_run_copy_list(const DLevel &L, int id, const DList &list);   /* ghost.cu */
void hpgmg_fill_ghosts(level_type *level, int id, int shape, int bc_version);

/* ---- restriction ------------------------------------------------------------------------------ */
__global__ void __launch_bounds__(128) restriction_kernel(const DLevel Lc, const int id_c, const DLevel Lf, const int id_f,
                                                          const blockCopy_type *__restrict__ blocks, const int type)
{
  PDL_WAIT();
  const blockCopy_type B = blocks[blockIdx.x];
  const double *__restrict__ rd;
  double *__restrict__ wr;
  int rj, rk, wj, wk;
  if (B.read.box >= 0) { rd = Lf.vec(B.read.box, id_f); rj = Lf.jStride; rk = Lf.kStride; }
  else                 { rd = B.read.ptr;               rj = B.read.jStride; rk = B.read.kStride; }
  if (B.write.box >= 0) { wr = Lc.vec(B.write.box, id_c); wj = Lc.jStride; wk = Lc.kStride; }
  else                  { wr = B.write.ptr;               wj = B.write.jStride; wk = B.write.kStride; }
  rd += B.read.i + B.read.j * rj + B.read.k * rk;
  wr += B.write.i + B.write.j * wj + B.write.k * wk;
  const int di = B.dim.i, dj = B.dim.j, cells = di * dj * B.dim.k;
  for (int c = threadIdx.x; c < cells; c += blockDim.x) {
    const int i = c % di, j = (c / di) % dj, k = c / (di * dj);
    const double *r = rd + 2 * i + 2 * j * rj + 2 * k * rk;
    double v;
    switch (type) {
      case RESTRICT_CELL:
        v = (r[0] + r[1] + r[rj] + r[1 + rj] + r[rk] + r[1 + rk] + r[rj + rk] + r[1 + rj + rk]) * 0.125;
        break;
      case RESTRICT_FACE_I:
        v = (r[0] + r[rj] + r[rk] + r[rj + rk]) * 0.25;
        break;
      case RESTRICT_FACE_J:
        v = (r[0] + r[1] + r[rk] + r[1 + rk]) * 0.25;
        break;
      default: /* RESTRICT_FACE_K */
        v = (r[0] + r[1] + r[rj] + r[1 + rj]) * 0.25;
        break;
    }
    wr[i + j * wj + k * wk] = v;
  }
}

/* cell restriction of box -> box entries: one thread per coarse cell, the 2x2x2 children read as four
 * 16-byte pairs (same summation order as restriction.c:54-57) */
__global__ void __launch_bounds__(256) restriction_cell_kernel(const DLevel Lc, const int id_c, const DLevel Lf, const int id_f,
                                                               const blockCopy_type *__restrict__ blocks)
{
  PDL_WAIT();
  const blockCopy_type B = blocks[blockIdx.x];
  const int di = B.dim.i, dj = B.dim.j, cells = di * dj * B.dim.k;
  const int c = blockIdx.y * blockDim.x + threadIdx.x;
  if (c >= cells) return;
  const int i = c % di, j = (c / di) % dj, k = c / (di * dj);
  const int rj = Lf.jStride, rk = Lf.kStride;
  const double *r = Lf.vec(B.read.box, id_f) + (B.read.i + 2 * i) + (B.read.j + 2 * j) * rj + (B.read.k + 2 * k) * rk;
  double v;
  if ((B.read.i & 1) == 0) {
    const double2 a = *reinterpret_cast<const double2 *>(r), b = *reinterpret_cast<const double2 *>(r + rj);
    const double2 c2 = *reinterpret_cast<const double2 *>(r + rk), d = *reinterpret_cast<const double2 *>(r + rj + rk);
    v = (a.x + a.y + b.x + b.y + c2.x + c2.y + d.x + d.y) * 0.125;
  } else {
    v = (r[0] + r[1] + r[rj] + r[1 + rj] + r[rk] + r[1 + rk] + r[rj + rk] + r[1 + rj + rk]) * 0.125;
  }
  Lc.vec(B.write.box, id_c)[(B.write.i + i) + (B.write.j + j) * Lc.jStride + (B.write.k + k) * Lc.kStride] = v;
}

static void run_restriction_list(level_type *level_c, int id_c, level_type *level_f, int id_f, const DList &list, int type)
{
  if (list.n <= 0) return;
  /* a rank that owns no coarse boxes still packs for others: give the kernel a valid (empty) DLevel */
  LAUNCH(restriction_kernel, list.n, 128, 0, dl_of(level_c), id_c, dl_of(level_f), id_f, list.blocks, type);
}

extern "C" void restriction(level_type *level_c, int id_c, level_type *level_f, int id_f, int restrictionType)
{
  ProfileScope prof_(&level_f->timers.restriction_total);
  if (hpgmg_ablate(16)) return;
  hpgmg_note_vector_written(level_c, id_c);
  hpgmg_device_level *Df = HPGMG_DEV(level_f), *Dc = HPGMG_DEV(level_c);
  communicator_type *Cf = &level_f->restriction[restrictionType], *Cc = &level_c->restriction[restrictionType];
  const int remote = (Cf->num_sends > 0) || (Cc->num_recvs > 0);
  /* peer-memory path (comm.cu): the pack list writes into the receivers' buffers; registered collectively, so both ends agree */
  DList peer_pack = { NULL, 0 };
  const int p2p_send = Cf->num_sends > 0 && hpgmg_comm_xfer_send_lookup(Cf, (const blockCopy_type **)&peer_pack.blocks, &peer_pack.n);
  const int p2p_recv = Cc->num_recvs > 0 && hpgmg_comm_xfer_recv_lookup(Cc);
  const int p2p = p2p_send || p2p_recv;
  if (remote && p2p) {
    if (p2p_send) {
      hpgmg_comm_xfer_pre(Cf);
      run_restriction_list(level_c, id_c, level_f, id_f, peer_pack, restrictionType);                            /* pack into the peers */
      hpgmg_comm_xfer_post(Cf);
    }
  } else if (remote) {
    run_restriction_list(level_c, id_c, level_f, id_f, Df->restriction[restrictionType][0], restrictionType);   /* pack */
    hpgmg_comm_transfer(level_f, Cf, level_c, Cc, 0x5);
  }
  const DList &local = Df->restriction[restrictionType][1];
  if (restrictionType == RESTRICT_CELL && local.n > 0) {                                                        /* local, fast path */
    const int half = level_f->box_dim / 2;
    const int cells = half * (half < BLOCKCOPY_TILE_J ? half : BLOCKCOPY_TILE_J) * (half < BLOCKCOPY_TILE_K ? half : BLOCKCOPY_TILE_K);
    LAUNCH(restriction_cell_kernel, dim3(local.n, (cells + 255) / 256), 256, 0, dl_of(level_c), id_c, dl_of(level_f), id_f, local.blocks);
  } else
    run_restriction_list(level_c, id_c, level_f, id_f, local, restrictionType);                                 /* local */
  if (remote) {
    if (p2p_recv) hpgmg_comm_xfer_wait(Cc);
    else if (!p2p) hpgmg_comm_transfer_wait(level_f, Cf, level_c, Cc);
    hpgmg_run_copy_list(Dc->L, id_c, Dc->restriction[restrictionType][2]);                                      /* unpack */
    if (p2p_recv) hpgmg_comm_xfer_ack(Cc);
  }
}

/* ---- interpolation (every kernel reads at most W/2 coarse ghost layers: v2 runs on 1- and 2-layer levels, v4 needs 2) ---------------------------------------------------------------------------- */
/* 1-D volume-averaged prolongation of one coarse cell into its two children.
 * quadratic (v2): lo = c0 + 1/8 (c- - c+),  hi = c0 - 1/8 (c- - c+)
 * quartic  (v4): lo = c0 + 22/128 (c-1 - c+1) + -3/128 (c-2 - c+2),  hi = c0 - ... - ...            */
__device__ __forceinline__ void prolong3(const double cm, const double c0, const double cp, double &lo, double &hi)
{
  const double c1 = 1.0 / 8.0;
  lo = (c0 + c1 * (cm - cp));
  hi = (c0 - c1 * (cm - cp));
}
__device__ __forceinline__ void prolong5(const double cmm, const double cm, const double c0, const double cp, const double cpp, double &lo, double &hi)
{
  const double c2 = -3.0 / 128.0;
  const double c1 = 22.0 / 128.0;
  lo = (c0 + c1 * (cm - cp) + c2 * (cmm - cpp));
  hi = (c0 - c1 * (cm - cp) - c2 * (cmm - cpp));
}

/* box -> MESSAGE entries (the fine boxes belong to another rank, mg.c:246-270), W = 3 (v2) or 5 (v4): the message is dense
 * [k][j][i] at fine resolution.  The reference interpolates "in place" into its send buffer with prescale 0.0, i.e. it
 * computes 0.0*old + value (blockCopy.c:153 remark) -- old being what the buffer held from the previous message.  With peer
 * memory the message is written straight into the RECEIVER's buffer; reading `old` from there would be an NVLink round trip
 * per cell, so the rank's own send buffer is kept as a mirror: old is read from it, the value goes to both.  Fine i-pairs
 * leave as 16-byte stores (the 8-byte stores of the generic kernel reached the peer half-empty: 80 us per message). */
template <int W>
__global__ void __launch_bounds__(128) interpolation_pack_kernel(const DLevel Lc, const int id_c, const blockCopy_type *__restrict__ blocks,
                                                                 const blockCopy_type *__restrict__ mirror_blocks)
{
  PDL_WAIT();
  constexpr int R = W / 2;
  const blockCopy_type B = blocks[blockIdx.x];
  const int rj = Lc.jStride, rk = Lc.kStride, wj = B.write.jStride, wk = B.write.kStride;
  const double *__restrict__ rd = Lc.vec(B.read.box, id_c);
  double *__restrict__ wr = B.write.ptr;
  double *__restrict__ mr = mirror_blocks ? mirror_blocks[blockIdx.x].write.ptr : B.write.ptr;       /* where `old` lives */
  const bool twice = mirror_blocks != nullptr;
  const int di = B.dim.i, dj = B.dim.j, cells = di * dj * B.dim.k;
  for (int c = threadIdx.x; c < cells; c += blockDim.x) {
    const int ii = c % di, jj = (c / di) % dj, kk = c / (di * dj);
    const double *r = rd + (ii + B.read.i) + (jj + B.read.j) * rj + (kk + B.read.k) * rk;
    double fj[2][2][W];
#pragma unroll
    for (int K = 0; K < W; K++) {
      double fi[2][W];
#pragma unroll
      for (int J = 0; J < W; J++) {
        const double *p = r + (J - R) * rj + (K - R) * rk;
        if constexpr (W == 3) prolong3(p[-1], p[0], p[1], fi[0][J], fi[1][J]);
        else                  prolong5(p[-2], p[-1], p[0], p[1], p[2], fi[0][J], fi[1][J]);
      }
#pragma unroll
      for (int I = 0; I < 2; I++) {
        if constexpr (W == 3) prolong3(fi[I][0], fi[I][1], fi[I][2], fj[I][0][K], fj[I][1][K]);
        else                  prolong5(fi[I][0], fi[I][1], fi[I][2], fi[I][3], fi[I][W - 1], fj[I][0][K], fj[I][1][K]);
      }
    }
    const int off = (2 * ii + B.write.i) + (2 * jj + B.write.j) * wj + (2 * kk + B.write.k) * wk;
    const bool vec2 = ((off & 1) == 0) && ((reinterpret_cast<uintptr_t>(wr) & 15) == 0) && ((reinterpret_cast<uintptr_t>(mr) & 15) == 0) && ((wj & 1) == 0) && ((wk & 1) == 0);
#pragma unroll
    for (int J = 0; J < 2; J++) {
      double lo[2], hi[2];
#pragma unroll
      for (int I = 0; I < 2; I++) {
        if constexpr (W == 3) prolong3(fj[I][J][0], fj[I][J][1], fj[I][J][2], lo[I], hi[I]);
        else                  prolong5(fj[I][J][0], fj[I][J][1], fj[I][J][2], fj[I][J][3], fj[I][J][W - 1], lo[I], hi[I]);
      }
      const int o = off + J * wj;
      const double a0 = 0.0 * mr[o] + lo[0], a1 = 0.0 * mr[o + 1] + lo[1], b0 = 0.0 * mr[o + wk] + hi[0], b1 = 0.0 * mr[o + wk + 1] + hi[1];
      if (vec2) {
        *reinterpret_cast<double2 *>(wr + o) = make_double2(a0, a1);
        *reinterpret_cast<double2 *>(wr + o + wk) = make_double2(b0, b1);
        if (twice) { *reinterpret_cast<double2 *>(mr + o) = make_double2(a0, a1); *reinterpret_cast<double2 *>(mr + o + wk) = make_double2(b0, b1); }
      } else {
        wr[o] = a0;  wr[o + 1] = a1;  wr[o + wk] = b0;  wr[o + wk + 1] = b1;
        if (twice) { mr[o] = a0;  mr[o + 1] = a1;  mr[o + wk] = b0;  mr[o + wk + 1] = b1; }
      }
    }
  }
}

/* box -> box entries, staged through shared memory: a thread block takes a
 * 32 x 4 x 2 sub-tile of coarse cells of one list entry, loads the tile plus its W/2-cell halo once
 * (instead of every thread fetching 27 / 125 overlapping values through L1), and writes each fine
 * i-pair as one 16-byte access. */
template <int W>
__global__ void __launch_bounds__(256) interpolation_tiled_kernel(const DLevel Lf, const int id_f, const double prescale,
                                                                  const DLevel Lc, const int id_c,
                                                                  const blockCopy_type *__restrict__ blocks)
{
  PDL_WAIT();
  constexpr int R = W / 2, CI = 32, CJ = 4, CK = 2;
  constexpr int SI = CI + 2 * R, SJ = CJ + 2 * R, SK = CK + 2 * R;
  __shared__ double tile[SK][SJ][SI];
  const blockCopy_type B = blocks[blockIdx.x];
  const int di = B.dim.i, dj = B.dim.j, dk = B.dim.k;
  const int ni = (di + CI - 1) / CI, nj = (dj + CJ - 1) / CJ;
  const int ti0 = ((int)blockIdx.y % ni) * CI, tj0 = (((int)blockIdx.y / ni) % nj) * CJ, tk0 = ((int)blockIdx.y / (ni * nj)) * CK;
  if (tk0 >= dk) return;
  const int rj = Lc.jStride, rk = Lc.kStride, wj = Lf.jStride, wk = Lf.kStride;
  const double *__restrict__ rd = Lc.vec(B.read.box, id_c) + (B.read.i + ti0 - R) + (B.read.j + tj0 - R) * rj + (B.read.k + tk0 - R) * rk;
  const int tid = threadIdx.x + CI * (threadIdx.y + CJ * threadIdx.z);
  /* only the part of the halo tile that some coarse cell of this sub-tile needs */
  const int ei = min(CI, di - ti0) + 2 * R, ej = min(CJ, dj - tj0) + 2 * R, ek = min(CK, dk - tk0) + 2 * R;
  for (int e = tid; e < SI * SJ * SK; e += CI * CJ * CK) {
    const int i = e % SI, j = (e / SI) % SJ, k = e / (SI * SJ);
    if (i < ei && j < ej && k < ek) tile[k][j][i] = rd[i + j * rj + k * rk];
  }
  __syncthreads();
  const int ii = ti0 + threadIdx.x, jj = tj0 + threadIdx.y, kk = tk0 + threadIdx.z;
  if (ii >= di || jj >= dj || kk >= dk) return;
  const int cx = threadIdx.x + R, cy = threadIdx.y + R, cz = threadIdx.z + R;
  double fi[2][W][W];
#pragma unroll
  for (int K = 0; K < W; K++)
#pragma unroll
  for (int J = 0; J < W; J++) {
    const double *p = &tile[cz + K - R][cy + J - R][cx];
    if constexpr (W == 3) prolong3(p[-1], p[0], p[1], fi[0][J][K], fi[1][J][K]);
    else                  prolong5(p[-2], p[-1], p[0], p[1], p[2], fi[0][J][K], fi[1][J][K]);
  }
  double fj[2][2][W];
#pragma unroll
  for (int K = 0; K < W; K++)
#pragma unroll
  for (int I = 0; I < 2; I++) {
    if constexpr (W == 3) prolong3(fi[I][0][K], fi[I][1][K], fi[I][2][K], fj[I][0][K], fj[I][1][K]);
    else                  prolong5(fi[I][0][K], fi[I][1][K], fi[I][2][K], fi[I][3][K], fi[I][W - 1][K], fj[I][0][K], fj[I][1][K]);
  }
  double *w = Lf.vec(B.write.box, id_f) + (2 * ii + B.write.i) + (2 * jj + B.write.j) * wj + (2 * kk + B.write.k) * wk;
  const bool vec2 = (((B.write.i) & 1) == 0);             /* fine i-pairs are 16-byte aligned when the entry starts on an even cell */
#pragma unroll
  for (int J = 0; J < 2; J++) {
    double lo[2], hi[2];
#pragma unroll
    for (int I = 0; I < 2; I++) {
      if constexpr (W == 3) prolong3(fj[I][J][0], fj[I][J][1], fj[I][J][2], lo[I], hi[I]);
      else                  prolong5(fj[I][J][0], fj[I][J][1], fj[I][J][2], fj[I][J][3], fj[I][J][W - 1], lo[I], hi[I]);
    }
    double *w0 = w + J * wj;
    if (vec2 && prescale == 0.0) {
      /* interpolation_fcycle: 0.0*old + new.  The old value is not read (8 of 17 B per fine cell): for finite old values the
       * result is the same number (blockCopy.c:153 makes finite destinations the caller's duty: 0.0*NaN), at most the sign
       * of an exact zero differs. */
      *reinterpret_cast<double2 *>(w0) = make_double2(lo[0], lo[1]);
      *reinterpret_cast<double2 *>(w0 + wk) = make_double2(hi[0], hi[1]);
    } else if (vec2) {
      double2 a = *reinterpret_cast<double2 *>(w0), b2 = *reinterpret_cast<double2 *>(w0 + wk);
      a.x = prescale * a.x + lo[0];   a.y = prescale * a.y + lo[1];
      b2.x = prescale * b2.x + hi[0]; b2.y = prescale * b2.y + hi[1];
      *reinterpret_cast<double2 *>(w0) = a;
      *reinterpret_cast<double2 *>(w0 + wk) = b2;
    } else {
      w0[0] = prescale * w0[0] + lo[0];        w0[1] = prescale * w0[1] + lo[1];
      w0[wk] = prescale * w0[wk] + hi[0];      w0[wk + 1] = prescale * w0[wk + 1] + hi[1];
    }
  }
}

/* The same arithmetic again, marching along k: a thread owns one (i, j) column of coarse cells of a list entry.
 * Per coarse PLANE it loads the W x W values around its column once, runs the i- and j-passes (W + 2 one-
 * dimensional prolongations) and pushes the four (fine i, fine j) results into a W-deep register window; the k-pass
 * of coarse cell k then reads that window.  A coarse cell costs W*W loads and W+2+4 prolongations instead of
 * W*W*W loads and W*W+2W+4 (the tiled kernel above is LSU-bound on exactly those loads); the W-1 planes of run-in
 * are paid once per entry (8 planes deep, mg.c:274-277).  Lanes run along i, so the loads are coalesced rows
 * straight through L1.  Same prolong3/prolong5 calls on the same operands in the same order: same bits. */
template <int W>
__global__ void __launch_bounds__(256) interpolation_march_kernel(const DLevel Lf, const int id_f, const double prescale,
                                                                  const DLevel Lc, const int id_c,
                                                                  const blockCopy_type *__restrict__ blocks)
{
  PDL_WAIT();
  constexpr int R = W / 2;
  const blockCopy_type B = blocks[blockIdx.x];
  const int di = B.dim.i, dj = B.dim.j, dk = B.dim.k;
  const int col = blockIdx.y * blockDim.x + threadIdx.x;
  if (col >= di * dj) return;
  const int ii = col % di, jj = col / di;
  const int rj = Lc.jStride, rk = Lc.kStride, wj = Lf.jStride, wk = Lf.kStride;
  const double *__restrict__ r = Lc.vec(B.read.box, id_c) + (B.read.i + ii) + (B.read.j + jj) * rj + (B.read.k - R) * rk;   /* plane k-R of the column */
  double *w = Lf.vec(B.write.box, id_f) + (2 * ii + B.write.i) + (2 * jj + B.write.j) * wj + B.write.k * wk;
  const bool vec2 = ((B.write.i & 1) == 0);
  double win[2][2][W];                                            /* [fine i][fine j][coarse plane k-R .. k+R] */
#pragma unroll 1
  for (int K = 0; K < dk + 2 * R; K++, r += rk) {
    /* i-pass on the W rows of this coarse plane, then the j-pass */
    double fi[2][W];
#pragma unroll
    for (int J = 0; J < W; J++) {
      const double *p = r + (J - R) * rj;
      if constexpr (W == 3) prolong3(p[-1], p[0], p[1], fi[0][J], fi[1][J]);
      else                  prolong5(p[-2], p[-1], p[0], p[1], p[2], fi[0][J], fi[1][J]);
    }
#pragma unroll
    for (int I = 0; I < 2; I++) {
#pragma unroll
      for (int q = 0; q < W - 1; q++) { win[I][0][q] = win[I][0][q + 1]; win[I][1][q] = win[I][1][q + 1]; }
      if constexpr (W == 3) prolong3(fi[I][0], fi[I][1], fi[I][2], win[I][0][W - 1], win[I][1][W - 1]);
      else                  prolong5(fi[I][0], fi[I][1], fi[I][2], fi[I][3], fi[I][4], win[I][0][W - 1], win[I][1][W - 1]);
    }
    if (K < 2 * R) continue;                                      /* window not full yet */
    /* k-pass for coarse cell K-2R and commit its 8 fine cells */
    double *w0 = w + 2 * (K - 2 * R) * wk;
#pragma unroll
    for (int J = 0; J < 2; J++) {
      double lo[2], hi[2];
#pragma unroll
      for (int I = 0; I < 2; I++) {
        if constexpr (W == 3) prolong3(win[I][J][0], win[I][J][1], win[I][J][2], lo[I], hi[I]);
        else                  prolong5(win[I][J][0], win[I][J][1], win[I][J][2], win[I][J][3], win[I][J][4], lo[I], hi[I]);
      }
      double *wr = w0 + J * wj;
      if (vec2 && prescale == 0.0) {                             /* see interpolation_tiled_kernel: the old value is not read */
        *reinterpret_cast<double2 *>(wr) = make_double2(lo[0], lo[1]);
        *reinterpret_cast<double2 *>(wr + wk) = make_double2(hi[0], hi[1]);
      } else if (vec2) {
        double2 a = *reinterpret_cast<double2 *>(wr), b2 = *reinterpret_cast<double2 *>(wr + wk);
        a.x = prescale * a.x + lo[0];   a.y = prescale * a.y + lo[1];
        b2.x = prescale * b2.x + hi[0]; b2.y = prescale * b2.y + hi[1];
        *reinterpret_cast<double2 *>(wr) = a;
        *reinterpret_cast<double2 *>(wr + wk) = b2;
      } else {
        wr[0] = prescale * wr[0] + lo[0];        wr[1] = prescale * wr[1] + lo[1];
        wr[wk] = prescale * wr[wk] + hi[0];      wr[wk + 1] = prescale * wr[wk + 1] + hi[1];
      }
    }
  }
}

/* ---- piecewise-constant prolongation (interpolation_p0): every fine cell = prescale*fine + its coarse parent; no ghost cells ---- */
/* box -> box entries: one thread per fine i-pair (both cells share the parent), 16-byte accesses where the pair is aligned
 * (create_vectors aligns cell 0, so: where the entry starts on an even fine cell) */
__global__ void __launch_bounds__(256) interpolation_p0_kernel(const DLevel Lf, const int id_f, const double prescale,
                                                               const DLevel Lc, const int id_c, const blockCopy_type *__restrict__ blocks)
{
  PDL_WAIT();
  const blockCopy_type B = blocks[blockIdx.x];
  const int di = B.dim.i, fj = 2 * B.dim.j, fk = 2 * B.dim.k;     /* coarse i (= fine pairs), fine j, fine k */
  const int t = blockIdx.y * blockDim.x + threadIdx.x;
  if (t >= di * fj * fk) return;
  const int ii = t % di, j = (t / di) % fj, k = t / (di * fj);
  const double c = Lc.vec(B.read.box, id_c)[(B.read.i + ii) + (B.read.j + (j >> 1)) * Lc.jStride + (B.read.k + (k >> 1)) * Lc.kStride];
  double *w = Lf.vec(B.write.box, id_f) + (B.write.i + 2 * ii) + (B.write.j + j) * Lf.jStride + (B.write.k + k) * Lf.kStride;
  if ((B.write.i & 1) == 0) {
    double2 o = *reinterpret_cast<double2 *>(w);
    o.x = prescale * o.x + c;  o.y = prescale * o.y + c;
    *reinterpret_cast<double2 *>(w) = o;
  } else {
    w[0] = prescale * w[0] + c;  w[1] = prescale * w[1] + c;
  }
}

/* box -> MESSAGE entries: the sender interpolates into the message with prescale 0.0, i.e. 0.0*old + value; `old` is read from
 * the rank's own send buffer when the message goes straight into the receiver's memory (see interpolation_pack_kernel) */
__global__ void __launch_bounds__(128) interpolation_p0_pack_kernel(const DLevel Lc, const int id_c, const blockCopy_type *__restrict__ blocks,
                                                                    const blockCopy_type *__restrict__ mirror_blocks)
{
  PDL_WAIT();
  const blockCopy_type B = blocks[blockIdx.x];
  const int rj = Lc.jStride, rk = Lc.kStride, wj = B.write.jStride, wk = B.write.kStride;
  const double *__restrict__ rd = Lc.vec(B.read.box, id_c) + B.read.i + B.read.j * rj + B.read.k * rk;
  const int w0 = B.write.i + B.write.j * wj + B.write.k * wk;
  double *__restrict__ wr = B.write.ptr + w0;
  double *__restrict__ mr = (mirror_blocks ? mirror_blocks[blockIdx.x].write.ptr : B.write.ptr) + w0;
  const bool twice = mirror_blocks != nullptr;
  const int fi = 2 * B.dim.i, fj = 2 * B.dim.j, cells = fi * fj * 2 * B.dim.k;
  for (int c = threadIdx.x; c < cells; c += blockDim.x) {
    const int i = c % fi, j = (c / fi) % fj, k = c / (fi * fj);
    const int o = i + j * wj + k * wk;
    const double v = 0.0 * mr[o] + rd[(i >> 1) + (j >> 1) * rj + (k >> 1) * rk];
    wr[o] = v;
    if (twice) mr[o] = v;
  }
}

/* fine-level unpack of prolonged data received from another rank: write = prescale*write + recv
 * (IncrementBlock, blockCopy.c:108-156) */
__global__ void __launch_bounds__(128) increment_blocks_kernel(const DLevel L, const int id, const double prescale, const blockCopy_type *__restrict__ blocks)
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
    double *w = wr + i + j * wj + k * wk;
    w[0] = prescale * w[0] + rd[i + j * rj + k * rk];
  }
}

/* the kernels of prolongation W: 1 piecewise constant (p0), 3 quadratic (v2), 5 quartic (v4) */
template <int W>
static void launch_interpolation_pack(const DLevel &Lc, const int id_c, const DList &list, const blockCopy_type *mirror)
{
  if (list.n <= 0) return;
  if constexpr (W == 1) LAUNCH(interpolation_p0_pack_kernel, list.n, 128, 0, Lc, id_c, list.blocks, mirror);
  else                  LAUNCH(interpolation_pack_kernel<W>, list.n, 128, 0, Lc, id_c, list.blocks, mirror);
}

template <int W>
static void interpolation_driver(level_type *level_f, int id_f, double prescale_f, level_type *level_c, int id_c)
{
  ProfileScope prof_(&level_f->timers.interpolation_total);
  if (hpgmg_ablate(16)) return;
  hpgmg_note_vector_written(level_f, id_f);
  hpgmg_device_level *Df = HPGMG_DEV(level_f), *Dc = HPGMG_DEV(level_c);
  communicator_type *Cc = &level_c->interpolation, *Cf = &level_f->interpolation;
  const int remote = (Cc->num_sends > 0) || (Cf->num_recvs > 0);
  DList peer_pack = { NULL, 0 };
  const int p2p_send = Cc->num_sends > 0 && hpgmg_comm_xfer_send_lookup(Cc, (const blockCopy_type **)&peer_pack.blocks, &peer_pack.n);
  const int p2p_recv = Cf->num_recvs > 0 && hpgmg_comm_xfer_recv_lookup(Cf);
  const int p2p = p2p_send || p2p_recv;
  if (remote && p2p) {
    if (p2p_send) {                                                  /* interpolate straight into the fine boxes' owners (comm.cu) */
      hpgmg_comm_xfer_pre(Cc);
      launch_interpolation_pack<W>(Dc->L, id_c, peer_pack, Dc->interpolation[0].blocks);
      hpgmg_comm_xfer_post(Cc);
    }
  } else if (remote) {
    const DList &pack = Dc->interpolation[0];
    launch_interpolation_pack<W>(Dc->L, id_c, pack, (const blockCopy_type *)NULL);
    hpgmg_comm_transfer(level_c, Cc, level_f, Cf, 0x7);
  }
  const DList &local = Dc->interpolation[1];
  if constexpr (W == 1) {
    if (local.n > 0) {
      /* local entries are box -> box tiles of at most 10000 x 8 x 8 coarse cells (mg.c:274-277) */
      const int half = level_f->box_dim / 2;
      const int pairs = half * 2 * (half < BLOCKCOPY_TILE_J ? half : BLOCKCOPY_TILE_J) * 2 * (half < BLOCKCOPY_TILE_K ? half : BLOCKCOPY_TILE_K);
      LAUNCH(interpolation_p0_kernel, dim3(local.n, (pairs + 255) / 256), dim3(256), 0, Df->L, id_f, prescale_f, Dc->L, id_c, local.blocks);
    }
  } else if (local.n > 0) {
    /* local entries are box -> box tiles of at most 10000 x 8 x 8 coarse cells (mg.c:274-277) */
    const int half = level_f->box_dim / 2;
    const int di = half, dj = half < BLOCKCOPY_TILE_J ? half : BLOCKCOPY_TILE_J, dk = half < BLOCKCOPY_TILE_K ? half : BLOCKCOPY_TILE_K;
    const int subtiles = ((di + 31) / 32) * ((dj + 3) / 4) * ((dk + 1) / 2);
    static int march = -1;
    if (march < 0) { const char *e = getenv("HPGMG_B200_INTERP_MARCH"); march = e ? atoi(e) : 512; }   /* minimum columns per entry: the planes of a column are sequential, small levels need the width */
    if (march && dk >= 4 && di * dj >= march)
      LAUNCH(interpolation_march_kernel<W>, dim3(local.n, (di * dj + 255) / 256), dim3(256), 0, Df->L, id_f, prescale_f, Dc->L, id_c, local.blocks);
    else
      LAUNCH(interpolation_tiled_kernel<W>, dim3(local.n, subtiles), dim3(32, 4, 2), 0, Df->L, id_f, prescale_f, Dc->L, id_c, local.blocks);
  }
  if (remote) {
    if (p2p_recv) hpgmg_comm_xfer_wait(Cf);
    else if (!p2p) hpgmg_comm_transfer_wait(level_c, Cc, level_f, Cf);
    const DList &unpack = Df->interpolation[2];
    if (unpack.n > 0) LAUNCH(increment_blocks_kernel, unpack.n, 128, 0, Df->L, id_f, prescale_f, unpack.blocks);
    if (p2p_recv) hpgmg_comm_xfer_ack(Cf);
  }
}

extern "C" void interpolation_v2(level_type *level_f, int id_f, double prescale_f, level_type *level_c, int id_c)
{
  hpgmg_fill_ghosts(level_c, id_c, STENCIL_SHAPE_BOX, 2);       /* exchange_boundary(BOX) + apply_BCs_v2(BOX), fused */
  interpolation_driver<3>(level_f, id_f, prescale_f, level_c, id_c);
}

extern "C" void interpolation_v4(level_type *level_f, int id_f, double prescale_f, level_type *level_c, int id_c)
{
  hpgmg_fill_ghosts(level_c, id_c, STENCIL_SHAPE_BOX, 4);       /* exchange_boundary(BOX) + apply_BCs_v4(BOX), fused */
  interpolation_driver<5>(level_f, id_f, prescale_f, level_c, id_c);
}

/* interpolation_p0.c: reads only the coarse parents, so no ghost fill */
extern "C" void interpolation_p0(level_type *level_f, int id_f, double prescale_f, level_type *level_c, int id_c)
{
  interpolation_driver<1>(level_f, id_f, prescale_f, level_c, id_c);
}

/* operators.fv4.c:204-205: v2 / v4; operators.fv2.c: p0 / v2 */
extern "C" void interpolation_vcycle(level_type *level_f, int id_f, double prescale_f, level_type *level_c, int id_c)
{
#ifdef HPGMG_FV2
  interpolation_p0(level_f, id_f, prescale_f, level_c, id_c);
#else
  interpolation_v2(level_f, id_f, prescale_f, level_c, id_c);
#endif
}
extern "C" void interpolation_fcycle(level_type *level_f, int id_f, double prescale_f, level_type *level_c, int id_c)
{
#ifdef HPGMG_FV2
  interpolation_v2(level_f, id_f, prescale_f, level_c, id_c);
#else
  interpolation_v4(level_f, id_f, prescale_f, level_c, id_c);
#endif
}
