/*
 * mg.c -- multigrid hierarchy construction and the V / F cycles for the B200 build.
 *
 * Restates /root/reference/finite-volume/source/mg.c: build_interpolation :181, build_restriction
 * :484, MGBuild :842 (level table :895-952), MGDestroy :1027, richardson_error :1113, MGVCycle
 * :1135, MGSolve :1168, FMGSolve :1237, FMGSolve2 :1348, MGPCG :1500, MGPrintTiming :54.
 *
 * The cycle bodies only ENQUEUE work on the GPU stream.  A whole FMGSolve is ~1.7k kernel
 * launches (SURVEY.md appendix C), so the body is recorded once into a CUDA graph and replayed;
 * the two norms the reference prints (mg.c:1265,1322) are left in device scalars and read back
 * once, after the solve, which is the only host<->device synchronisation of a solve.
 */
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <math.h>

#include "hpgmg_b200.h"
#include "runtime.h"

void hpgmg_free_communicator(communicator_type *c);   /* level.c */

/* ------------------------------------------------------------------------------------------ */
/* one fine-box <-> coarse-box relation of an inter-level transfer */
typedef struct {
  int sendRank, sendBoxID, sendBox;
  int recvRank, recvBoxID, recvBox;
  int i, j, k;                       /* offset of the fine box's image inside the coarse box */
} transfer_msg;

/* Buffers are ordered by (sendRank, sendBoxID); the reference (mg.c:38-48) stops there and relies
 * on a stable sort when one coarse box feeds several fine boxes.  Adding recvBoxID as the last key
 * gives that same order deterministically on both ends. */
static int cmp_transfer_msg(const void *pa, const void *pb)
{
  const transfer_msg *a = (const transfer_msg *)pa, *b = (const transfer_msg *)pb;
  if (a->sendRank  != b->sendRank)  return (a->sendRank  > b->sendRank)  ? 1 : -1;
  if (a->sendBoxID != b->sendBoxID) return (a->sendBoxID > b->sendBoxID) ? 1 : -1;
  if (a->recvBoxID != b->recvBoxID) return (a->recvBoxID > b->recvBoxID) ? 1 : -1;
  return 0;
}

static int sorted_unique(int *v, int n)
{
  qsort(v, n, sizeof(int), qsortInt);
  int m = 0;
  for (int i = 0; i < n; i++)
    if (m == 0 || v[i] != v[m - 1]) v[m++] = v[i];
  return m;
}

static int local_index_of_box(const level_type *L, int global_id)
{
  for (int b = 0; b < L->num_my_boxes; b++)
    if (L->my_boxes[b].global_box_id == global_id) return b;
  return -1;
}

static inline int box_id(const level_type *L, int bi, int bj, int bk)
{
  return bi + bj * L->boxes_in.i + bk * L->boxes_in.i * L->boxes_in.j;
}

static void alloc_neighbours(int n, int **ranks, int **sizes, double ***buffers)
{
  int m = n > 0 ? n : 1;
  *ranks   = (int *)calloc((size_t)m, sizeof(int));
  *sizes   = (int *)calloc((size_t)m, sizeof(int));
  *buffers = (double **)calloc((size_t)m, sizeof(double *));
}

/* dimensions of the coarse image of one fine box of side `fine_dim` (mg.c:574-588) */
static void restricted_extent(int type, int fine_dim, int *ei, int *ej, int *ek)
{
  *ei = *ej = *ek = fine_dim / 2;
  if (type == RESTRICT_FACE_I) (*ei)++;
  if (type == RESTRICT_FACE_J) (*ej)++;
  if (type == RESTRICT_FACE_K) (*ek)++;
}

/* ------------------------------------------------------------------------------------------ */
/* Restriction program of every level for one restriction type (mg.c:484-831).
 * levels[l].restriction[type] holds: [0] restrict my fine boxes into send buffers,
 * [1] restrict my fine boxes into my coarse boxes, and (on the coarse side, stored on level l
 * for data arriving from l-1) [2] copy received images into my coarse boxes. */
static void build_restriction(mg_type *MG, int type)
{
  for (int l = 0; l < MG->num_levels; l++) {
    level_type *L = MG->levels[l];
    communicator_type *C = &L->restriction[type];
    memset(C, 0, sizeof(*C));

    /* ---- fine side: pack + local ---------------------------------------------------- */
    if (l < MG->num_levels - 1 && L->num_my_boxes > 0) {
      level_type *Lc = MG->levels[l + 1];
      const int ratio_i = L->boxes_in.i / Lc->boxes_in.i;      /* fine boxes per coarse box, per axis */
      const int ratio_j = L->boxes_in.j / Lc->boxes_in.j;
      const int ratio_k = L->boxes_in.k / Lc->boxes_in.k;
      const int half = L->box_dim / 2;
      transfer_msg *msg = (transfer_msg *)malloc((size_t)L->num_my_boxes * sizeof(transfer_msg));
      int *ranks = (int *)malloc((size_t)L->num_my_boxes * sizeof(int));
      int nRemote = 0;
      for (int f = 0; f < L->num_my_boxes; f++) {
        int fi = L->my_boxes[f].low.i / L->box_dim, fj = L->my_boxes[f].low.j / L->box_dim, fk = L->my_boxes[f].low.k / L->box_dim;
        int cid = box_id(Lc, fi * Lc->boxes_in.i / L->boxes_in.i, fj * Lc->boxes_in.j / L->boxes_in.j, fk * Lc->boxes_in.k / L->boxes_in.k);
        transfer_msg *m = &msg[f];
        m->sendRank = L->rank_of_box[L->my_boxes[f].global_box_id];
        m->sendBoxID = L->my_boxes[f].global_box_id;   m->sendBox = f;
        m->recvRank = Lc->rank_of_box[cid];            m->recvBoxID = cid;
        m->recvBox = local_index_of_box(Lc, cid);
        m->i = half * (fi % ratio_i);  m->j = half * (fj % ratio_j);  m->k = half * (fk % ratio_k);
        if (m->recvRank != L->my_rank) ranks[nRemote++] = m->recvRank;
      }
      qsort(msg, L->num_my_boxes, sizeof(transfer_msg), cmp_transfer_msg);
      const int nRanks = sorted_unique(ranks, nRemote);
      int ei, ej, ek;
      restricted_extent(type, L->box_dim, &ei, &ej, &ek);
      const int elem = ei * ej * ek;

      C->num_sends = nRanks;
      if (nRanks > 0) {
        alloc_neighbours(nRanks, &C->send_ranks, &C->send_sizes, &C->send_buffers);
        double *bulk = (double *)MALLOC((size_t)nRemote * elem * sizeof(double));
        for (int r = 0; r < nRanks; r++) {
          int offset = 0;
          C->send_buffers[r] = bulk;
          for (int m = 0; m < L->num_my_boxes; m++) if (msg[m].recvRank == ranks[r]) {
            const box_type *fb = &L->my_boxes[msg[m].sendBox];
            append_block_to_list(&C->blocks[0], &C->allocated_blocks[0], &C->num_blocks[0], ei, ej, ek,
                                 msg[m].sendBox, NULL, 0, 0, 0, fb->jStride, fb->kStride, 2,
                                 -1, C->send_buffers[r], offset, 0, 0, ei, ei * ej, 1,
                                 BLOCKCOPY_TILE_I, BLOCKCOPY_TILE_J, BLOCKCOPY_TILE_K, 0);
            offset += elem;
          }
          C->send_ranks[r] = ranks[r];
          C->send_sizes[r] = offset;
          bulk += offset;
        }
      }
      for (int m = 0; m < L->num_my_boxes; m++) if (msg[m].recvRank == Lc->my_rank) {
        const box_type *fb = &L->my_boxes[msg[m].sendBox];
        const box_type *cb = &Lc->my_boxes[msg[m].recvBox];
        append_block_to_list(&C->blocks[1], &C->allocated_blocks[1], &C->num_blocks[1], ei, ej, ek,
                             msg[m].sendBox, NULL, 0, 0, 0, fb->jStride, fb->kStride, 2,
                             msg[m].recvBox, NULL, msg[m].i, msg[m].j, msg[m].k, cb->jStride, cb->kStride, 1,
                             BLOCKCOPY_TILE_I, BLOCKCOPY_TILE_J, BLOCKCOPY_TILE_K, 0);
      }
      free(msg);
      free(ranks);
    }

    /* ---- coarse side: unpack ---------------------------------------------------------- */
    if (l > 0 && L->num_my_boxes > 0) {
      level_type *Lf = MG->levels[l - 1];
      const int ratio_i = Lf->boxes_in.i / L->boxes_in.i;
      const int ratio_j = Lf->boxes_in.j / L->boxes_in.j;
      const int ratio_k = Lf->boxes_in.k / L->boxes_in.k;
      const int cap = ratio_i * ratio_j * ratio_k * L->num_my_boxes;
      transfer_msg *msg = (transfer_msg *)malloc((size_t)cap * sizeof(transfer_msg));
      int *ranks = (int *)malloc((size_t)cap * sizeof(int));
      int nRemote = 0;
      for (int c = 0; c < L->num_my_boxes; c++) {
        int ci = L->my_boxes[c].low.i / L->box_dim, cj = L->my_boxes[c].low.j / L->box_dim, ck = L->my_boxes[c].low.k / L->box_dim;
        for (int bk = 0; bk < ratio_k; bk++)
        for (int bj = 0; bj < ratio_j; bj++)
        for (int bi = 0; bi < ratio_i; bi++) {
          int fid = box_id(Lf, ratio_i * ci + bi, ratio_j * cj + bj, ratio_k * ck + bk);
          if (Lf->rank_of_box[fid] == L->my_rank) continue;
          transfer_msg *m = &msg[nRemote];
          m->sendRank = Lf->rank_of_box[fid];   m->sendBoxID = fid;   m->sendBox = -1;
          m->recvRank = L->rank_of_box[L->my_boxes[c].global_box_id];
          m->recvBoxID = L->my_boxes[c].global_box_id;   m->recvBox = c;
          m->i = bi * Lf->box_dim / 2;  m->j = bj * Lf->box_dim / 2;  m->k = bk * Lf->box_dim / 2;
          ranks[nRemote++] = m->sendRank;
        }
      }
      qsort(msg, nRemote, sizeof(transfer_msg), cmp_transfer_msg);
      const int nRanks = sorted_unique(ranks, nRemote);
      int ei, ej, ek;
      restricted_extent(type, Lf->box_dim, &ei, &ej, &ek);
      const int elem = ei * ej * ek;

      C->num_recvs = nRanks;
      if (nRanks > 0) {
        alloc_neighbours(nRanks, &C->recv_ranks, &C->recv_sizes, &C->recv_buffers);
        double *bulk = (double *)hpgmg_rt_alloc_comm((size_t)nRemote * elem * sizeof(double));      /* peer-visible: senders store straight into it */
        for (int r = 0; r < nRanks; r++) {
          int offset = 0;
          C->recv_buffers[r] = bulk;
          for (int m = 0; m < nRemote; m++) if (msg[m].sendRank == ranks[r]) {
            const box_type *cb = &L->my_boxes[msg[m].recvBox];
            append_block_to_list(&C->blocks[2], &C->allocated_blocks[2], &C->num_blocks[2], ei, ej, ek,
                                 -1, C->recv_buffers[r], offset, 0, 0, ei, ei * ej, 1,
                                 msg[m].recvBox, NULL, msg[m].i, msg[m].j, msg[m].k, cb->jStride, cb->kStride, 1,
                                 BLOCKCOPY_TILE_I, BLOCKCOPY_TILE_J, BLOCKCOPY_TILE_K, 0);
            offset += elem;
          }
          C->recv_ranks[r] = ranks[r];
          C->recv_sizes[r] = offset;
          bulk += offset;
        }
      }
      free(msg);
      free(ranks);
    }
  }
}

/* ------------------------------------------------------------------------------------------ */
/* Interpolation program of every level (mg.c:181-475).  Stored on the COARSE level l for data
 * going to l-1: [0] interpolate my coarse regions into send buffers (already at fine
 * resolution), [1] interpolate into my own fine boxes; and on the FINE level: [2] add received
 * fine-resolution images into my boxes. */
static void build_interpolation(mg_type *MG)
{
  for (int l = 0; l < MG->num_levels; l++) {
    level_type *L = MG->levels[l];
    communicator_type *C = &L->interpolation;
    memset(C, 0, sizeof(*C));

    /* ---- coarse side: pack + local ---------------------------------------------------- */
    if (l > 0 && L->num_my_boxes > 0) {
      level_type *Lf = MG->levels[l - 1];
      const int ratio_i = Lf->boxes_in.i / L->boxes_in.i;
      const int ratio_j = Lf->boxes_in.j / L->boxes_in.j;
      const int ratio_k = Lf->boxes_in.k / L->boxes_in.k;
      const int cap = ratio_i * ratio_j * ratio_k * L->num_my_boxes;
      const int half = Lf->box_dim / 2;
      transfer_msg *msg = (transfer_msg *)malloc((size_t)cap * sizeof(transfer_msg));
      int *ranks = (int *)malloc((size_t)cap * sizeof(int));
      int nMsg = 0, nRemote = 0;
      for (int c = 0; c < L->num_my_boxes; c++) {
        int cid = L->my_boxes[c].global_box_id;
        int ci = L->my_boxes[c].low.i / L->box_dim, cj = L->my_boxes[c].low.j / L->box_dim, ck = L->my_boxes[c].low.k / L->box_dim;
        for (int bk = 0; bk < ratio_k; bk++)
        for (int bj = 0; bj < ratio_j; bj++)
        for (int bi = 0; bi < ratio_i; bi++) {
          int fid = box_id(Lf, ratio_i * ci + bi, ratio_j * cj + bj, ratio_k * ck + bk);
          transfer_msg *m = &msg[nMsg++];
          m->sendRank = L->rank_of_box[cid];     m->sendBoxID = cid;   m->sendBox = c;
          m->recvRank = Lf->rank_of_box[fid];    m->recvBoxID = fid;   m->recvBox = local_index_of_box(Lf, fid);
          m->i = bi * half;  m->j = bj * half;  m->k = bk * half;
          if (m->recvRank != L->my_rank) ranks[nRemote++] = m->recvRank;
        }
      }
      qsort(msg, nMsg, sizeof(transfer_msg), cmp_transfer_msg);
      const int nRanks = sorted_unique(ranks, nRemote);
      const int fdim = Lf->box_dim;
      const int elem = fdim * fdim * fdim;

      C->num_sends = nRanks;
      if (nRanks > 0) {
        alloc_neighbours(nRanks, &C->send_ranks, &C->send_sizes, &C->send_buffers);
        double *bulk = (double *)MALLOC((size_t)nRemote * elem * sizeof(double));   /* zeroed: 0.0*NaN hazard, mg.c:275 */
        for (int r = 0; r < nRanks; r++) {
          int offset = 0;
          C->send_buffers[r] = bulk;
          for (int m = 0; m < nMsg; m++) if (msg[m].recvRank == ranks[r]) {
            const box_type *cb = &L->my_boxes[msg[m].sendBox];
            append_block_to_list(&C->blocks[0], &C->allocated_blocks[0], &C->num_blocks[0], half, half, half,
                                 msg[m].sendBox, NULL, msg[m].i, msg[m].j, msg[m].k, cb->jStride, cb->kStride, 1,
                                 -1, C->send_buffers[r], offset, 0, 0, fdim, fdim * fdim, 2,
                                 BLOCKCOPY_TILE_I, BLOCKCOPY_TILE_J, BLOCKCOPY_TILE_K, 0);
            offset += elem;
          }
          C->send_ranks[r] = ranks[r];
          C->send_sizes[r] = offset;
          bulk += offset;
        }
      }
      for (int m = 0; m < nMsg; m++) if (msg[m].recvRank == MG->my_rank) {
        const box_type *cb = &L->my_boxes[msg[m].sendBox];
        const box_type *fb = &Lf->my_boxes[msg[m].recvBox];
        append_block_to_list(&C->blocks[1], &C->allocated_blocks[1], &C->num_blocks[1], half, half, half,
                             msg[m].sendBox, NULL, msg[m].i, msg[m].j, msg[m].k, cb->jStride, cb->kStride, 1,
                             msg[m].recvBox, NULL, 0, 0, 0, fb->jStride, fb->kStride, 2,
                             BLOCKCOPY_TILE_I, BLOCKCOPY_TILE_J, BLOCKCOPY_TILE_K, 0);
      }
      free(msg);
      free(ranks);
    }

    /* ---- fine side: unpack -------------------------------------------------------------- */
    if (l < MG->num_levels - 1 && L->num_my_boxes > 0) {
      level_type *Lc = MG->levels[l + 1];
      transfer_msg *msg = (transfer_msg *)malloc((size_t)L->num_my_boxes * sizeof(transfer_msg));
      int *ranks = (int *)malloc((size_t)L->num_my_boxes * sizeof(int));
      int nRemote = 0;
      for (int f = 0; f < L->num_my_boxes; f++) {
        int fid = L->my_boxes[f].global_box_id;
        int fi = L->my_boxes[f].low.i / L->box_dim, fj = L->my_boxes[f].low.j / L->box_dim, fk = L->my_boxes[f].low.k / L->box_dim;
        int cid = box_id(Lc, fi * Lc->boxes_in.i / L->boxes_in.i, fj * Lc->boxes_in.j / L->boxes_in.j, fk * Lc->boxes_in.k / L->boxes_in.k);
        if (Lc->rank_of_box[cid] == L->my_rank) continue;
        transfer_msg *m = &msg[nRemote];
        m->sendRank = Lc->rank_of_box[cid];   m->sendBoxID = cid;   m->sendBox = -1;
        m->recvRank = L->rank_of_box[fid];    m->recvBoxID = fid;   m->recvBox = f;
        m->i = m->j = m->k = 0;
        ranks[nRemote++] = m->sendRank;
      }
      qsort(msg, nRemote, sizeof(transfer_msg), cmp_transfer_msg);
      const int nRanks = sorted_unique(ranks, nRemote);
      const int dim = L->box_dim;
      const int elem = dim * dim * dim;

      C->num_recvs = nRanks;
      if (nRanks > 0) {
        alloc_neighbours(nRanks, &C->recv_ranks, &C->recv_sizes, &C->recv_buffers);
        double *bulk = (double *)hpgmg_rt_alloc_comm((size_t)nRemote * elem * sizeof(double));      /* peer-visible: senders store straight into it */
        for (int r = 0; r < nRanks; r++) {
          int offset = 0;
          C->recv_buffers[r] = bulk;
          for (int m = 0; m < nRemote; m++) if (msg[m].sendRank == ranks[r]) {
            const box_type *fb = &L->my_boxes[msg[m].recvBox];
            append_block_to_list(&C->blocks[2], &C->allocated_blocks[2], &C->num_blocks[2], dim, dim, dim,
                                 -1, C->recv_buffers[r], offset, 0, 0, dim, dim * dim, 1,
                                 msg[m].recvBox, NULL, 0, 0, 0, fb->jStride, fb->kStride, 1,
                                 BLOCKCOPY_TILE_I, BLOCKCOPY_TILE_J, BLOCKCOPY_TILE_K, 0);
            offset += elem;
          }
          C->recv_ranks[r] = ranks[r];
          C->recv_sizes[r] = offset;
          bulk += offset;
        }
      }
      free(msg);
      free(ranks);
    }
  }
}

/* ------------------------------------------------------------------------------------------ */
/* The level table: how dim / box size / box count / rank count evolve from one level to the
 * next.  Six rules tried in this order (mg.c:895-952):
 *   1 halve the boxes while they are bigger than MG_AGGLOMERATION_START
 *   2 merge 2x2x2 boxes into one (same box size, half the boxes per side)
 *   3..5 (domains whose side has an odd factor `odd`>1) collapse to one box / fewer ranks when the
 *        side reaches 2*odd, 4*odd, 8*odd
 *   6 halve the boxes on the same ranks
 * A box may never get smaller than the stencil radius. */
typedef struct { int nProcs, dim, boxes_in, box_dim, ghosts; } level_spec;

static int next_level_spec(const level_spec *f, int odd, int radius, level_spec *c)
{
  *c = *f;
  c->dim = f->dim / 2;
  if ((f->box_dim % 2 == 0) && (f->box_dim > MG_AGGLOMERATION_START) && (f->box_dim / 2 >= radius)) {
    c->box_dim = f->box_dim / 2;
  } else if ((f->boxes_in % 2 == 0) && (f->box_dim >= radius)) {
    c->boxes_in = f->boxes_in / 2;
  } else if ((odd != 1) && (f->dim == 2 * odd) && (f->dim / 2 >= radius)) {
    c->nProcs = 1;  c->box_dim = f->dim / 2;  c->boxes_in = 1;
  } else if ((odd != 1) && (f->dim == 4 * odd) && (f->box_dim / 2 >= radius)) {
    c->nProcs = odd < f->nProcs ? odd : f->nProcs;  c->box_dim = f->box_dim / 2;
  } else if ((odd != 1) && (f->dim == 8 * odd) && (f->box_dim / 2 >= radius)) {
    c->nProcs = odd * odd < f->nProcs ? odd * odd : f->nProcs;  c->box_dim = f->box_dim / 2;
  } else if ((f->box_dim % 2 == 0) && (f->box_dim / 2 >= radius)) {
    c->box_dim = f->box_dim / 2;
  } else {
    return 0;
  }
  return 1;
}

/* Ownership agglomeration (multi-GPU only).  The reference keeps a level spread over all ranks until its boxes merge
 * (rule 2) -- fine for CPUs, where a coarse-level ghost exchange costs a microsecond.  Between GPUs every exchange of a
 * level that is all latency costs an NVLink round trip, ~300 times per solve.  So levels whose boxes have at most
 * `g_agglomerate_box` cells per side, or that are at most 4 times that wide in total (64^3 cells: one GPU runs such a
 * level faster than several can exchange its halos), and every coarser level are OWNED by rank 0: the box structure -- and therefore
 * every bit of the result -- is unchanged, only rank_of_box differs; the transfers into and out of such a level are the
 * all-to-one / one-to-all messages the reference's own rank-shrinking rules (mg.c:918-941) already produce.
 * 0 reproduces the reference's decomposition exactly. */
static int g_agglomerate_box = -1;
void hpgmg_b200_set_agglomeration(int box_dim) { g_agglomerate_box = box_dim < 0 ? 0 : box_dim; }
int  hpgmg_b200_get_agglomeration(void)
{
  if (g_agglomerate_box < 0) {
    const char *e = getenv("HPGMG_B200_AGGLOMERATE_BOX");
    g_agglomerate_box = e ? atoi(e) : 16;
  }
  return g_agglomerate_box;
}

void MGBuild(mg_type *MG, level_type *fine, double a, double b, int minCoarseGridDim)
{
  const double t0 = hpgmg_rt_wtime();
  const int chatty = (fine->my_rank == 0) && hpgmg_rt_verbose();
  MG->my_rank = fine->my_rank;
  MG->timers.MGBuild = 0;
  MG->timers.MGSolve = 0;
  MG->MGSolves_performed = 0;

  /* depth allowed by the domain size alone, and the odd part of the domain side */
  int maxLevels = 1, odd = fine->dim.i;
  while ((odd >= 2 * minCoarseGridDim) && ((odd & 1) == 0)) { maxLevels++; odd /= 2; }
  if (maxLevels > 100) maxLevels = 100;

  level_spec spec[100];
  spec[0].nProcs = fine->num_ranks;   spec[0].dim = fine->dim.i;   spec[0].boxes_in = fine->boxes_in.i;
  spec[0].box_dim = fine->box_dim;    spec[0].ghosts = fine->box_ghosts;

  MG->levels = (level_type **)malloc((size_t)maxLevels * sizeof(level_type *));
  MG->levels[0] = fine;
  MG->num_levels = 1;
  while (MG->num_levels < maxLevels) {
    int l = MG->num_levels;
    if (!next_level_spec(&spec[l - 1], odd, stencil_get_radius(), &spec[l])) break;
    if (spec[l].dim < minCoarseGridDim) break;
    if (spec[l].nProcs > 1 && hpgmg_b200_get_agglomeration() > 0 &&
        (spec[l].box_dim <= hpgmg_b200_get_agglomeration() || spec[l].dim <= 4 * hpgmg_b200_get_agglomeration())) spec[l].nProcs = 1;   /* owned by rank 0 from here down */
    MG->num_levels++;
  }

  for (int l = 1; l < MG->num_levels; l++) {
    level_type *L = (level_type *)malloc(sizeof(level_type));
    int numVectors = MG->levels[l - 1]->numVectors;
    if (l == MG->num_levels - 1) numVectors += IterativeSolver_NumVectors();   /* Krylov vectors live on the bottom level */
    create_level(L, spec[l].boxes_in, spec[l].box_dim, spec[l].ghosts, numVectors,
                 MG->levels[l - 1]->boundary_condition.type, MG->levels[l - 1]->my_rank, spec[l].nProcs);
    L->h = 2.0 * MG->levels[l - 1]->h;
    MG->levels[l] = L;
  }

  if (chatty) { fprintf(stdout, "\n  Building restriction and interpolation lists... "); fflush(stdout); }
  build_restriction(MG, RESTRICT_CELL);
  build_restriction(MG, RESTRICT_FACE_I);
  build_restriction(MG, RESTRICT_FACE_J);
  build_restriction(MG, RESTRICT_FACE_K);
  build_interpolation(MG);
  for (int l = 0; l < MG->num_levels; l++) hpgmg_device_level_upload_transfer_lists(MG->levels[l]);
  for (int l = 0; l + 1 < MG->num_levels; l++) hpgmg_restriction_map_prepare(MG->levels[l], MG->levels[l + 1]);   /* residual fused with restriction (smooth.cu) */
  /* collective: swap buffer / flag addresses of every inter-level message (comm.cu) */
  for (int l = 0; l + 1 < MG->num_levels; l++) {
    for (int t = 0; t < 4; t++) hpgmg_comm_register_transfer(&MG->levels[l]->restriction[t], &MG->levels[l + 1]->restriction[t]);
    hpgmg_comm_register_transfer(&MG->levels[l + 1]->interpolation, &MG->levels[l]->interpolation);
  }
  if (chatty) { fprintf(stdout, "done\n"); fflush(stdout); }

  /* a rank is active on level l if it owns boxes there or on any coarser level (mg.c:985-986).
   * Inactive ranks skip the level entirely, including its reductions. */
  for (int l = 1; l < MG->num_levels; l++) {
    MG->levels[l]->active = 0;
    for (int ll = l; ll < MG->num_levels; ll++)
      if (MG->levels[ll]->num_my_boxes > 0) MG->levels[l]->active = 1;
  }

  if (chatty) fprintf(stdout, "\n");
  if (!hpgmg_rt_layout_only())        /* layout-only mode builds the lists but cannot run kernels */
    for (int l = 1; l < MG->num_levels; l++) rebuild_operator(MG->levels[l], MG->levels[l - 1], a, b);
  if (chatty) fprintf(stdout, "\n");

  for (int l = 0; l < MG->num_levels; l++) {
    level_type *L = MG->levels[l];
    /* Poisson-like with periodic BCs: the solution is only defined up to a constant (mg.c:1009-1018).  Without
     * VECTOR_ALPHA "alpha is zero" always holds. */
#ifdef VECTOR_ALPHA
    /* layout-only mode has no vector data to read: alpha counts as nonzero there */
    const int alpha_is_zero = !hpgmg_rt_layout_only() && (dot(L, VECTOR_ALPHA, VECTOR_ALPHA) == 0.0);
    L->must_subtract_mean = (L->boundary_condition.type == BC_PERIODIC && (a == 0 || alpha_is_zero)) ? 1 : 0;
#else
    L->must_subtract_mean = (L->boundary_condition.type == BC_PERIODIC) ? 1 : 0;
#endif
  }
  hpgmg_rt_sync();
  MG->timers.MGBuild += hpgmg_rt_wtime() - t0;
}

/* ------------------------------------------------------------------------------------------ */
static void hpgmg_forget_norms(const mg_type *MG);
static void hpgmg_pipe_drain(mg_type *MG);
void MGDestroy(mg_type *MG)
{
  const int chatty = (MG->my_rank == 0) && hpgmg_rt_verbose();
  hpgmg_pipe_drain(MG);                                 /* solves submitted with hpgmg_fmg_solve_host_submit and never waited for */
  hpgmg_rt_sync();
  hpgmg_graph_drop_all(MG);
  hpgmg_forget_norms(MG);
  if (chatty) { fprintf(stdout, "attempting to free the restriction and interpolation lists... "); fflush(stdout); }
  for (int l = MG->num_levels - 1; l >= 0; l--) {
    hpgmg_comm_unregister_transfer(&MG->levels[l]->interpolation);
    hpgmg_free_communicator(&MG->levels[l]->interpolation);
    for (int t = 3; t >= 0; t--) { hpgmg_comm_unregister_transfer(&MG->levels[l]->restriction[t]); hpgmg_free_communicator(&MG->levels[l]->restriction[t]); }
  }
  if (chatty) fprintf(stdout, "done\n");
  for (int l = MG->num_levels - 1; l > 0; l--) {       /* level 0 belongs to the caller */
    destroy_level(MG->levels[l]);
    free(MG->levels[l]);
  }
  free(MG->levels);
  MG->levels = NULL;
  MG->num_levels = 0;
}

void MGResetTimers(mg_type *MG)
{
  for (int l = 0; l < MG->num_levels; l++) reset_level_timers(MG->levels[l]);
  MG->timers.MGSolve = 0;
  MG->MGSolves_performed = 0;
}

/* ------------------------------------------------------------------------------------------ */
/* Richardson estimate of the discretisation error and the observed order (mg.c:1113-1131):
 * ||u^2h - R u^h|| and log2 of its ratio to the 4h/2h pair. */
static double g_last_error = 0.0, g_last_order = 0.0;
double hpgmg_last_richardson_error(void) { return g_last_error; }
double hpgmg_last_richardson_order(void) { return g_last_order; }

void richardson_error(mg_type *MG, int levelh, int u_id)
{
  level_type *Lh = MG->levels[levelh], *L2h = MG->levels[levelh + 1], *L4h = MG->levels[levelh + 2];
  restriction(L2h, VECTOR_TEMP, Lh,  u_id, RESTRICT_CELL);
  restriction(L4h, VECTOR_TEMP, L2h, u_id, RESTRICT_CELL);
  add_vectors(L2h, VECTOR_TEMP, 1.0, u_id, -1.0, VECTOR_TEMP);
  add_vectors(L4h, VECTOR_TEMP, 1.0, u_id, -1.0, VECTOR_TEMP);
  double e2h = norm(L2h, VECTOR_TEMP);
  double e4h = norm(L4h, VECTOR_TEMP);
  g_last_error = e2h;
  g_last_order = log(e4h / e2h) / log(2);
  if (MG->my_rank == 0 && hpgmg_rt_verbose()) {
    fprintf(stdout, "  h=%0.15e  ||error||=%0.15e\n", Lh->h, e2h);
    fprintf(stdout, "  order=%0.3f\n", g_last_order);
    fflush(stdout);
  }
}

/* ------------------------------------------------------------------------------------------ */
/* One V-cycle from `level` down to the bottom and back (mg.c:1135-1164). Enqueue-only. */
void MGVCycle(mg_type *MG, int e_id, int R_id, double a, double b, int level)
{
  level_type *L = MG->levels[level];
  if (!L->active) return;
  if (hpgmg_coarse_chain_eligible(MG, level)) {          /* small, rank-local levels: the whole sub-cycle is one kernel */
    hpgmg_coarse_cycle(MG, level, 0, 0, e_id, R_id, a, b);
    return;
  }
  if (level == MG->num_levels - 1) {
    IterativeSolver(L, e_id, R_id, a, b, MG_DEFAULT_BOTTOM_NORM);
    return;
  }
  level_type *Lc = MG->levels[level + 1];
  smooth(L, e_id, R_id, a, b);
  hpgmg_residual_then_restriction(Lc, R_id, L, VECTOR_TEMP, e_id, R_id, a, b);      /* residual(); restriction(): mg.c:1150-1151 */
  zero_vector(Lc, e_id);
  MGVCycle(MG, e_id, R_id, a, b, level + 1);
  interpolation_vcycle(L, e_id, 1.0, Lc, e_id);
  smooth(L, e_id, R_id, a, b);
}

/* ------------------------------------------------------------------------------------------ */
/* bookkeeping shared by the solve drivers */
/* ||F|| and ||r|| of the last solve, kept per hierarchy (the reference only prints them, mg.c:1325-1329) */
typedef struct { const mg_type *owner; double norm_of_F, norm_of_residual; } solve_norms;
#define MAX_TRACKED_HIERARCHIES 16
static solve_norms g_last[MAX_TRACKED_HIERARCHIES];
static int g_last_next = 0;
static solve_norms *last_norms_of(const mg_type *MG, int create)
{
  for (int i = 0; i < MAX_TRACKED_HIERARCHIES; i++) if (g_last[i].owner == MG) return &g_last[i];
  if (!create) return NULL;
  solve_norms *s = &g_last[g_last_next];              /* round robin: the oldest hierarchy's record is recycled */
  g_last_next = (g_last_next + 1) % MAX_TRACKED_HIERARCHIES;
  s->owner = MG;  s->norm_of_F = s->norm_of_residual = 0.0;
  return s;
}
static void record_norms(const mg_type *MG, double norm_of_F, double norm_of_residual)
{
  solve_norms *s = last_norms_of(MG, 1);
  s->norm_of_F = norm_of_F;  s->norm_of_residual = norm_of_residual;
}
double hpgmg_last_norm_of_F(const mg_type *MG)        { const solve_norms *s = last_norms_of(MG, 0); return s ? s->norm_of_F : 0.0; }
double hpgmg_last_norm_of_residual(const mg_type *MG) { const solve_norms *s = last_norms_of(MG, 0); return s ? s->norm_of_residual : 0.0; }

/* Can a whole solve on this hierarchy be recorded into a CUDA graph?  Only if nothing in it needs a host
 * read-back: no mean subtraction (periodic), no per-operator timers, and a bottom solve that runs as one
 * device kernel (single-block coarse cycle or single-block BiCGStab) -- the host-driven BiCGStab of
 * solvers.c synchronises on every dot / norm. */
int hpgmg_bicgstab_device_eligible(const level_type *level);      /* bicgstab.cu */
static int solve_is_capturable(mg_type *MG, const level_type *L)
{
  if (!hpgmg_rt_use_graphs() || hpgmg_rt_profile() || L->must_subtract_mean == 1) return 0;
  const int bottom = MG->num_levels - 1;
  const level_type *B = MG->levels[bottom];
  if (!B->active) return 1;                            /* this rank never touches the bottom level */
  return hpgmg_coarse_chain_eligible(MG, bottom) || hpgmg_bicgstab_device_eligible(B);
}

/* the bottom solver counts its iterations on the device (HPGMG_SLOT_KRYLOV); every driver zeroes the slot
 * before enqueueing cycles and adds it to the bottom level's counter when it next synchronises */
static void hpgmg_forget_norms(const mg_type *MG) { solve_norms *s = last_norms_of(MG, 0); if (s) s->owner = NULL; }
static void krylov_count_begin(void) { hpgmg_rt_zero_scalar(HPGMG_SLOT_KRYLOV); }
static void krylov_count_collect(mg_type *MG)
{
  double its = 0.0;
  hpgmg_rt_read_scalars(&its, HPGMG_SLOT_KRYLOV, 1);
  MG->levels[MG->num_levels - 1]->Krylov_iterations += (int)its;
  hpgmg_rt_zero_scalar(HPGMG_SLOT_KRYLOV);
}

static int g_fmg_post_vcycles = 0;     /* the reference's -DUNLIMIT_FMG_ITERATIONS => 20 (mg.c:1243-1247) */
void hpgmg_b200_set_fmg_post_vcycles(int n) { g_fmg_post_vcycles = n; }

static long long solve_key(int kind, int onLevel, int u_id, int F_id, double a, double b)
{
  long long k = kind;
  k = k * 131 + onLevel;  k = k * 131 + u_id;  k = k * 131 + F_id;  k = k * 131 + hpgmg_rt_smoother();
  k = k * 7 + hpgmg_rt_bottom_solver();                        /* a graph recorded under one bottom solver never replays under another */
  unsigned long long ua, ub;
  memcpy(&ua, &a, 8);  memcpy(&ub, &b, 8);
  k ^= (long long)(ua * 0x9E3779B97F4A7C15ull) ^ (long long)(ub * 0xC2B2AE3D27D4EB4Full);
  return k;
}

/* counters that the reference bumps on the host while it runs the cycle; a replayed graph does
 * not execute host code, so they are applied once per solve from these per-level increments */
static void count_vcycle_visits(mg_type *MG, int onLevel)
{
  for (int l = MG->num_levels - 2; l >= onLevel; l--) MG->levels[l]->vcycles_from_this_level++;
}

/* residual + max-norm of the current iterate, result left in scalar slot NORM_R (mg.c:1316-1322) */
static void enqueue_residual_norm(level_type *L, int e_id, int F_id, double a, double b)
{
  if (L->must_subtract_mean == 1) {
    double average = mean(L, e_id);                     /* synchronises: periodic problems are not graph-captured */
    shift_vector(L, e_id, e_id, -average);
  }
  hpgmg_residual_norm_async(L, VECTOR_TEMP, e_id, F_id, a, b, HPGMG_SLOT_NORM_R);
}

/* ------------------------------------------------------------------------------------------ */
/* One F-cycle (mg.c:1237-1344): ||F||, R=F, restrict R to the bottom, bottom solve, then for
 * every level going up: 4th-order interpolation of the coarse solution as initial guess followed
 * by one V-cycle.  Solves in place (e_id == u_id). */
static void enqueue_fcycle_after_rhs(mg_type *MG, int onLevel, int e_id, int R_id, double a, double b);
static void enqueue_fcycle(mg_type *MG, int onLevel, int e_id, int R_id, int F_id, double a, double b)
{
  hpgmg_copy_norm_async(MG->levels[onLevel], R_id, F_id, HPGMG_SLOT_NORM_F);      /* ||F|| and R = F (mg.c:1265-1269) */
  enqueue_fcycle_after_rhs(MG, onLevel, e_id, R_id, a, b);
}
static void enqueue_fcycle_after_rhs(mg_type *MG, int onLevel, int e_id, int R_id, double a, double b)
{
  for (int l = onLevel; l < MG->num_levels - 1; l++)
    restriction(MG->levels[l + 1], R_id, MG->levels[l], R_id, RESTRICT_CELL);
  int bottom = MG->num_levels - 1;
  /* the finest level from which everything down to the bottom can run in the single-block kernel */
  int coarse_from = MG->num_levels;
  for (int l = bottom; l >= onLevel && MG->levels[l]->active && hpgmg_coarse_chain_eligible(MG, l); l--) coarse_from = l;
  int next = MG->num_levels - 2;
  if (coarse_from <= bottom) {
    /* zero(e_bottom); bottom solve; interpolation_fcycle + MGVCycle for l = bottom-1..coarse_from */
    hpgmg_coarse_cycle(MG, coarse_from, 1, bottom > onLevel, e_id, R_id, a, b);
    next = coarse_from - 1;
  } else {
    if (bottom > onLevel) zero_vector(MG->levels[bottom], e_id);
    IterativeSolver(MG->levels[bottom], e_id, R_id, a, b, MG_DEFAULT_BOTTOM_NORM);
  }
  for (int l = next; l >= onLevel; l--) {
    interpolation_fcycle(MG->levels[l], e_id, 0.0, MG->levels[l + 1], e_id);
    MGVCycle(MG, e_id, R_id, a, b, l);
  }
}

void FMGSolve(mg_type *MG, int onLevel, int u_id, int F_id, double a, double b, double rtol)
{
  MG->MGSolves_performed++;
  level_type *L = MG->levels[onLevel];
  if (!L->active) return;
  const int e_id = u_id, R_id = VECTOR_R;
  const int chatty = (L->my_rank == 0) && hpgmg_rt_verbose();
  if (chatty) fprintf(stdout, "FMGSolve... ");
  const double t0 = hpgmg_rt_wtime();

  const int capturable = solve_is_capturable(MG, L);
  const long long key = solve_key(1, onLevel, u_id, F_id, a, b);
  hpgmg_rt_timer_start();
  if (!capturable || hpgmg_graph_begin(MG, key)) {
    hpgmg_rt_zero_scalar(HPGMG_SLOT_KRYLOV);
    enqueue_fcycle(MG, onLevel, e_id, R_id, F_id, a, b);
    enqueue_residual_norm(L, e_id, F_id, a, b);
    if (capturable) hpgmg_graph_end(MG, key);
  }
  hpgmg_rt_timer_stop();
  count_vcycle_visits(MG, onLevel);

  double s[3];
  hpgmg_rt_read_scalars(s, HPGMG_SLOT_NORM_F, 3);         /* the solve's only synchronisation */
  double norm_of_F = s[0], norm_of_residual = s[1];
  MG->levels[MG->num_levels - 1]->Krylov_iterations += (int)s[2];   /* counted on the device by the bottom solver */
  if (chatty) fprintf(stdout, "f-cycle     norm=%1.15e  rel=%1.15e  ", norm_of_residual, norm_of_residual / norm_of_F);

  /* optional post-F V-cycles until converged (UNLIMIT_FMG_ITERATIONS) */
  for (int v = 0; v < g_fmg_post_vcycles && !(norm_of_residual / norm_of_F < rtol); v++) {
    L->vcycles_from_this_level++;
    const long long vkey = solve_key(2, onLevel, u_id, F_id, a, b);
    if (!capturable || hpgmg_graph_begin(MG, vkey)) {
      hpgmg_rt_zero_scalar(HPGMG_SLOT_KRYLOV);
      MGVCycle(MG, e_id, R_id, a, b, onLevel);
      enqueue_residual_norm(L, e_id, F_id, a, b);
      if (capturable) hpgmg_graph_end(MG, vkey);
    }
    hpgmg_rt_read_scalars(s, HPGMG_SLOT_NORM_R, 2);
    norm_of_residual = s[0];
    MG->levels[MG->num_levels - 1]->Krylov_iterations += (int)s[1];
    if (chatty) fprintf(stdout, "\n            v-cycle=%2d  norm=%1.15e  rel=%1.15e  ", v + 1, norm_of_residual, norm_of_residual / norm_of_F);
  }

  record_norms(MG, norm_of_F, norm_of_residual);
  const double dt = hpgmg_rt_wtime() - t0;
  MG->timers.MGSolve += dt;
  if (chatty) fprintf(stdout, "done (%f seconds)\n", dt);
}

/* ------------------------------------------------------------------------------------------ */
/* FMGSolve with HOST buffers -- the end-to-end call (bench.py's e2e): f_host and u_host hold the CELLS of this rank's boxes,
 * dense, box-major, [k][j][i] per box.  One recorded graph does: upload f into a staging buffer; unpack it into F fused
 * with the first step of FMGSolve (||F||, R = F); zero u; the F-cycle; then the download of u (pack kernel + copy on a
 * side stream) OVERLAPPED with the final residual and its norm on the compute stream.  Returns the F-cycle residual norm. */
static long long hash_pointer(const void *p) { return (long long)((unsigned long long)(size_t)p * 0x9E3779B97F4A7C15ull); }
unsigned long long hpgmg_fmg_solve_host_bytes(mg_type *MG, int onLevel)
{
  const level_type *L = MG->levels[onLevel];
  return (unsigned long long)L->num_my_boxes * L->box_dim * L->box_dim * L->box_dim * sizeof(double);
}
double hpgmg_fmg_solve_host(mg_type *MG, int onLevel, int u_id, int F_id, double a, double b, double rtol, const double *f_host, double *u_host)
{
  (void)rtol;
  level_type *L = MG->levels[onLevel];
  const size_t bytes = (size_t)hpgmg_fmg_solve_host_bytes(MG, onLevel);
  if ((L->box_dim & 1) || !L->active) {                 /* odd boxes: no 16-byte pairs; plain path */
    fprintf(stderr, "hpgmg_fmg_solve_host: needs an even box size and an active level\n");
    exit(1);
  }
  MG->MGSolves_performed++;
  const int e_id = u_id, R_id = VECTOR_R;
  double *stage_f = bytes ? (double *)hpgmg_rt_staging(0, bytes) : NULL;       /* (re)allocated before any recording starts */
  double *stage_u = bytes ? (double *)hpgmg_rt_staging(1, bytes) : NULL;
  const int capturable = solve_is_capturable(MG, L);
  const long long key = solve_key(7, onLevel, u_id, F_id, a, b) ^ hash_pointer(f_host) ^ (hash_pointer(u_host) << 1);
  hpgmg_rt_timer_start();
  if (!capturable || hpgmg_graph_begin(MG, key)) {
    if (bytes) hpgmg_rt_copy_h2d(stage_f, f_host, bytes);
    hpgmg_rt_zero_scalar(HPGMG_SLOT_KRYLOV);
    zero_vector(L, u_id);                                                        /* hpgmg-fv.c:78 */
    hpgmg_unpack_copy_norm_async(L, F_id, R_id, stage_f, HPGMG_SLOT_NORM_F);
    enqueue_fcycle_after_rhs(MG, onLevel, e_id, R_id, a, b);
    if (L->must_subtract_mean == 1) {                                            /* periodic: the mean is removed from u first (mg.c:1317-1320) */
      enqueue_residual_norm(L, e_id, F_id, a, b);
      hpgmg_pack_async(L, u_id, stage_u);
      if (bytes) hpgmg_rt_copy_d2h(u_host, stage_u, bytes);
    } else {
      hpgmg_rt_side_begin();                                                     /* u is final: download it ... */
      hpgmg_pack_async(L, u_id, stage_u);
      if (bytes) hpgmg_rt_copy_d2h(u_host, stage_u, bytes);
      hpgmg_rt_side_end();
      enqueue_residual_norm(L, e_id, F_id, a, b);                                /* ... while the residual and its norm are computed */
      hpgmg_rt_side_join();
    }
    if (capturable) hpgmg_graph_end(MG, key);
  }
  hpgmg_rt_timer_stop();
  count_vcycle_visits(MG, onLevel);
  double s[3];
  hpgmg_rt_read_scalars(s, HPGMG_SLOT_NORM_F, 3);
  MG->levels[MG->num_levels - 1]->Krylov_iterations += (int)s[2];
  record_norms(MG, s[0], s[1]);
  return s[1];
}

/* ------------------------------------------------------------------------------------------ */
/* The end-to-end solve with DEVICE arrays of the whole domain (include/hpgmg_b200.h).  The caller's arrays are read and written by
 * plain launches around the recorded solve -- unpack f into F fused with ||F|| and R = F, then [zero u, the F-cycle, the residual
 * norm], then pack u -- so the recording is keyed by the hierarchy and the solve's parameters, not by the arrays' addresses: a
 * program that hands in a new tensor every call replays one graph.  Same kernels and order as hpgmg_fmg_solve_host, same bits. */
double hpgmg_fmg_solve_device(mg_type *MG, int onLevel, int u_id, int F_id, double a, double b, double rtol, const double *f_dev, double *u_dev, void *stream)
{
  (void)rtol;
  level_type *L = MG->levels[onLevel];
  if ((L->box_dim & 1) || !L->active) {
    fprintf(stderr, "hpgmg_fmg_solve_device: needs an even box size and an active level\n");
    exit(1);
  }
  hpgmg_rt_check_device_array("hpgmg_fmg_solve_device", "f_dev", f_dev);
  hpgmg_rt_check_device_array("hpgmg_fmg_solve_device", "u_dev", u_dev);
  MG->MGSolves_performed++;
  const int e_id = u_id, R_id = VECTOR_R;
  const int capturable = solve_is_capturable(MG, L);
  const long long key = solve_key(4, onLevel, u_id, F_id, a, b);
  hpgmg_rt_wait_for_stream(stream);                                              /* f is complete */
  hpgmg_rt_timer_start();
  hpgmg_grid_unpack_copy_norm_async(L, F_id, R_id, f_dev, HPGMG_SLOT_NORM_F);
  if (!capturable || hpgmg_graph_begin(MG, key)) {
    hpgmg_rt_zero_scalar(HPGMG_SLOT_KRYLOV);
    zero_vector(L, u_id);                                                        /* hpgmg-fv.c:78 */
    enqueue_fcycle_after_rhs(MG, onLevel, e_id, R_id, a, b);
    enqueue_residual_norm(L, e_id, F_id, a, b);                                  /* periodic: removes the mean from u first */
    if (capturable) hpgmg_graph_end(MG, key);
  }
  hpgmg_grid_pack_async(L, u_id, u_dev);
  hpgmg_rt_timer_stop();
  count_vcycle_visits(MG, onLevel);
  double s[3];
  hpgmg_rt_read_scalars(s, HPGMG_SLOT_NORM_F, 3);                                /* u is written */
  MG->levels[MG->num_levels - 1]->Krylov_iterations += (int)s[2];
  record_norms(MG, s[0], s[1]);
  return s[1];
}

/* ------------------------------------------------------------------------------------------ */
/* The same end-to-end solve, PIPELINED for back-to-back solves: submit() enqueues upload, solve and download of one solve
 * and returns at once; wait() blocks until that solve's u_host and norms are complete.  Two solves may be in flight: while
 * solve n computes, f of solve n+1 travels up and u of solve n-1 travels down on their own streams (PCIe is full duplex),
 * so a stream of solves runs at max(compute, upload, download) per solve instead of their sum.  Each slot owns its staging
 * buffers; the caller must not touch f_host / u_host of a submitted solve before wait() returns, and submits at most two
 * solves before waiting for the older one.  Results are bit-identical to hpgmg_fmg_solve_host. */
typedef struct { mg_type *MG; int onLevel, busy; } pipe_slot;
static pipe_slot g_pipe[2];
static int g_pipe_next = 0;
int hpgmg_fmg_solve_host_submit(mg_type *MG, int onLevel, int u_id, int F_id, double a, double b, double rtol, const double *f_host, double *u_host)
{
  (void)rtol;
  level_type *L = MG->levels[onLevel];
  const size_t bytes = (size_t)hpgmg_fmg_solve_host_bytes(MG, onLevel);
  if ((L->box_dim & 1) || !L->active) {
    fprintf(stderr, "hpgmg_fmg_solve_host_submit: needs an even box size and an active level\n");
    exit(1);
  }
  const int slot = g_pipe_next;
  if (g_pipe[slot].busy) {
    fprintf(stderr, "hpgmg_fmg_solve_host_submit: two solves are already in flight; wait for ticket %d first\n", slot);
    exit(1);
  }
  g_pipe_next ^= 1;
  g_pipe[slot].MG = MG;  g_pipe[slot].onLevel = onLevel;  g_pipe[slot].busy = 1;
  MG->MGSolves_performed++;
  const int e_id = u_id, R_id = VECTOR_R;
  double *stage_f = bytes ? (double *)hpgmg_rt_staging(2 * slot, bytes) : NULL;
  double *stage_u = bytes ? (double *)hpgmg_rt_staging(2 * slot + 1, bytes) : NULL;
  const int capturable = solve_is_capturable(MG, L);
  hpgmg_rt_pipe_upload(slot, stage_f, f_host, bytes);                            /* upload stream; the compute stream waits for it */
  const long long key = solve_key(8 + slot, onLevel, u_id, F_id, a, b);
  if (!capturable || hpgmg_graph_begin(MG, key)) {
    hpgmg_rt_zero_scalar(HPGMG_SLOT_KRYLOV);
    zero_vector(L, u_id);                                                        /* hpgmg-fv.c:78 */
    hpgmg_unpack_copy_norm_async(L, F_id, R_id, stage_f, HPGMG_SLOT_NORM_F);
    enqueue_fcycle_after_rhs(MG, onLevel, e_id, R_id, a, b);
    if (L->must_subtract_mean != 1) hpgmg_pack_async(L, u_id, stage_u);          /* u is final */
    if (capturable) hpgmg_graph_end(MG, key);
  }
  if (L->must_subtract_mean == 1) {                                              /* periodic: the mean is removed from u first (mg.c:1317-1320) */
    enqueue_residual_norm(L, e_id, F_id, a, b);
    hpgmg_pack_async(L, u_id, stage_u);
    hpgmg_rt_pipe_download(slot, u_host, stage_u, bytes);
  } else {
    hpgmg_rt_pipe_download(slot, u_host, stage_u, bytes);                        /* download stream ... */
    enqueue_residual_norm(L, e_id, F_id, a, b);                                  /* ... while the residual and its norm are computed */
  }
  hpgmg_rt_pipe_scalars(slot);
  count_vcycle_visits(MG, onLevel);
  return slot;
}
static void hpgmg_pipe_drain(mg_type *MG)
{
  for (int t = 0; t < 2; t++)
    if (g_pipe[t].busy && g_pipe[t].MG == MG) { double s[3]; hpgmg_rt_pipe_wait(t, s); g_pipe[t].busy = 0; g_pipe[t].MG = NULL; }
}
double hpgmg_fmg_solve_host_wait(mg_type *MG, int ticket)
{
  if (ticket < 0 || ticket > 1 || !g_pipe[ticket].busy || g_pipe[ticket].MG != MG) {
    fprintf(stderr, "hpgmg_fmg_solve_host_wait: ticket %d is not an outstanding solve of this hierarchy\n", ticket);
    exit(1);
  }
  double s[3];
  hpgmg_rt_pipe_wait(ticket, s);
  g_pipe[ticket].busy = 0;
  MG->levels[MG->num_levels - 1]->Krylov_iterations += (int)s[2];
  record_norms(MG, s[0], s[1]);
  return s[1];
}

/* ------------------------------------------------------------------------------------------ */
/* V-cycles to convergence from a zero initial guess (mg.c:1168-1233). */
void MGSolve(mg_type *MG, int onLevel, int u_id, int F_id, double a, double b, double rtol)
{
  MG->MGSolves_performed++;
  level_type *L = MG->levels[onLevel];
  if (!L->active) return;
  const int e_id = u_id, R_id = VECTOR_R, maxVCycles = 20;
  const int chatty = (L->my_rank == 0) && hpgmg_rt_verbose();
  if (chatty) fprintf(stdout, "MGSolve... ");
  const double t0 = hpgmg_rt_wtime();
  const int capturable = solve_is_capturable(MG, L);

  hpgmg_rt_timer_start();
  hpgmg_norm_async(L, F_id, HPGMG_SLOT_NORM_F);
  zero_vector(L, e_id);
  scale_vector(L, R_id, 1.0, F_id);
  double s[3] = { 1.0, 0.0, 0.0 };
  for (int v = 0; v < maxVCycles; v++) {
    L->vcycles_from_this_level++;
    const long long key = solve_key(3, onLevel, u_id, F_id, a, b);
    if (!capturable || hpgmg_graph_begin(MG, key)) {
      hpgmg_rt_zero_scalar(HPGMG_SLOT_KRYLOV);
      MGVCycle(MG, e_id, R_id, a, b, onLevel);
      enqueue_residual_norm(L, e_id, F_id, a, b);
      if (capturable) hpgmg_graph_end(MG, key);
    }
    hpgmg_rt_read_scalars(s, HPGMG_SLOT_NORM_F, 3);
    MG->levels[MG->num_levels - 1]->Krylov_iterations += (int)s[2];
    if (chatty) fprintf(stdout, v > 0 ? "\n           v-cycle=%2d  norm=%1.15e  rel=%1.15e  " : "v-cycle=%2d  norm=%1.15e  rel=%1.15e  ",
                        v + 1, s[1], s[1] / s[0]);
    if (s[1] / s[0] < rtol) break;
  }
  hpgmg_rt_timer_stop();
  record_norms(MG, s[0], s[1]);
  const double dt = hpgmg_rt_wtime() - t0;
  MG->timers.MGSolve += dt;
  if (chatty) fprintf(stdout, "done (%f seconds)\n", dt);
}

/* ------------------------------------------------------------------------------------------ */
/* F-cycles in residual-correction form (mg.c:1348-1495): R = F - A u, solve A e = R with an
 * F-cycle, u += e, repeat until converged (at most 20 F-cycles, then maxVCycles V-cycles = 0). */
void FMGSolve2(mg_type *MG, int onLevel, int u_id, int F_id, double a, double b, double rtol)
{
  MG->MGSolves_performed++;
  level_type *L = MG->levels[onLevel];
  if (!L->active) return;
  const int e_id = VECTOR_E, R_id = VECTOR_R;
  int maxFCycles = 20;
  const int chatty = (L->my_rank == 0) && hpgmg_rt_verbose();
  if (chatty) fprintf(stdout, "FMGSolve... ");
  const double t0 = hpgmg_rt_wtime();

  hpgmg_rt_timer_start();
  krylov_count_begin();
  residual(L, R_id, u_id, F_id, a, b);
  double norm_of_residual = norm(L, R_id);
  double norm_of_F = norm(L, F_id);
  if (chatty) fprintf(stdout, "            norm=%1.15e  rel=%1.15e\n", norm_of_residual, norm_of_residual / norm_of_F);
  if (norm_of_residual / norm_of_F < rtol) maxFCycles = 0;

  for (int f = 0; f < maxFCycles; f++) {
    for (int l = onLevel; l < MG->num_levels - 1; l++)
      restriction(MG->levels[l + 1], R_id, MG->levels[l], R_id, RESTRICT_CELL);
    int bottom = MG->num_levels - 1;
    if (bottom > onLevel) zero_vector(MG->levels[bottom], e_id);
    IterativeSolver(MG->levels[bottom], e_id, R_id, a, b, MG_DEFAULT_BOTTOM_NORM);
    for (int l = MG->num_levels - 2; l >= onLevel; l--) {
      interpolation_fcycle(MG->levels[l], e_id, 0.0, MG->levels[l + 1], e_id);
      MG->levels[l]->vcycles_from_this_level++;
      MGVCycle(MG, e_id, R_id, a, b, l);
    }
    add_vectors(L, u_id, 1.0, u_id, 1.0, e_id);
    if (L->must_subtract_mean == 1) {
      double average = mean(L, u_id);
      shift_vector(L, u_id, u_id, -average);
    }
    residual(L, R_id, u_id, F_id, a, b);
    norm_of_residual = norm(L, R_id);
    krylov_count_collect(MG);
    if (chatty) fprintf(stdout, "            f-cycle=%2d  norm=%1.15e  rel=%1.15e\n", f + 1, norm_of_residual, norm_of_residual / norm_of_F);
    if (norm_of_residual / norm_of_F < rtol) break;
  }
  hpgmg_rt_timer_stop();
  record_norms(MG, norm_of_F, norm_of_residual);
  const double dt = hpgmg_rt_wtime() - t0;
  MG->timers.MGSolve += dt;
  if (chatty) fprintf(stdout, "            done (%f seconds)\n\n", dt);
}

/* ------------------------------------------------------------------------------------------ */
/* Conjugate gradients preconditioned by one V-cycle (mg.c:1500-1607; Saad alg. 9.1). */
void MGPCG(mg_type *MG, int onLevel, int x_id, int F_id, double a, double b, double rtol)
{
  level_type *L = MG->levels[onLevel];
  if (!L->active) return;
  for (int l = 0; l < MG->num_levels; l++) create_vectors(MG->levels[l], VECTORS_RESERVED + 3);
  const int r_id = VECTOR_R, p_id = VECTORS_RESERVED + 0, Ap_id = VECTORS_RESERVED + 1, z_id = VECTORS_RESERVED + 2;
  const int chatty = (L->my_rank == 0) && hpgmg_rt_verbose();
  if (chatty) fprintf(stdout, "MGPCG...  ");
  const double t0 = hpgmg_rt_wtime();
  MG->MGSolves_performed++;
  const int jMax = 20;
  int j = 0, failed = 0, converged = 0;

  krylov_count_begin();
  zero_vector(L, x_id);
  residual(L, r_id, x_id, F_id, a, b);
  if (L->must_subtract_mean == 1) { double m = mean(L, r_id); shift_vector(L, r_id, r_id, -m); }
  double norm_of_r0 = norm(L, r_id), norm_of_r = norm_of_r0;
  if (norm_of_r0 == 0.0) converged = 1;
  L->vcycles_from_this_level++;
  zero_vector(L, z_id);
  MGVCycle(MG, z_id, r_id, a, b, onLevel);
  scale_vector(L, p_id, 1.0, z_id);
  double r_dot_z = dot(L, r_id, z_id);
  while (j < jMax && !failed && !converged) {
    j++;  L->Krylov_iterations++;
    apply_op(L, Ap_id, p_id, a, b);
    double Ap_dot_p = dot(L, Ap_id, p_id);
    if (Ap_dot_p == 0.0) { failed = 1; break; }
    double alpha = r_dot_z / Ap_dot_p;
    if (isinf(alpha)) { failed = 1; break; }
    add_vectors(L, x_id, 1.0, x_id,  alpha, p_id);
    add_vectors(L, r_id, 1.0, r_id, -alpha, Ap_id);
    if (L->must_subtract_mean == 1) { double m = mean(L, r_id); shift_vector(L, r_id, r_id, -m); }
    residual(L, VECTOR_TEMP, x_id, F_id, a, b);
    norm_of_r = norm(L, VECTOR_TEMP);
    if (norm_of_r == 0.0) { converged = 1; break; }
    if (chatty) {
      if (j > 1) fprintf(stdout, "\n          ");
      fprintf(stdout, "iter=%3d  norm=%1.15e  rel=%1.15e  ", j, norm_of_r, norm_of_r / norm_of_r0);
    }
    if (norm_of_r / norm_of_r0 < rtol) break;
    L->vcycles_from_this_level++;
    zero_vector(L, z_id);
    MGVCycle(MG, z_id, r_id, a, b, onLevel);
    double r_dot_z_new = dot(L, r_id, z_id);
    if (r_dot_z_new == 0.0) { failed = 1; break; }
    double beta = r_dot_z_new / r_dot_z;
    if (isinf(beta)) { failed = 1; break; }
    add_vectors(L, p_id, 1.0, z_id, beta, p_id);
    r_dot_z = r_dot_z_new;
  }
  krylov_count_collect(MG);
  record_norms(MG, norm_of_r0, norm_of_r);
  const double dt = hpgmg_rt_wtime() - t0;
  MG->timers.MGSolve += dt;
  if (chatty) fprintf(stdout, "done (%f seconds)\n", dt);
}

/* ------------------------------------------------------------------------------------------ */
/* Per-level, per-operator-class table of average seconds per solve (mg.c:54-161).  The level
 * timers are only filled in when hpgmg_b200_profile_operators(1) is on (each operator is then
 * bracketed by CUDA events); otherwise only the totals at the bottom are meaningful. */
static void timing_row(const char *label, mg_type *MG, int from, double scale, size_t field_offset)
{
  double total = 0;
  printf("%-26s", label);
  for (int l = from; l < MG->num_levels; l++) {
    double t = scale * *(double *)((char *)&MG->levels[l]->timers + field_offset);
    total += t;
    printf("%12.6f ", t);
  }
  printf("%12.6f\n", total);
}

void MGPrintTiming(mg_type *MG, int fromLevel)
{
  if (MG->my_rank != 0) return;
  const int n = MG->num_levels;
  const double scale = 1.0 / (double)(MG->MGSolves_performed > 0 ? MG->MGSolves_performed : 1);
  typedef level_type LT;
  printf("\n\n");
  printf("level                     "); for (int l = fromLevel; l < n; l++) printf("%12d ", l - fromLevel); printf("\n");
  printf("level dimension           "); for (int l = fromLevel; l < n; l++) printf("%10d^3 ", MG->levels[l]->dim.i); printf("\n");
  printf("box dimension             "); for (int l = fromLevel; l < n; l++) printf("%10d^3 ", MG->levels[l]->box_dim); printf("       total\n");
  printf("------------------        "); for (int l = fromLevel; l < n + 1; l++) printf("------------ "); printf("\n");
#define ROW(label, f) timing_row(label, MG, fromLevel, scale, offsetof(LT, timers.f) - offsetof(LT, timers))
  ROW("smooth", smooth);
  ROW("residual", residual);
  ROW("applyOp", apply_op);
  ROW("BLAS1", blas1);
  ROW("BLAS3", blas3);
  ROW("Boundary Conditions", boundary_conditions);
  ROW("Restriction", restriction_total);
  ROW("  local restriction", restriction_local);
  ROW("  pack peer buffers", restriction_pack);
  ROW("  unpack peer buffers", restriction_unpack);
  ROW("Interpolation", interpolation_total);
  ROW("  local interpolation", interpolation_local);
  ROW("  pack peer buffers", interpolation_pack);
  ROW("  unpack peer buffers", interpolation_unpack);
  ROW("Ghost Zone Exchange", ghostZone_total);
  ROW("  local exchange", ghostZone_local);
  ROW("  pack peer buffers", ghostZone_pack);
  ROW("  unpack peer buffers", ghostZone_unpack);
  ROW("  wait for peers", ghostZone_wait);
  ROW("collectives", collectives);
  printf("------------------        "); for (int l = fromLevel; l < n + 1; l++) printf("------------ "); printf("\n");
  ROW("Total by level", Total);
#undef ROW
  printf("\n");
  printf("   Total time in MGBuild  %12.6f seconds\n", MG->timers.MGBuild);
  printf("   Total time in MGSolve  %12.6f seconds\n", scale * MG->timers.MGSolve);
  printf("      number of v-cycles  %12d\n", MG->levels[fromLevel]->vcycles_from_this_level / (MG->MGSolves_performed > 0 ? MG->MGSolves_performed : 1));
  printf("Bottom solver iterations  %12d\n", MG->levels[n - 1]->Krylov_iterations / (MG->MGSolves_performed > 0 ? MG->MGSolves_performed : 1));
  printf("\n\n");
  fflush(stdout);
}
