/*
 * device_level.cu -- the device mirror of a level: DLevel (slab geometry) and device copies of the
 * block lists the host built in level.c / mg.c (the same blockCopy_type records the reference
 * walks with OpenMP: level.c:367-465 BCs, :498-922 ghost exchange, mg.c:181-831 transfers).
 */
#include <string.h>
#include <vector>
#include <algorithm>
#include "common.cuh"
#include "stencil.cuh"

static void upload_list(DList *dst, const blockCopy_type *src, int n)
{
  if (dst->blocks && !hpgmg_rt_layout_only()) { CUDA_CHECK(cudaStreamSynchronize(g_stream)); CUDA_CHECK(cudaFree(dst->blocks)); }
  dst->blocks = NULL;
  dst->n = n;
  if (n <= 0 || hpgmg_rt_layout_only()) return;
  CUDA_CHECK(cudaMalloc(&dst->blocks, (size_t)n * sizeof(blockCopy_type)));
  CUDA_CHECK(cudaMemcpyAsync(dst->blocks, src, (size_t)n * sizeof(blockCopy_type), cudaMemcpyHostToDevice, g_stream));
  CUDA_CHECK(cudaStreamSynchronize(g_stream));
}

static void free_list(DList *l)
{
  if (l->blocks) CUDA_CHECK(cudaFree(l->blocks));
  l->blocks = NULL;
  l->n = 0;
}

template <class T>
static T *upload_items(const std::vector<T> &v)
{
  if (v.empty()) return NULL;
  T *d = NULL;
  CUDA_CHECK(cudaMalloc(&d, v.size() * sizeof(T)));
  CUDA_CHECK(cudaMemcpyAsync(d, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice, g_stream));
  CUDA_CHECK(cudaStreamSynchronize(g_stream));
  return d;
}

static void free_fill_tables(hpgmg_device_level *D)
{
  TileTable &TT = D->tile_fill;
  if (TT.ranges) CUDA_CHECK(cudaFree(TT.ranges));
  if (TT.copies) CUDA_CHECK(cudaFree(TT.copies));
  if (TT.bc) CUDA_CHECK(cudaFree(TT.bc));
  memset(&TT, 0, sizeof(TT));
  for (int s = 0; s < STENCIL_MAX_SHAPES; s++) {
    FillTable &T = D->fill[s];
    if (T.copies) CUDA_CHECK(cudaFree(T.copies));
    if (T.bc) CUDA_CHECK(cudaFree(T.bc));
    if (T.late) CUDA_CHECK(cudaFree(T.late));
    if (T.copies2) CUDA_CHECK(cudaFree(T.copies2));
    if (T.copies1) CUDA_CHECK(cudaFree(T.copies1));
    if (T.bc2) CUDA_CHECK(cudaFree(T.bc2));
    if (T.bc1) CUDA_CHECK(cudaFree(T.bc1));
    memset(&T, 0, sizeof(T));
  }
}

/* Tile shape of the fused box kernels (stencil_box.cuh) for boxes of n^3 cells; 0 if they do not cover the size */
extern "C" int hpgmg_box_tile_shape(int n, int *ti, int *tj, int *tk)
{
  if (n != 4 && n != 8 && n != 16 && n != 32) return 0;
  *ti = n < 16 ? n : 16;  *tj = n < 8 ? n : 8;  *tk = 4;
  return 1;
}

/* Bin the NO_CORNERS fill of a level by compute tile (TileTable, common.cuh): every record goes to each tile whose
 * staged halo tile [tk+4][tj+4][ti+4] contains its (nearest) ghost cell; a column's deeper ghost cells then lie in it too,
 * because box ghost zones and tile halos are both 2 cells deep and tiles are at least 4 cells wide. */
static void build_tile_table(level_type *level, hpgmg_device_level *D, const std::vector<FillCopy> &copies, const std::vector<FillBC> &bc)
{
  int ti, tj, tk;
  const int n = level->box_dim, g = level->box_ghosts;
  if (g != 2 || !hpgmg_box_tile_shape(n, &ti, &tj, &tk)) return;
  const int jS = level->box_jStride, kS = level->box_kStride;
  const long per_box = (long)level->numVectors * level->box_volume;
  const int ni = n / ti, nj = n / tj, nk = n / tk, per = ni * nj * nk, ntiles = per * level->num_my_boxes;
  const int sw = ti + 4, sh = tj + 4;
  std::vector<std::vector<TileCopy> > tc((size_t)ntiles);
  std::vector<std::vector<TileBC> > tb((size_t)ntiles);
  auto for_each_tile = [&](int dst, auto &&emit) {
    const int box = (int)(dst / per_box);
    const int pos = (int)(dst - box * per_box);
    const int c[3] = { pos % jS - g, (pos % kS) / jS - g, pos / kS - g };     /* the ghost cell, box coordinates */
    const int t[3] = { ti, tj, tk }, cnt[3] = { ni, nj, nk };
    int lo[3], hi[3];
    for (int a = 0; a < 3; a++) {
      /* tiles q with  q*t - 2 <= c < q*t + t + 2 */
      lo[a] = (c[a] - t[a] - 1 + t[a] - 1 + 64 * t[a]) / t[a] - 64;             /* ceil((c - t - 1) / t), arguments kept positive */
      hi[a] = (c[a] + 2 + 64 * t[a]) / t[a] - 64;                               /* floor((c + 2) / t) */
      if (lo[a] < 0) lo[a] = 0;
      if (hi[a] > cnt[a] - 1) hi[a] = cnt[a] - 1;
    }
    for (int qk = lo[2]; qk <= hi[2]; qk++) for (int qj = lo[1]; qj <= hi[1]; qj++) for (int qi = lo[0]; qi <= hi[0]; qi++) {
      const int tile = box * per + qi + ni * (qj + nj * qk);
      const int sidx = (c[0] - qi * ti + 2) + sw * ((c[1] - qj * tj + 2) + sh * (c[2] - qk * tk + 2));
      emit(tile, sidx);
    }
  };
  for (size_t e = 0; e < copies.size(); e++) {
    const FillCopy &r = copies[e];
    for_each_tile(r.dst, [&](int tile, int sidx) { TileCopy t = { r.src, r.dst, sidx, 0 }; tc[tile].push_back(t); });
  }
  for (size_t e = 0; e < bc.size(); e++) {
    const FillBC &r = bc[e];
    for_each_tile(r.dst, [&](int tile, int sidx) { TileBC t = { r.src, r.dst, sidx, r.subtype }; tb[tile].push_back(t); });
  }
  std::vector<TileRange> ranges((size_t)ntiles);
  std::vector<TileCopy> allc;
  std::vector<TileBC> allb;
  for (int t = 0; t < ntiles; t++) {
    TileRange R = { (int)allc.size(), (int)tc[t].size(), (int)allb.size(), (int)tb[t].size() };
    ranges[t] = R;
    allc.insert(allc.end(), tc[t].begin(), tc[t].end());
    allb.insert(allb.end(), tb[t].begin(), tb[t].end());
  }
  TileTable &TT = D->tile_fill;
  TT.ranges = upload_items(ranges);
  TT.copies = upload_items(allc);
  TT.bc = upload_items(allb);
  TT.ntiles = ntiles;  TT.ti = ti;  TT.tj = tj;  TT.tk = tk;
}

/* Expand the local ghost-exchange list and the BC list of every shape into per-cell / per-column records
 * (see FillTable in common.cuh).  The lists themselves are the reference's (level.c:367-465, 498-922);
 * this only flattens them and resolves, for each BC column, where its interior values come from. */
static void build_fill_tables(level_type *level, hpgmg_device_level *D)
{
  free_fill_tables(D);
  D->fill_nvec = level->numVectors;
  if (level->num_my_boxes == 0 || level->box_ghosts != STENCIL_RADIUS) return;      /* 2 ghost layers (fv4) or 1 (fv2) */
  const int jS = level->box_jStride, kS = level->box_kStride, n = level->box_dim, g = level->box_ghosts;
  const long per_box = (long)level->numVectors * level->box_volume;
  const long origin = (long)g * (1 + jS + kS);
  if (per_box * level->num_my_boxes >= 2147483647L) return;           /* offsets are 32-bit: fall back to the list kernels */
  /* local index of every box I own, by global id */
  const int total = level->boxes_in.i * level->boxes_in.j * level->boxes_in.k;
  std::vector<int> local_of(total, -1);
  for (int b = 0; b < level->num_my_boxes; b++) local_of[level->my_boxes[b].global_box_id] = b;

  for (int s = 0; s < STENCIL_MAX_SHAPES; s++) {
    std::vector<FillCopy> copies;
    const blockCopy_type *xb = level->exchange_ghosts[s].blocks[1];
    for (int e = 0; e < level->exchange_ghosts[s].num_blocks[1]; e++) {
      const blockCopy_type &B = xb[e];
      const long rb = B.read.box * per_box + origin, wb = B.write.box * per_box + origin;
      for (int k = 0; k < B.dim.k; k++) for (int j = 0; j < B.dim.j; j++) for (int i = 0; i < B.dim.i; i++) {
        FillCopy c = { (int)(rb + (B.read.i + i) + (long)(B.read.j + j) * jS + (long)(B.read.k + k) * kS),
                       (int)(wb + (B.write.i + i) + (long)(B.write.j + j) * jS + (long)(B.write.k + k) * kS) };
        copies.push_back(c);
      }
    }
    std::vector<FillBC> now, late;
    const blockCopy_type *bb = level->boundary_condition.blocks[s];
    for (int e = 0; e < level->boundary_condition.num_blocks[s]; e++) {
      const blockCopy_type &B = bb[e];
      const int nrm[3] = { (B.subtype % 3) - 1, ((B.subtype % 9) / 3) - 1, (B.subtype / 9) - 1 };
      const int lo[3] = { B.read.i, B.read.j, B.read.k }, ext[3] = { B.dim.i, B.dim.j, B.dim.k };
      const long st[3] = { 1, jS, kS };
      const box_type &box = level->my_boxes[B.read.box];
      const int bc[3] = { box.low.i / n, box.low.j / n, box.low.k / n };
      const int e0 = nrm[0] ? 1 : ext[0], e1 = nrm[1] ? 1 : ext[1], e2 = nrm[2] ? 1 : ext[2];
      for (int c = 0; c < e0 * e1 * e2; c++) {
        const int p[3] = { c % e0, (c / e0) % e1, c / (e0 * e1) };
        long cell = 0, image = 0;
        int nb[3] = { bc[0], bc[1], bc[2] }, shifted = 0;
        for (int a = 0; a < 3; a++) {
          if (nrm[a]) {                                   /* normal axis: nearest ghost cell, same in both frames */
            const int t = nrm[a] < 0 ? -1 : n;
            cell += t * st[a];  image += t * st[a];
          } else {
            const int q = p[a] + lo[a];                   /* tangential coordinate, possibly in a ghost range */
            cell += q * st[a];
            if (q < 0)       { nb[a] -= 1; image += (q + n) * st[a]; shifted = 1; }
            else if (q >= n) { nb[a] += 1; image += (q - n) * st[a]; shifted = 1; }
            else             image += q * st[a];
          }
        }
        FillBC it;
        it.dst = (int)(B.read.box * per_box + origin + cell);
        it.src = it.dst;
        it.subtype = B.subtype;
        it.pad = 0;
        if (!shifted) { now.push_back(it); continue; }
        /* the region the column reads is filled by exchange_boundary from box nb (always inside the domain) */
        const int gid = nb[0] + nb[1] * level->boxes_in.i + nb[2] * level->boxes_in.i * level->boxes_in.j;
        const int lb = (nb[0] < 0 || nb[1] < 0 || nb[2] < 0 || nb[0] >= level->boxes_in.i || nb[1] >= level->boxes_in.j || nb[2] >= level->boxes_in.k) ? -1 : local_of[gid];
        if (lb >= 0) { it.src = (int)(lb * per_box + origin + image); now.push_back(it); }
        else late.push_back(it);                          /* owned by another GPU: read my own ghost cells after the unpack */
      }
    }
    /* columns are independent of each other: group faces, edges and corners so that the threads of a warp run
     * the same extrapolation (1-D, 16-point, 64-point) instead of serialising all three */
    auto normals = [](const FillBC &it) { return ((it.subtype % 3) != 1) + (((it.subtype % 9) / 3) != 1) + ((it.subtype / 9) != 1); };
    auto by_kind = [&](const FillBC &x, const FillBC &y) { return normals(x) < normals(y); };
    std::stable_sort(now.begin(), now.end(), by_kind);
    std::stable_sort(late.begin(), late.end(), by_kind);
    if (s == STENCIL_SHAPE_NO_CORNERS && late.empty() && level->exchange_ghosts[s].num_sends == 0 && level->exchange_ghosts[s].num_recvs == 0)
      build_tile_table(level, D, copies, now);
    FillTable &T = D->fill[s];
    {
      /* pairs for the fill kernel (FillTable, common.cuh).  Offsets count doubles from the start of a box vector; create_vectors
       * aligns cell 0 (offset `origin`) to 16 bytes and strides are even, so an offset of origin's parity is a 16-byte aligned
       * address (any even offset with 2 ghost layers, any odd one with 1). */
      const int odd = (int)(origin & 1);
      std::vector<FillCopy> c2, c1;
      for (size_t e = 0; e < copies.size(); e++) {
        if (e + 1 < copies.size() && ((copies[e].src ^ odd) & 1) == 0 && ((copies[e].dst ^ odd) & 1) == 0 && copies[e + 1].src == copies[e].src + 1 && copies[e + 1].dst == copies[e].dst + 1) {
          c2.push_back(copies[e]);
          e++;
        } else c1.push_back(copies[e]);
      }
      std::vector<FillBC> b2, b1;
      for (size_t e = 0; e < now.size(); e++) {
        const bool i_tangential = (now[e].subtype % 3) == 1;                    /* the domain normal has no i component */
        if (i_tangential && e + 1 < now.size() && ((now[e].src ^ odd) & 1) == 0 && ((now[e].dst ^ odd) & 1) == 0 && now[e + 1].subtype == now[e].subtype &&
            now[e + 1].src == now[e].src + 1 && now[e + 1].dst == now[e].dst + 1) {
          b2.push_back(now[e]);
          e++;
        } else b1.push_back(now[e]);
      }
      auto normals = [](const FillBC &it) { return ((it.subtype % 3) != 1) + (((it.subtype % 9) / 3) != 1) + ((it.subtype / 9) != 1); };
      auto by_kind = [&](const FillBC &x, const FillBC &y) { return normals(x) < normals(y); };
      std::stable_sort(b2.begin(), b2.end(), by_kind);
      std::stable_sort(b1.begin(), b1.end(), by_kind);
      T.copies2 = upload_items(c2);  T.ncopies2 = (int)c2.size();
      T.copies1 = upload_items(c1);  T.ncopies1 = (int)c1.size();
      T.bc2 = upload_items(b2);      T.nbc2 = (int)b2.size();
      T.bc1 = upload_items(b1);      T.nbc1 = (int)b1.size();
    }
    T.copies = upload_items(copies);  T.ncopies = (int)copies.size();
    T.bc = upload_items(now);         T.nbc = (int)now.size();
    T.late = upload_items(late);      T.nlate = (int)late.size();
  }
}

extern "C" void hpgmg_device_level_rebind_vectors(level_type *level)
{
  hpgmg_device_level *D = HPGMG_DEV(level);
  DLevel &L = D->L;
  if (L.base != NULL) hpgmg_graph_drop_all(NULL);     /* create_vectors moved the slab: recorded solves hold the old pointers */
  L.nboxes = level->num_my_boxes;
  L.nvec = level->numVectors;
  L.dim = level->box_dim;
  L.ghosts = level->box_ghosts;
  L.jStride = level->box_jStride;
  L.kStride = level->box_kStride;
  L.volume = level->box_volume;
  L.origin = level->box_ghosts * (1 + level->box_jStride + level->box_kStride);
  L.base = (level->num_my_boxes > 0) ? level->my_boxes[0].vectors[0] : NULL;
  if (!hpgmg_rt_layout_only() && D->fill_nvec != 0 && D->fill_nvec != level->numVectors) build_fill_tables(level, D);   /* offsets contain numVectors */
}

extern "C" void hpgmg_device_level_create(level_type *level)
{
  hpgmg_device_level *D = (hpgmg_device_level *)calloc(1, sizeof(hpgmg_device_level));
  HPGMG_SET_DEV(level, D);
  hpgmg_device_level_rebind_vectors(level);

  if (hpgmg_rt_layout_only()) return;
  const int nb = level->num_my_boxes;
  if (nb > 0) {
    int *low = (int *)malloc((size_t)nb * 3 * sizeof(int));
    for (int b = 0; b < nb; b++) {
      low[3 * b + 0] = level->my_boxes[b].low.i;
      low[3 * b + 1] = level->my_boxes[b].low.j;
      low[3 * b + 2] = level->my_boxes[b].low.k;
    }
    CUDA_CHECK(cudaMalloc(&D->low, (size_t)nb * 3 * sizeof(int)));
    CUDA_CHECK(cudaMemcpyAsync(D->low, low, (size_t)nb * 3 * sizeof(int), cudaMemcpyHostToDevice, g_stream));
    CUDA_CHECK(cudaStreamSynchronize(g_stream));
    free(low);
  }
  for (int s = 0; s < STENCIL_MAX_SHAPES; s++) {
    upload_list(&D->bc[s], level->boundary_condition.blocks[s], level->boundary_condition.num_blocks[s]);
    for (int p = 0; p < 3; p++)
      upload_list(&D->exchange[s][p], level->exchange_ghosts[s].blocks[p], level->exchange_ghosts[s].num_blocks[p]);
  }
  build_fill_tables(level, D);
  D->ntiles = level->num_my_blocks;
  if (D->ntiles > 0) {
    CUDA_CHECK(cudaMalloc(&D->tiles, (size_t)D->ntiles * sizeof(blockCopy_type)));
    CUDA_CHECK(cudaMemcpyAsync(D->tiles, level->my_blocks, (size_t)D->ntiles * sizeof(blockCopy_type), cudaMemcpyHostToDevice, g_stream));
    CUDA_CHECK(cudaMalloc(&D->tile_partials, (size_t)D->ntiles * sizeof(double)));
    CUDA_CHECK(cudaStreamSynchronize(g_stream));
  }
}

extern "C" void hpgmg_device_level_upload_transfer_lists(level_type *level)
{
  hpgmg_device_level *D = HPGMG_DEV(level);
  for (int t = 0; t < 4; t++)
    for (int p = 0; p < 3; p++)
      upload_list(&D->restriction[t][p], level->restriction[t].blocks[p], level->restriction[t].num_blocks[p]);
  for (int p = 0; p < 3; p++)
    upload_list(&D->interpolation[p], level->interpolation.blocks[p], level->interpolation.num_blocks[p]);
}

extern "C" void hpgmg_device_level_destroy(level_type *level)
{
  hpgmg_device_level *D = HPGMG_DEV(level);
  if (!D) return;
  if (hpgmg_rt_layout_only()) { free(D); HPGMG_SET_DEV(level, NULL); return; }
  CUDA_CHECK(cudaStreamSynchronize(g_stream));
  for (int s = 0; s < STENCIL_MAX_SHAPES; s++) {
    free_list(&D->bc[s]);
    for (int p = 0; p < 3; p++) free_list(&D->exchange[s][p]);
  }
  for (int t = 0; t < 4; t++) for (int p = 0; p < 3; p++) free_list(&D->restriction[t][p]);
  for (int p = 0; p < 3; p++) free_list(&D->interpolation[p]);
  free_fill_tables(D);
  if (D->low) CUDA_CHECK(cudaFree(D->low));
  if (D->restrict_map) CUDA_CHECK(cudaFree(D->restrict_map));
  if (D->l1inv_alloc) hpgmg_rt_free(D->l1inv_alloc);
  if (D->tiles) CUDA_CHECK(cudaFree(D->tiles));
  if (D->tile_partials) CUDA_CHECK(cudaFree(D->tile_partials));
  free(D);
  HPGMG_SET_DEV(level, NULL);
}
