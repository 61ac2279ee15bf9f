/*
 * common.cuh -- what every CUDA translation unit of the library shares: the compute stream, the
 * launch counter, error checking and the by-value description of a level's HBM layout.
 *
 * There is no host fallback: every kernel is a __global__ function for sm_100a launched on the
 * library's stream; if no device is present hpgmg_b200_init() fails and nothing else works.
 */
#ifndef HPGMG_B200_COMMON_CUH
#define HPGMG_B200_COMMON_CUH

#include <cuda_runtime.h>
#include <stdint.h>
#include <stddef.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "hpgmg_b200.h"
#include "../runtime.h"

extern cudaStream_t g_stream;                   /* compute stream (runtime.cu)                    */
extern unsigned long long g_launches;           /* kernels enqueued; graph replays add their nodes */
extern int g_capturing;                         /* inside a stream capture?                        */

void hpgmg_cuda_check(cudaError_t e, const char *what, const char *file, int line);
#define CUDA_CHECK(x) hpgmg_cuda_check((x), #x, __FILE__, __LINE__)

/* Launch on the compute stream and count it.  Kernels are launched with programmatic stream
 * serialization (programmatic dependent launch): the next kernel's blocks may be scheduled while the
 * previous kernel drains, and every kernel starts with PDL_WAIT() (griddepcontrol.wait), which
 * blocks until the previous kernel's memory operations are complete and visible.  On the hundreds of
 * microsecond-sized kernels of the coarse levels this hides most of the launch gap. */
#ifndef HPGMG_PDL_EARLY
#define HPGMG_PDL_EARLY 0   /* measured: 7.00 vs 6.45 ms per `7 8` solve -- waiting grids take slots from the running one */
#endif
/* launch_dependents first: the NEXT kernel's blocks may be scheduled as soon as every block of this one has
 * started; they then sit in their own griddepcontrol.wait until this grid has completed and flushed, so
 * nothing is ever read early -- only the launch latency of the next kernel is taken off the critical path. */
#if HPGMG_PDL_EARLY
#define PDL_WAIT() asm volatile("griddepcontrol.launch_dependents;\n\tgriddepcontrol.wait;" ::: "memory")
#else
#define PDL_WAIT() asm volatile("griddepcontrol.wait;" ::: "memory")
#endif
extern int g_use_pdl;
void hpgmg_refuse_launch(const char *kernel);
template <typename... KArgs, typename... Args>
static inline void hpgmg_launch(const char *name, void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, Args &&...args)
{
  if (hpgmg_rt_layout_only()) hpgmg_refuse_launch(name);
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = grid;  cfg.blockDim = block;  cfg.dynamicSmemBytes = smem;  cfg.stream = g_stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = g_use_pdl ? 1 : 0;
  CUDA_CHECK(cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...));
  g_launches++;
}
/* cooperative launch: every block of the grid is resident at once (needed by kernels with a grid-wide barrier) */
template <typename... KArgs, typename... Args>
static inline void hpgmg_launch_cooperative(const char *name, void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, Args &&...args)
{
  if (hpgmg_rt_layout_only()) hpgmg_refuse_launch(name);
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = grid;  cfg.blockDim = block;  cfg.dynamicSmemBytes = smem;  cfg.stream = g_stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeCooperative;
  attr[0].val.cooperative = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  CUDA_CHECK(cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...));
  g_launches++;
}
/* the whole grid as ONE thread-block cluster (<= 16 blocks): barrier.cluster is a hardware barrier between
 * its blocks, with release/acquire semantics for global memory too */
template <typename... KArgs, typename... Args>
static inline void hpgmg_launch_cluster(const char *name, void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, Args &&...args)
{
  if (hpgmg_rt_layout_only()) hpgmg_refuse_launch(name);
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = grid;  cfg.blockDim = block;  cfg.dynamicSmemBytes = smem;  cfg.stream = g_stream;
  cudaLaunchAttribute attr[2];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = grid.x;  attr[0].val.clusterDim.y = 1;  attr[0].val.clusterDim.z = 1;
  attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[1].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = g_use_pdl ? 2 : 1;
  CUDA_CHECK(cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...));
  g_launches++;
}
__device__ __forceinline__ void cluster_barrier()
{
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
#define LAUNCH(kernel, grid, block, smem, ...) hpgmg_launch(#kernel, kernel, dim3(grid), dim3(block), (size_t)(smem), __VA_ARGS__)

/* One level's HBM layout, passed by value to kernels: a single slab [box][vector][k][j][i], every
 * box the same padded cube (reference level.c:935-938).  vec(b,id) points at cell (0,0,0). */
struct DLevel {
  double *base;
  int nboxes, nvec;
  int dim, ghosts;
  int jStride, kStride, volume;
  int origin;                                   /* ghosts*(1+jStride+kStride)                      */
  __host__ __device__ __forceinline__ double *vec(int box, int id) const
  {
    return base + ((size_t)box * (size_t)nvec + (size_t)id) * (size_t)volume + origin;
  }
};

/* a device copy of one blockCopy_type list */
struct DList {
  blockCopy_type *blocks;
  int n;
};

/* Flat work tables of a level's ghost fill (built on the host from the reference-identical block lists,
 * device_level.cu): one record per ghost cell copied inside this GPU and one per BC column.  Offsets
 * are in doubles from (DLevel::base + id*volume), i.e. they already contain box and cell.
 * A BC column whose tangential coordinates lie in a ghost region reads the image of that region in the
 * LOCAL neighbour box (src != dst), so copies and BCs have no mutual dependency and run as one kernel;
 * columns that depend on a box owned by another GPU are "late": they read the box's own ghost cells
 * after the unpack. */
#define COARSE_MAX_CELLS 4096
struct FillCopy { int src, dst; };
struct FillBC   { int dst, src, subtype, pad; };
struct FillTable {
  FillCopy *copies;  int ncopies;
  FillBC   *bc;      int nbc;         /* local-source columns */
  FillBC   *late;    int nlate;       /* columns that need data from another GPU first */
  /* the same copies and local-source columns regrouped for the fill kernel: items that are neighbours in i and 16-byte
   * aligned on both sides are ONE item moving two doubles (copies2, bc2: columns i and i+1 of a face / edge whose normal
   * has no i component); the rest stay single (copies1, bc1).  Half the items, 16-byte accesses. */
  FillCopy *copies2; int ncopies2;
  FillCopy *copies1; int ncopies1;
  FillBC   *bc2;     int nbc2;
  FillBC   *bc1;     int nbc1;
};

/* The same ghost fill (NO_CORNERS shape) binned by the compute tile that needs each value: the fused box kernels
 * (stencil_box.cuh) stage a tile of x with its halo in shared memory and resolve the halo themselves -- cells of
 * the neighbouring box and boundary-condition columns go straight into the staged tile -- so a sweep needs no
 * separate fill kernel.  A record is listed under every tile whose halo contains its ghost cell(s).
 * sidx: index of the (nearest) ghost cell in the staged tile [TK+4][TJ+4][TI+4]. */
struct TileCopy { int src, dst, sidx, pad; };
struct TileBC   { int src, dst, sidx, subtype; };
struct TileRange { int copy0, ncopy, bc0, nbc; };
struct TileTable {
  TileRange *ranges;                            /* [nboxes * tiles per box], box-major, then k, j, i */
  TileCopy  *copies;
  TileBC    *bc;
  int ntiles, ti, tj, tk;                       /* tile shape the table was binned for; ntiles == 0: not available */
};

/* device mirror hanging off level_type::fluxes */
struct hpgmg_device_level {
  DLevel L;
  int   *low;                                   /* device [nboxes][3]: global coords of cell 0,0,0 */
  DList  bc[STENCIL_MAX_SHAPES];
  DList  exchange[STENCIL_MAX_SHAPES][3];
  DList  restriction[4][3];
  DList  interpolation[3];
  FillTable fill[STENCIL_MAX_SHAPES];
  TileTable tile_fill;                          /* NO_CORNERS fill binned per compute tile (boxes of 4^3 .. 32^3 whose neighbours are all on this GPU) */
  int fill_nvec;                                /* numVectors the fill offsets were built for */
  int dinv_is_unit_diagonal;                    /* VECTOR_DINV was last written by rebuild_operator_blackbox with >= 4 colours per
                                                   dimension (no two cells of a colour inside one stencil): away from the boundary it
                                                   then holds exactly 1/(A applied to the unit vector), which the GSRB kernel may
                                                   recompute instead of reading.  Cleared by every other writer of the vector
                                                   (hpgmg_note_vector_written: BLAS1, transfers, smoothers, uploads). */
  int   *restrict_map;                          /* device [nboxes][4]: coarse box and coarse cell of cell (0,0,0) of every box (smooth.cu: residual fused with restriction) */
  int    restrict_map_state;                    /* 0 not looked at yet, 1 available, -1 the level's restriction is not box-to-box on this GPU */
  double *l1inv;                                /* default build, L1-Jacobi only: the L1 row inverse, [box][k][j][i] with the geometry of one
                                                   slab vector (the vector map has no room for it); written by rebuild_operator_blackbox */
  double *tile_partials;                        /* scratch for dot/mean: one double per compute tile */
  blockCopy_type *tiles;                        /* device copy of level->my_blocks                  */
  int     ntiles;
};

/* per-operator timers of the reference (level->timers.*, e.g. gsrb.c:37,130): only when
 * hpgmg_b200_profile_operators(1) is on; each bracket then synchronises the stream (graphs are off
 * in that mode), so MGPrintTiming shows the same table as the reference. */
struct ProfileScope {
  double *field, *total;
  double t0;
  ProfileScope(double *f, double *tot = NULL) : field(NULL), total(tot), t0(0.0)
  {
    if (!hpgmg_rt_profile()) return;
    field = f;
    CUDA_CHECK(cudaStreamSynchronize(g_stream));
    t0 = hpgmg_rt_wtime();
  }
  ~ProfileScope()
  {
    if (!field) return;
    CUDA_CHECK(cudaStreamSynchronize(g_stream));
    const double dt = hpgmg_rt_wtime() - t0;
    *field += dt;
    if (total) *total += dt;
  }
};

/* timing experiments only (HPGMG_B200_ABLATE=bitmask): skip a class of kernels to see what it costs inside the
 * replayed graph; results are garbage in that mode.  1 ghost fills dim>=64, 2 ghost fills dim<64, 4 coarse kernel,
 * 8 stencil kernels dim<64, 16 restriction/interpolation, 32 residual dim>=64, 64 smoother sweeps dim>=64, 128 BLAS1/norm */
static inline int hpgmg_ablate(const int bit)
{
  static int mask = -1;
  if (mask < 0) { const char *e = getenv("HPGMG_B200_ABLATE"); mask = e ? atoi(e) : 0; }
  return mask & bit;
}

static inline const DLevel &dl_of(const level_type *level) { return HPGMG_DEV(level)->L; }

/* Every operator that writes vector `id` of a level through the public API says so: a diagonal that no longer
 * comes from rebuild_operator_blackbox must be read from memory again, and recorded solves that baked the
 * shortcut in are dropped (runtime.cu). */
void hpgmg_dinv_overwritten(level_type *level);
static inline void hpgmg_note_vector_written(level_type *level, const int id)
{
  if (id == VECTOR_DINV && HPGMG_DEV(level) && HPGMG_DEV(level)->dinv_is_unit_diagonal) hpgmg_dinv_overwritten(level);
}

/* max over non-negative doubles through their bit pattern (IEEE order == unsigned integer order) */
__device__ __forceinline__ void atomic_max_nonneg(double *addr, double v)
{
  atomicMax((unsigned long long *)addr, (unsigned long long)__double_as_longlong(v));
}

#endif
