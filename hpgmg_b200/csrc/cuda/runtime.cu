/*
 * runtime.cu -- device selection, the compute stream, device memory, scalar slots, CUDA-graph
 * record/replay and the host<->device copies of the public C-ABI (include/hpgmg_b200.h).
 *
 * The reference has no counterpart (it is a host program: MALLOC is posix_memalign,
 * level.c:24-40; timers are omp_get_wtime, timers/omp.c).  One process drives one GPU.
 */
#include <string.h>
#include <time.h>
#include <sys/mman.h>
#include <map>
#include <vector>

#include <cuda_profiler_api.h>
#include "common.cuh"

cudaStream_t g_stream = 0;
unsigned long long g_launches = 0;
int g_capturing = 0;
int g_use_pdl = 1;
extern "C" void hpgmg_b200_use_pdl(int on) { if ((on ? 1 : 0) != g_use_pdl) hpgmg_graph_drop_all(NULL); g_use_pdl = on ? 1 : 0; }

void hpgmg_dinv_overwritten(level_type *level)
{
  HPGMG_DEV(level)->dinv_is_unit_diagonal = 0;
  hpgmg_graph_drop_all(NULL);                       /* recorded sweeps formed 1/Aii in registers */
}

static int g_initialised = 0;
static int g_device = -1;
static int g_verbose = 1;
static int g_smoother = HPGMG_SMOOTHER_GSRB;
static int g_use_graphs = 1;
static int g_profile = 0;
static double *g_scalars = NULL;            /* device, HPGMG_NUM_SCALARS doubles */
static double *g_scalars_host = NULL;       /* pinned mirror                      */
static cudaEvent_t g_ev0, g_ev1;
static double g_last_device_seconds = 0.0;
#define NSTAGING 4                                /* dense cells of f / u of the end-to-end solve: [0],[1] slot 0; [2],[3] slot 1 */
static void *g_staging[NSTAGING] = { NULL, NULL, NULL, NULL };
static size_t g_staging_bytes[NSTAGING] = { 0, 0, 0, 0 };
static cudaStream_t g_side_stream = 0, g_main_stream_saved = 0;
static cudaEvent_t g_ev_fork = 0, g_ev_join = 0;

/* Layout-only mode: the host-side data model (decomposition, block lists, level table) can be built
 * and inspected on a machine without a GPU.  Allocations become inaccessible address-space
 * reservations (any dereference faults), nothing is copied and every kernel launch aborts -- it is
 * a way to test the index mapping, not a compute path. */
static int g_layout_only = 0;
static std::map<void *, size_t> g_reservations;
extern "C" void hpgmg_b200_set_layout_only(int on) { g_layout_only = on; }
extern "C" int  hpgmg_rt_layout_only(void) { return g_layout_only; }
void hpgmg_refuse_launch(const char *kernel)
{
  fprintf(stderr, "hpgmg_b200: kernel %s requested in layout-only mode; compute needs a B200 (no CPU fallback)\n", kernel);
  abort();
}

void hpgmg_cuda_check(cudaError_t e, const char *what, const char *file, int line)
{
  if (e == cudaSuccess) return;
  fprintf(stderr, "hpgmg_b200: CUDA error %s (%s) at %s:%d in `%s`\n", cudaGetErrorName(e), cudaGetErrorString(e), file, line, what);
  fflush(stderr);
  abort();
}

static void require_init(const char *who)
{
  if (g_initialised || g_layout_only) return;
  /* lazy init on device 0 (or HPGMG_B200_DEVICE / LOCAL_RANK) so that a reference-style main()
   * that knows nothing about GPUs still works; failure is fatal -- there is no CPU path */
  int dev = 0;
  const char *e = getenv("HPGMG_B200_DEVICE");
  if (!e) e = getenv("LOCAL_RANK");
  if (e) dev = atoi(e);
  if (hpgmg_b200_init(dev) != 0) {
    fprintf(stderr, "hpgmg_b200: %s needs a CUDA device (sm_100a) and none could be initialised; there is no CPU fallback\n", who);
    exit(1);
  }
}

extern "C" int hpgmg_b200_init(int device_ordinal)
{
  if (g_initialised) return 0;
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess || count == 0) {
    fprintf(stderr, "hpgmg_b200_init: no CUDA device (%s)\n", e == cudaSuccess ? "count=0" : cudaGetErrorString(e));
    return 1;
  }
  if (device_ordinal < 0 || device_ordinal >= count) device_ordinal = device_ordinal % count;
  e = cudaSetDevice(device_ordinal);
  if (e != cudaSuccess) { fprintf(stderr, "hpgmg_b200_init: cudaSetDevice(%d): %s\n", device_ordinal, cudaGetErrorString(e)); return 2; }
  cudaDeviceProp prop;
  CUDA_CHECK(cudaGetDeviceProperties(&prop, device_ordinal));
  if (prop.major < 10) {
    fprintf(stderr, "hpgmg_b200_init: device %d is sm_%d%d; this library carries sm_100a code only\n", device_ordinal, prop.major, prop.minor);
    return 3;
  }
  g_device = device_ordinal;
  { const char *e = getenv("HPGMG_B200_NO_PDL"); if (e && atoi(e)) g_use_pdl = 0; }
  CUDA_CHECK(cudaStreamCreateWithFlags(&g_stream, cudaStreamNonBlocking));
  CUDA_CHECK(cudaMalloc(&g_scalars, HPGMG_NUM_SCALARS * sizeof(double)));
  CUDA_CHECK(cudaMemset(g_scalars, 0, HPGMG_NUM_SCALARS * sizeof(double)));
  CUDA_CHECK(cudaMallocHost(&g_scalars_host, HPGMG_NUM_SCALARS * sizeof(double)));
  CUDA_CHECK(cudaEventCreate(&g_ev0));
  CUDA_CHECK(cudaEventCreate(&g_ev1));
  g_initialised = 1;
  return 0;
}

extern "C" void hpgmg_b200_finalize(void)
{
  if (!g_initialised) return;
  cudaStreamSynchronize(g_stream);
  hpgmg_graph_drop_all(NULL);
  cudaFree(g_scalars);  cudaFreeHost(g_scalars_host);
  for (int w = 0; w < NSTAGING; w++) { if (g_staging[w]) cudaFree(g_staging[w]); g_staging[w] = NULL; g_staging_bytes[w] = 0; }
  hpgmg_rt_pipe_destroy();
  if (g_side_stream) { cudaStreamDestroy(g_side_stream); cudaEventDestroy(g_ev_fork); cudaEventDestroy(g_ev_join); g_side_stream = 0; }
  cudaEventDestroy(g_ev0);  cudaEventDestroy(g_ev1);
  cudaStreamDestroy(g_stream);
  g_stream = 0;  g_initialised = 0;
}

extern "C" void hpgmg_b200_sync(void) { require_init("sync"); CUDA_CHECK(cudaStreamSynchronize(g_stream)); }
extern "C" const char *hpgmg_b200_backend(void) { return "cuda-sm_100a"; }
extern "C" void *hpgmg_b200_stream(void) { require_init("stream"); return (void *)g_stream; }
extern "C" int hpgmg_b200_device(void) { return g_device; }

extern "C" void hpgmg_b200_set_smoother(int which)
{
  if (which != HPGMG_SMOOTHER_GSRB && which != HPGMG_SMOOTHER_CHEBY && which != HPGMG_SMOOTHER_JACOBI && which != HPGMG_SMOOTHER_L1JACOBI) {
    fprintf(stderr, "hpgmg_b200_set_smoother: %d is not a smoother (0 GSRB, 1 Chebyshev, 2 Jacobi, 3 L1-Jacobi); keeping %d\n", which, g_smoother);
    return;
  }
  g_smoother = which;
}
extern "C" int  hpgmg_b200_get_smoother(void) { return g_smoother; }
extern "C" void hpgmg_b200_set_verbose(int on) { g_verbose = on; }
extern "C" void hpgmg_b200_use_graphs(int on) { g_use_graphs = on; }
extern "C" void hpgmg_b200_profile_operators(int on) { g_profile = on; }

extern "C" int hpgmg_rt_verbose(void) { return g_verbose; }
extern "C" int hpgmg_rt_smoother(void) { return g_smoother; }
extern "C" int hpgmg_rt_use_graphs(void) { return g_use_graphs; }
extern "C" int hpgmg_rt_profile(void) { return g_profile; }
extern "C" int hpgmg_rt_sm_count(void)
{
  static int sms = 0;
  if (!sms) {
    int dev = 0;
    CUDA_CHECK(cudaGetDevice(&dev));
    CUDA_CHECK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    if (sms <= 0) sms = 148;
  }
  return sms;
}
extern "C" double hpgmg_rt_wtime(void)
{
  struct timespec ts;
  clock_gettime(CLOCK_MONOTONIC, &ts);
  return (double)ts.tv_sec + 1e-9 * (double)ts.tv_nsec;
}

/* ------------------------------------------------------------------------------------------ */
extern "C" void *hpgmg_rt_alloc_zero(size_t bytes)
{
  require_init("alloc");
  if (bytes == 0) bytes = 8;
  if (g_layout_only) {
    void *r = mmap(NULL, bytes, PROT_NONE, MAP_PRIVATE | MAP_ANONYMOUS | MAP_NORESERVE, -1, 0);
    if (r == MAP_FAILED) { fprintf(stderr, "hpgmg_b200: cannot reserve %zu bytes of address space\n", bytes); exit(0); }
    g_reservations[r] = bytes;
    return r;
  }
  void *p = NULL;
  cudaError_t e = cudaMalloc(&p, bytes);
  if (e != cudaSuccess) {
    fprintf(stderr, "hpgmg_b200: cudaMalloc(%zu bytes) failed: %s\n", bytes, cudaGetErrorString(e));
    exit(0);                                           /* the reference exits on malloc failure too (level.c:339) */
  }
  CUDA_CHECK(cudaMemsetAsync(p, 0, bytes, g_stream));
  return p;
}
extern "C" void hpgmg_rt_free(void *p)
{
  if (!p) return;
  if (g_layout_only) {
    std::map<void *, size_t>::iterator it = g_reservations.find(p);
    if (it != g_reservations.end()) { munmap(p, it->second); g_reservations.erase(it); }
    return;
  }
  if (hpgmg_rt_is_comm_memory(p)) { hpgmg_rt_free_comm(p); return; }   /* bump-allocated from the peer-visible arena: recycled when every rank is done with it */
  CUDA_CHECK(cudaStreamSynchronize(g_stream));
  CUDA_CHECK(cudaFree(p));
}
extern "C" void *MALLOC(size_t size) { return hpgmg_rt_alloc_zero(size); }
extern "C" void  FREE(void *ptr) { hpgmg_rt_free(ptr); }

extern "C" void hpgmg_rt_copy_d2d(void *dst, const void *src, size_t bytes) { if (g_layout_only) return; CUDA_CHECK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToDevice, g_stream)); }
extern "C" void hpgmg_rt_copy_h2d(void *dst, const void *src, size_t bytes) { if (g_layout_only) return; CUDA_CHECK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, g_stream)); }
extern "C" void hpgmg_rt_copy_d2h(void *dst, const void *src, size_t bytes) { if (g_layout_only) return; CUDA_CHECK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, g_stream)); }
extern "C" void hpgmg_rt_sync(void) { if (g_initialised && !g_layout_only) CUDA_CHECK(cudaStreamSynchronize(g_stream)); }

extern "C" void *hpgmg_b200_host_alloc_pinned(size_t bytes)
{
  require_init("pinned alloc");
  void *p = NULL;
  CUDA_CHECK(cudaMallocHost(&p, bytes ? bytes : 8));
  return p;
}
extern "C" void hpgmg_b200_host_free_pinned(void *p) { if (p) CUDA_CHECK(cudaFreeHost(p)); }

extern "C" void hpgmg_download_box_vector(level_type *level, int box, int id, double *host)
{
  const box_type *B = &level->my_boxes[box];
  hpgmg_rt_copy_d2h(host, B->vectors[id], (size_t)B->volume * sizeof(double));
  hpgmg_rt_sync();
}
extern "C" void hpgmg_upload_box_vector(level_type *level, int box, int id, const double *host)
{
  const box_type *B = &level->my_boxes[box];
  hpgmg_rt_copy_h2d(B->vectors[id], host, (size_t)B->volume * sizeof(double));
  hpgmg_rt_sync();
  hpgmg_note_vector_written(level, id);               /* a caller-supplied diagonal is read, not recomputed */
}

/* ------------------------------------------------------------------------------------------ */
extern "C" double *hpgmg_rt_scalar_slots(void) { require_init("scalars"); return g_scalars; }
extern "C" void hpgmg_rt_zero_scalar(int slot)
{
  CUDA_CHECK(cudaMemsetAsync(g_scalars + slot, 0, sizeof(double), g_stream));
}
extern "C" void hpgmg_rt_read_scalars(double *host, int first, int count)
{
  if (g_capturing) { fprintf(stderr, "hpgmg_b200: a host read-back (dot / norm / mean value) was requested inside a recorded solve; the caller must not capture this path\n"); abort(); }
  CUDA_CHECK(cudaMemcpyAsync(g_scalars_host + first, g_scalars + first, (size_t)count * sizeof(double), cudaMemcpyDeviceToHost, g_stream));
  CUDA_CHECK(cudaStreamSynchronize(g_stream));
  memcpy(host, g_scalars_host + first, (size_t)count * sizeof(double));
}

/* ------------------------------------------------------------------------------------------ */
/* CUDA-graph record / replay keyed by (owner, key) */
struct GraphEntry {
  const void *owner;
  long long key;
  cudaGraphExec_t exec;
  unsigned long long kernels;
};
static std::vector<GraphEntry> g_graphs;
static unsigned long long g_capture_start_launches = 0;

extern "C" int hpgmg_graph_begin(const void *owner, long long key)
{
  for (size_t i = 0; i < g_graphs.size(); i++) {
    if (g_graphs[i].owner == owner && g_graphs[i].key == key) {
      CUDA_CHECK(cudaGraphLaunch(g_graphs[i].exec, g_stream));
      g_launches += g_graphs[i].kernels;
      return 0;
    }
  }
  CUDA_CHECK(cudaStreamBeginCapture(g_stream, cudaStreamCaptureModeThreadLocal));
  g_capturing = 1;
  g_capture_start_launches = g_launches;
  return 1;
}

extern "C" void hpgmg_graph_end(const void *owner, long long key)
{
  cudaGraph_t graph = NULL;
  CUDA_CHECK(cudaStreamEndCapture(g_stream, &graph));
  g_capturing = 0;
  GraphEntry e;
  e.owner = owner;  e.key = key;  e.kernels = g_launches - g_capture_start_launches;
  CUDA_CHECK(cudaGraphInstantiate(&e.exec, graph, 0));
  CUDA_CHECK(cudaGraphDestroy(graph));
  g_graphs.push_back(e);
  /* the capture only recorded the work: run it now */
  CUDA_CHECK(cudaGraphLaunch(e.exec, g_stream));
}

extern "C" void hpgmg_graph_drop_all(const void *owner)
{
  if (g_capturing) { fprintf(stderr, "hpgmg_b200: the hierarchy was modified (vectors re-allocated / operator rebuilt / kernel switches) inside a recorded solve\n"); abort(); }
  for (size_t i = 0; i < g_graphs.size();) {
    if (owner == NULL || g_graphs[i].owner == owner) {
      cudaGraphExecDestroy(g_graphs[i].exec);
      g_graphs.erase(g_graphs.begin() + i);
    } else i++;
  }
}

/* ------------------------------------------------------------------------------------------ */
extern "C" void hpgmg_rt_timer_start(void) { CUDA_CHECK(cudaEventRecord(g_ev0, g_stream)); }
extern "C" void hpgmg_rt_timer_stop(void) { CUDA_CHECK(cudaEventRecord(g_ev1, g_stream)); }
extern "C" double hpgmg_b200_device_seconds_last_solve(void)
{
  float ms = 0.f;
  CUDA_CHECK(cudaEventSynchronize(g_ev1));
  CUDA_CHECK(cudaEventElapsedTime(&ms, g_ev0, g_ev1));
  g_last_device_seconds = 1e-3 * (double)ms;
  return g_last_device_seconds;
}
/* bracket a region for `ncu --profile-from-start off` */
extern "C" void hpgmg_b200_profiler_start(void) { require_init("profiler"); CUDA_CHECK(cudaStreamSynchronize(g_stream)); cudaProfilerStart(); }
extern "C" void hpgmg_b200_profiler_stop(void) { CUDA_CHECK(cudaStreamSynchronize(g_stream)); cudaProfilerStop(); }

/* event marks on the compute stream for callers that time several calls (bench.py) */
static cudaEvent_t g_marks[8];
static int g_marks_ready = 0;
extern "C" void hpgmg_b200_bench_mark(int idx)
{
  require_init("bench mark");
  if (!g_marks_ready) { for (int i = 0; i < 8; i++) CUDA_CHECK(cudaEventCreate(&g_marks[i])); g_marks_ready = 1; }
  CUDA_CHECK(cudaEventRecord(g_marks[idx & 7], g_stream));
}
extern "C" double hpgmg_b200_bench_elapsed_ms(int from, int to)
{
  float ms = 0.f;
  CUDA_CHECK(cudaEventSynchronize(g_marks[to & 7]));
  CUDA_CHECK(cudaEventElapsedTime(&ms, g_marks[from & 7], g_marks[to & 7]));
  return (double)ms;
}
extern "C" unsigned long long hpgmg_b200_kernel_launches(void) { return g_launches; }

/* ------------------------------------------------------------------------------------------ */
/* Plumbing of the end-to-end solve with HOST buffers (hpgmg_fmg_solve_host, mg.c): two device staging buffers that hold
 * the dense cells of f and u, and a side stream on which the download of u runs while the compute stream finishes the
 * solve (final residual + norm).  Fork and join are event edges, so they are recorded into the solve's CUDA graph. */

extern "C" void *hpgmg_rt_staging(int which, size_t bytes)
{
  require_init("staging");
  if (bytes > g_staging_bytes[which]) {
    CUDA_CHECK(cudaStreamSynchronize(g_stream));
    hpgmg_graph_drop_all(NULL);                        /* recorded end-to-end solves hold the old buffer */
    if (g_staging[which]) CUDA_CHECK(cudaFree(g_staging[which]));
    CUDA_CHECK(cudaMalloc(&g_staging[which], bytes));
    g_staging_bytes[which] = bytes;
  }
  return g_staging[which];
}
/* from here on the library's launches and copies go to the side stream, which first waits for everything enqueued so far */
extern "C" void hpgmg_rt_side_begin(void)
{
  if (!g_side_stream) {
    CUDA_CHECK(cudaStreamCreateWithFlags(&g_side_stream, cudaStreamNonBlocking));
    CUDA_CHECK(cudaEventCreateWithFlags(&g_ev_fork, cudaEventDisableTiming));
    CUDA_CHECK(cudaEventCreateWithFlags(&g_ev_join, cudaEventDisableTiming));
  }
  CUDA_CHECK(cudaEventRecord(g_ev_fork, g_stream));
  CUDA_CHECK(cudaStreamWaitEvent(g_side_stream, g_ev_fork, 0));
  g_main_stream_saved = g_stream;
  g_stream = g_side_stream;
}
/* back to the compute stream; the side work keeps running */
extern "C" void hpgmg_rt_side_end(void)
{
  CUDA_CHECK(cudaEventRecord(g_ev_join, g_stream));
  g_stream = g_main_stream_saved;
}
/* the compute stream waits for the side work */
extern "C" void hpgmg_rt_side_join(void) { CUDA_CHECK(cudaStreamWaitEvent(g_stream, g_ev_join, 0)); }

/* ------------------------------------------------------------------------------------------ */
/* Pipelined end-to-end solves (hpgmg_fmg_solve_host_submit / _wait, mg.c): two slots, each with its own staging buffers.
 * The upload of solve n+1 runs on its own stream while solve n computes, the download of solve n while solve n+1 computes
 * (PCIe is full duplex); the compute stream only ever waits for "f of this slot has arrived".  A slot is reused only after
 * the host has waited for its previous solve, so its staging buffers are free by then. */
static cudaStream_t g_up_stream = 0, g_down_stream = 0;
static cudaEvent_t g_ev_up[2], g_ev_packed[2], g_ev_down[2], g_ev_scal[2];
static double *g_pipe_scalars_host = NULL;            /* pinned, 2 x 4 doubles */
static void pipe_init(void)
{
  if (g_up_stream) return;
  CUDA_CHECK(cudaStreamCreateWithFlags(&g_up_stream, cudaStreamNonBlocking));
  CUDA_CHECK(cudaStreamCreateWithFlags(&g_down_stream, cudaStreamNonBlocking));
  for (int s = 0; s < 2; s++) {
    CUDA_CHECK(cudaEventCreateWithFlags(&g_ev_up[s], cudaEventDisableTiming));
    CUDA_CHECK(cudaEventCreateWithFlags(&g_ev_packed[s], cudaEventDisableTiming));
    CUDA_CHECK(cudaEventCreateWithFlags(&g_ev_down[s], cudaEventDisableTiming));
    CUDA_CHECK(cudaEventCreateWithFlags(&g_ev_scal[s], cudaEventDisableTiming));
  }
  CUDA_CHECK(cudaHostAlloc(&g_pipe_scalars_host, 8 * sizeof(double), cudaHostAllocMapped));
}
/* three doubles straight into mapped host memory: a D2H copy here would queue behind the 134 MB download of this very
 * solve on the copy engine and hold the compute stream (and with it the next solve) for its 2.5 ms */
__global__ void publish_scalars_kernel(double *host_mapped, const double *src)
{
  PDL_WAIT();
  if (threadIdx.x < 3) host_mapped[threadIdx.x] = src[threadIdx.x];
  __threadfence_system();
}
extern "C" void hpgmg_rt_pipe_destroy(void)
{
  if (!g_up_stream) return;
  cudaStreamSynchronize(g_up_stream);  cudaStreamSynchronize(g_down_stream);
  for (int s = 0; s < 2; s++) { cudaEventDestroy(g_ev_up[s]); cudaEventDestroy(g_ev_packed[s]); cudaEventDestroy(g_ev_down[s]); cudaEventDestroy(g_ev_scal[s]); }
  cudaStreamDestroy(g_up_stream);  cudaStreamDestroy(g_down_stream);
  cudaFreeHost(g_pipe_scalars_host);
  g_up_stream = g_down_stream = 0;  g_pipe_scalars_host = NULL;
}
/* f_host -> stage on the upload stream; the compute stream waits for it (and for nothing else) */
extern "C" void hpgmg_rt_pipe_upload(int slot, void *stage, const void *host, size_t bytes)
{
  pipe_init();
  if (bytes) CUDA_CHECK(cudaMemcpyAsync(stage, host, bytes, cudaMemcpyHostToDevice, g_up_stream));
  CUDA_CHECK(cudaEventRecord(g_ev_up[slot], g_up_stream));
  CUDA_CHECK(cudaStreamWaitEvent(g_stream, g_ev_up[slot], 0));
}
/* u has been packed into `stage` by everything enqueued so far on the compute stream: send it home on the download stream */
extern "C" void hpgmg_rt_pipe_download(int slot, void *host, const void *stage, size_t bytes)
{
  pipe_init();
  CUDA_CHECK(cudaEventRecord(g_ev_packed[slot], g_stream));
  CUDA_CHECK(cudaStreamWaitEvent(g_down_stream, g_ev_packed[slot], 0));
  if (bytes) CUDA_CHECK(cudaMemcpyAsync(host, stage, bytes, cudaMemcpyDeviceToHost, g_down_stream));
  CUDA_CHECK(cudaEventRecord(g_ev_down[slot], g_down_stream));
}
/* the solve's scalars (||F||, ||r||, Krylov iterations) as they are at this point of the compute stream */
extern "C" void hpgmg_rt_pipe_scalars(int slot)
{
  pipe_init();
  double *mapped = NULL;
  CUDA_CHECK(cudaHostGetDevicePointer(&mapped, g_pipe_scalars_host + 4 * slot, 0));
  LAUNCH(publish_scalars_kernel, 1, 32, 0, mapped, g_scalars + HPGMG_SLOT_NORM_F);
  CUDA_CHECK(cudaEventRecord(g_ev_scal[slot], g_stream));
}
extern "C" void hpgmg_rt_pipe_wait(int slot, double *scalars3)
{
  CUDA_CHECK(cudaEventSynchronize(g_ev_scal[slot]));
  CUDA_CHECK(cudaEventSynchronize(g_ev_down[slot]));
  memcpy(scalars3, g_pipe_scalars_host + 4 * slot, 3 * sizeof(double));
}
