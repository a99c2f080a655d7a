// ttmpc_api.cu -- the C-ABI (include/ttmpc.h) over the sm_100a kernels.
// Host-side only: argument checking, workspace management, staging copies.
#include <cuda_runtime.h>

#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <algorithm>
#include <atomic>
#include <condition_variable>
#include <mutex>
#include <thread>
#include <string>
#include <vector>

#include "ttmpc_device.cuh"
#include "ttmpc_launch.cuh"

using namespace ttmpc;

static thread_local std::string g_err;
static int fail(int code, const std::string &msg) { g_err = msg; return code; }
// the DQN entry points (ttdqn.cu) report through the same per-thread string, so that
// ttmpc_last_error() describes the last failure of ANY entry point of the library
namespace ttmpc { void set_last_error(const std::string &msg) { g_err = msg; } }
#define CUDA_TRY(x)                                                                     \
  do {                                                                                  \
    cudaError_t e__ = (x);                                                              \
    if (e__ != cudaSuccess)                                                             \
      return fail(TTMPC_ERR_CUDA, std::string(#x) + ": " + cudaGetErrorString(e__));    \
  } while (0)

extern "C" const char *ttmpc_last_error(void) { return g_err.c_str(); }
extern "C" int ttmpc_version(void) { return TTMPC_VERSION; }
extern "C" int ttmpc_set_device(int device) { CUDA_TRY(cudaSetDevice(device)); return TTMPC_OK; }
extern "C" int ttmpc_get_device(int *device) {
  if (!device) return fail(TTMPC_ERR_BAD_ARG, "null output");
  CUDA_TRY(cudaGetDevice(device));
  return TTMPC_OK;
}
extern "C" const char *ttmpc_exit_status_name(int code) {
  switch (code) {
    case TTMPC_CONVERGED: return "Converged";
    case TTMPC_NOT_CONVERGED_ITERATIONS: return "NotConvergedIterations";
    case TTMPC_NOT_CONVERGED_OUT_OF_TIME: return "NotConvergedOutOfTime";
    case TTMPC_NOT_FINITE: return "NotFiniteComputation";
    default: return "Unknown";
  }
}

// config/mpc_default.yaml + opengen 0.7.1 SolverConfiguration defaults, with
// initial_penalty 10 as set at mpc_generator.py:269.
extern "C" void ttmpc_default_config(ttmpc_config *c) {
  std::memset(c, 0, sizeof(*c));
  c->N_hor = 20; c->nu = 2; c->ns = 3; c->nq = 10;
  c->Nother = 10; c->Nstcobs = 10; c->nstcobs = 12; c->Ndynobs = 15; c->ndynobs = 6;
  c->ts = 0.2; c->vehicle_width = 0.5; c->social_margin = 0.2;
  c->lin_vel_min = -0.5; c->lin_vel_max = 1.5; c->ang_vel_max = 0.5;
  c->lin_acc_min = -1.0; c->lin_acc_max = 1.0; c->ang_acc_max = 3.0;
  c->tolerance = 1e-4; c->initial_tolerance = 1e-4; c->delta_tolerance = 1e-4;
  c->initial_penalty = 10.0; c->penalty_update_factor = 5.0;
  c->inner_tolerance_update_factor = 0.1; c->sufficient_decrease_coeff = 0.1;
  c->lbfgs_memory = 10; c->max_inner_iterations = 500; c->max_outer_iterations = 10;
  c->max_duration_ms = 5000;  // MAX_SOVLER_TIME = 5_000_000 us (mpc_generator.py:22)
}
extern "C" int ttmpc_num_params(const ttmpc_config *c) {
  const int N = c->N_hor;
  return 2 * c->ns + c->nu + c->nq + c->ns * N + N + c->ns * N * c->Nother +
         c->Nstcobs * c->nstcobs + c->Ndynobs * c->ndynobs * N + 2 * N;
}
extern "C" int ttmpc_num_decision(const ttmpc_config *c) { return c->nu * c->N_hor; }
extern "C" int ttmpc_num_alm(const ttmpc_config *c) { return 2 * c->N_hor; }
extern "C" int ttmpc_num_penalty(const ttmpc_config *c) { return c->Ndynobs; }

static int make_devcfg(const ttmpc_config *c, DevCfg *g) {
  if (!c) return fail(TTMPC_ERR_BAD_CONFIG, "null config");
  if (c->nu != 2 || c->ns != 3 || c->nq != 10 || c->ndynobs != 6)
    return fail(TTMPC_ERR_BAD_CONFIG, "nu/ns/nq/ndynobs must be 2/3/10/6 (unicycle, mpc_generator.py layout)");
  if (c->N_hor < 1 || c->N_hor > 32) return fail(TTMPC_ERR_BAD_CONFIG, "N_hor must be in 1..32");
  if (c->nstcobs % 3 != 0 || c->nstcobs / 3 > MAX_EDGE || (c->Nstcobs > 0 && c->nstcobs < 3))
    return fail(TTMPC_ERR_BAD_CONFIG, "nstcobs must be 3*edges with edges <= 8");
  if (c->Nother < 0 || c->Nstcobs < 0 || c->Ndynobs < 0 || c->Ndynobs > 64 || c->Nother > 32 ||
      c->Nstcobs > 32)
    return fail(TTMPC_ERR_BAD_CONFIG, "obstacle counts out of range (Nother, Nstcobs <= 32, Ndynobs <= 64)");
  if (c->lbfgs_memory < 1 || c->lbfgs_memory > MAX_MEM)
    return fail(TTMPC_ERR_BAD_CONFIG, "lbfgs_memory must be in 1..16");
  if (c->max_inner_iterations < 1 || c->max_outer_iterations < 1 || !(c->ts > 0.0))
    return fail(TTMPC_ERR_BAD_CONFIG, "iteration limits and ts must be positive");
  const int N = c->N_hor;
  g->N = N; g->Nother = c->Nother; g->Nstc = c->Nstcobs; g->nstcobs = c->nstcobs;
  g->ne = c->nstcobs / 3; g->Ndyn = c->Ndynobs; g->mem = c->lbfgs_memory;
  g->max_inner = c->max_inner_iterations; g->max_outer = c->max_outer_iterations;
  g->max_ns = c->max_duration_ms > 0 ? (unsigned long long)c->max_duration_ms * 1000000ull : 0ull;
  g->off_s = 0; g->off_q = 2 * c->ns + c->nu; g->off_r = g->off_q + c->nq;
  g->off_vref = g->off_r + c->ns * N; g->off_c = g->off_vref + N;
  g->off_os = g->off_c + c->ns * N * c->Nother;
  g->off_od = g->off_os + c->Nstcobs * c->nstcobs;
  g->off_qdyn = g->off_od + c->Ndynobs * c->ndynobs * N + N;
  g->np = g->off_qdyn + N;
  g->smem_per_warp = smem_bytes_per_warp(N, g->Nother, g->Nstc, g->nstcobs, g->Ndyn, g->mem);
  {
    // 2 scenes per CTA (default shapes: 4 CTAs per SM of the unrolled build at 255 registers per thread,
    // 6 of the rolled build at 168; each owner has one potential helper).  Small CTAs release their SM
    // share as soon as both scenes are done, which is what lets the next batch in (batches in flight:
    // +4 % over 4 scenes per CTA, same time for a batch alone).  Large configurations: one scene per CTA
    // if two do not fit.
    const size_t cap = 232448 - 256;
    if ((size_t)g->smem_per_warp > cap)
      return fail(TTMPC_ERR_UNSUPPORTED, "configuration does not fit in shared memory: " +
                  std::to_string(g->smem_per_warp) + " bytes of tables per scene, 227 KB per SM");
    // larger tables: the CTA size (2, 3, 4, else 1 scene) that keeps the most scenes resident per SM
    int wpb = 1, best = 0;
    for (int cand : {2, 3, 4, 1}) {
      const size_t per_cta = (size_t)g->smem_per_warp * cand + 96 + 1024;  // + CtaHelp + the 1 KB the driver reserves per CTA
      if ((size_t)g->smem_per_warp * cand > cap) continue;
      // 8 warps per SM: the register limit of the unrolled build (255 registers).  Both builds launch
      // this CTA size, and the unrolled one, which serves batches that fit its resident warps, must
      // not lose warps; the rolled build then holds as many of these CTAs as its 168 registers and
      // the shared memory allow (6 for the default shapes).
      const int ctas = (int)std::min<size_t>(233472 / per_cta, (size_t)(8 / cand));
      if (ctas * cand > best) { best = ctas * cand; wpb = cand; }
    }
    g->warps_per_block = wpb;
  }
  g->ts = c->ts; g->inv_ts = 1.0 / c->ts; g->h6 = c->ts / 6.0; g->veh_d2 = c->vehicle_width * c->vehicle_width; g->margin = c->social_margin;
  g->vmin = c->lin_vel_min; g->vmax = c->lin_vel_max; g->wmax = c->ang_vel_max;
  g->amin = c->lin_acc_min; g->amax = c->lin_acc_max; g->awmax = c->ang_acc_max;
  g->tol = c->tolerance; g->init_tol = c->initial_tolerance; g->delta_tol = c->delta_tolerance;
  g->c0 = c->initial_penalty; g->pen_factor = c->penalty_update_factor;
  g->tol_factor = c->inner_tolerance_update_factor; g->suff_dec = c->sufficient_decrease_coeff;
  return TTMPC_OK;
}

// ---------------------------------------------------------------- per-device workspace
// A Slot is everything ONE in-flight solve owns: the scene queue counter, the running average
// behind the early helpers, the dispatch order, the per-warp dynamic-obstacle tables and (host
// path) the streams, the `ready` counter and the staging buffers.  Solves issued on different
// CUDA streams (device path) or from different host threads (host path) get different slots, so
// consecutive batches can overlap on the GPU: the CTAs of batch k+1 become resident as the CTAs
// of batch k drain, and the tail of one batch (a handful of long scenes) is filled with the
// bulk of the next.  Solves on one stream are ordered by the stream and share a slot.
struct Slot {
  bool keyed = false;              // device path: bound to `key`
  cudaStream_t key = nullptr;
  bool host = false, host_busy = false;  // host path: taken by one ttmpc_solve_batch_host call at a time
  double *dyn_scratch = nullptr; size_t dyn_bytes = 0;
  int *work_counter = nullptr;
  unsigned long long *run_stats = nullptr;  // [0] evaluations, [1] finished scenes of the running launch
  int *ready = nullptr;           // device counter of scenes already copied (host path) + time-out flag
  int *h_ready = nullptr;         // pinned: one value per chunk
  cudaStream_t copy_stream = nullptr, exec_stream = nullptr;
  cudaEvent_t ev_inputs = nullptr;
  cudaEvent_t ev_done = nullptr;  // blocking-sync event: the host thread sleeps instead of spinning
  int *order = nullptr; size_t order_ints = 0;  // dispatch order + ranking scratch
  // device staging for the host API
  void *dbuf = nullptr; size_t dbytes = 0;
  void *hbuf = nullptr; size_t hbytes = 0;
};
constexpr int MAX_STREAM_SLOTS = 16, MAX_HOST_SLOTS = 8;
struct Workspace {
  int device = -1;
  int sm_count = 0;
  unsigned long long *stats = nullptr;  // 24 x u64, shared by every slot (atomics)
  std::vector<Slot *> slots;
};
static std::mutex g_mu;
static std::condition_variable g_cv;
static std::vector<Workspace> g_ws;

static int get_ws(Workspace **out) {
  int dev = 0;
  CUDA_TRY(cudaGetDevice(&dev));
  for (auto &w : g_ws)
    if (w.device == dev) { *out = &w; return TTMPC_OK; }
  Workspace w;
  w.device = dev;
  CUDA_TRY(cudaDeviceGetAttribute(&w.sm_count, cudaDevAttrMultiProcessorCount, dev));
  CUDA_TRY(cudaMalloc(&w.stats, 192));
  CUDA_TRY(cudaMemset(w.stats, 0, 192));
  g_ws.reserve(16);
  g_ws.push_back(w);
  *out = &g_ws.back();
  return TTMPC_OK;
}
static int new_slot(Workspace *w, Slot **out) {
  Slot *s = new Slot();
  CUDA_TRY(cudaMalloc(&s->work_counter, 64));
  CUDA_TRY(cudaMalloc(&s->run_stats, 64));
  CUDA_TRY(cudaMemset(s->run_stats, 0, 64));
  CUDA_TRY(cudaMalloc(&s->ready, 64));
  w->slots.push_back(s);
  *out = s;
  return TTMPC_OK;
}
// device path: the slot of this stream (g_mu held).  Bindings are kept while they fit; when a 17th
// stream shows up the device is drained once and every binding is dropped (streams come and go --
// a destroyed stream cannot be told from an idle one -- and an unbound slot keeps its buffers).
static int slot_for_stream(Workspace *w, cudaStream_t st, Slot **out) {
  for (int pass = 0; pass < 2; pass++) {
    int device_slots = 0;
    Slot *free_slot = nullptr;
    for (Slot *s : w->slots) {
      if (s->host) continue;
      device_slots++;
      if (s->keyed && s->key == st) { *out = s; return TTMPC_OK; }
      if (!s->keyed && !free_slot) free_slot = s;
    }
    if (!free_slot && device_slots < MAX_STREAM_SLOTS) {
      int rc = new_slot(w, &free_slot);
      if (rc) return rc;
    }
    if (free_slot) {
      free_slot->keyed = true; free_slot->key = st;
      *out = free_slot;
      return TTMPC_OK;
    }
    CUDA_TRY(cudaDeviceSynchronize());
    for (Slot *s : w->slots)
      if (!s->host) s->keyed = false;
  }
  return fail(TTMPC_ERR_CUDA, "no scene-queue slot for this stream");
}
// host path: a free host slot (waits when MAX_HOST_SLOTS calls are already in flight)
static int acquire_host_slot(Workspace **wout, Slot **out, int *busy_calls) {
  std::unique_lock<std::mutex> lk(g_mu);
  Workspace *w;
  int rc = get_ws(&w);
  if (rc) return rc;
  *wout = w;
  while (true) {
    int hosts = 0, busy = 1;
    for (Slot *s : w->slots) busy += (s->host && s->host_busy) ? 1 : 0;
    *busy_calls = busy;
    for (Slot *s : w->slots) {
      if (!s->host) continue;
      hosts++;
      if (!s->host_busy) { s->host_busy = true; *out = s; return TTMPC_OK; }
    }
    if (hosts < MAX_HOST_SLOTS) break;
    g_cv.wait(lk);
  }
  Slot *s;
  rc = new_slot(w, &s);
  if (rc) return rc;
  // a slot becomes a host slot only once everything it needs exists (a half-built one stays an
  // unbound device slot, which needs none of this)
  cudaError_t e = cudaHostAlloc(&s->h_ready, sizeof(int) * 4096, cudaHostAllocDefault);
  if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&s->copy_stream, cudaStreamNonBlocking);
  if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&s->exec_stream, cudaStreamNonBlocking);
  if (e == cudaSuccess) e = cudaEventCreateWithFlags(&s->ev_inputs, cudaEventDisableTiming);
  if (e == cudaSuccess) e = cudaEventCreateWithFlags(&s->ev_done, cudaEventDisableTiming | cudaEventBlockingSync);
  if (e != cudaSuccess)
    return fail(TTMPC_ERR_CUDA, std::string("host path: streams / pinned memory of a new slot: ") + cudaGetErrorString(e));
  s->host = true; s->host_busy = true;
  *out = s;
  return TTMPC_OK;
}
namespace {
struct HostSlotLease {  // returns the slot when the host call ends, whatever the exit path
  Slot *s = nullptr;
  bool clean = false;  // the call reached its end: both streams are known to be idle
  ~HostSlotLease() {
    if (!s) return;
    if (!clean) {
      // error exit: the gated kernel may still be waiting for chunks (it gives up after 2 s) and
      // writing into the slot's buffers, copies may be in flight.  Nobody may reuse or free those
      // buffers before the slot's streams have drained.
      if (s->copy_stream) cudaStreamSynchronize(s->copy_stream);
      if (s->exec_stream) cudaStreamSynchronize(s->exec_stream);
      cudaGetLastError();  // the failure was already reported to the caller
    }
    { std::lock_guard<std::mutex> lk(g_mu); s->host_busy = false; }
    g_cv.notify_one();
  }
};
}  // namespace
// Wait for a stream of the host path.  Large batches take milliseconds: the thread sleeps on a
// blocking-sync event (several calls are usually in flight, one spinning thread each would eat the
// cores the other ranks and the staging threads need); small batches spin for the lowest latency.
static int wait_stream(Slot *s, cudaStream_t st, int n_scenes) {
  if (n_scenes < 512) { CUDA_TRY(cudaStreamSynchronize(st)); return TTMPC_OK; }
  CUDA_TRY(cudaEventRecord(s->ev_done, st));
  CUDA_TRY(cudaEventSynchronize(s->ev_done));
  return TTMPC_OK;
}
static int ensure_dyn(Slot *w, size_t bytes) {
  if (bytes <= w->dyn_bytes) return TTMPC_OK;
  if (w->dyn_scratch) CUDA_TRY(cudaFree(w->dyn_scratch));
  w->dyn_scratch = nullptr; w->dyn_bytes = 0;
  CUDA_TRY(cudaMalloc(&w->dyn_scratch, bytes));
  w->dyn_bytes = bytes;
  return TTMPC_OK;
}
static int ensure_order(Slot *w, size_t ints) {
  if (ints <= w->order_ints) return TTMPC_OK;
  if (w->order) CUDA_TRY(cudaFree(w->order));
  w->order = nullptr; w->order_ints = 0;
  CUDA_TRY(cudaMalloc(&w->order, ints * sizeof(int)));
  w->order_ints = ints;
  return TTMPC_OK;
}
static int ensure_staging(Slot *w, size_t bytes) {
  if (bytes > w->dbytes) {
    if (w->dbuf) CUDA_TRY(cudaFree(w->dbuf));
    w->dbuf = nullptr; w->dbytes = 0;
    CUDA_TRY(cudaMalloc(&w->dbuf, bytes));
    // the fields of the result block are padded apart and come back in ONE device-to-host copy:
    // define the padding once (compute-sanitizer initcheck reads the copy source).  ON THE SLOT'S COPY
    // STREAM: the slot's streams are non-blocking, a memset on the legacy stream is not ordered with
    // them and would race the input copies that follow (it did: zeroed parameter chunks).  The exec
    // stream waits for ev_inputs, which is recorded on the copy stream after this.
    if (w->copy_stream) CUDA_TRY(cudaMemsetAsync(w->dbuf, 0, bytes, w->copy_stream));
    else { CUDA_TRY(cudaMemset(w->dbuf, 0, bytes)); CUDA_TRY(cudaDeviceSynchronize()); }
    w->dbytes = bytes;
  }
  if (bytes > w->hbytes) {
    if (w->hbuf) CUDA_TRY(cudaFreeHost(w->hbuf));
    w->hbuf = nullptr; w->hbytes = 0;
    CUDA_TRY(cudaHostAlloc(&w->hbuf, bytes, cudaHostAllocDefault));
    w->hbytes = bytes;
  }
  return TTMPC_OK;
}

static int grid_for_occupancy(Workspace *w, const DevCfg &g, int n_scenes, int bps, int *grid) {
  if (bps < 1) return fail(TTMPC_ERR_UNSUPPORTED, "configuration does not fit in shared memory");
  long long want = ((long long)n_scenes + g.warps_per_block - 1) / g.warps_per_block;
  long long cap = (long long)w->sm_count * bps;
  *grid = (int)(want < cap ? (want < 1 ? 1 : want) : cap);
  return TTMPC_OK;
}
static int grid_for(Workspace *w, const DevCfg &g, int n_scenes, int *grid) {
  int bps = 0;
  CUDA_TRY(solve_occupancy(g, &bps));
  return grid_for_occupancy(w, g, n_scenes, bps, grid);
}
// Two builds of the solve kernel, bit-identical results: unrolled hot loops (255 registers) when every
// scene has a warp from the start (latency-bound), rolled loops (168 registers, more resident warps:
// 12 per SM for the default shapes) when the batch queues behind the unrolled build's resident warps.
// The grid is sized from the occupancy of the build that runs.  TTMPC_CODE=small|unrolled forces one.
struct SolvePlan { int grid, blocks_per_sm; bool small_code; };
static int plan_solve(Workspace *w, const DevCfg &g, int n_scenes, SolvePlan *pl) {
  int bps = 0, grid = 0;
  CUDA_TRY(solve_occupancy(g, &bps));
  int rc = grid_for_occupancy(w, g, n_scenes, bps, &grid);
  if (rc) return rc;
  bool small_code = n_scenes > (long long)grid * g.warps_per_block;
  if (const char *e = std::getenv("TTMPC_CODE")) {
    if (e[0] == 's') small_code = true;
    else if (e[0] == 'u') small_code = false;
  }
  if (small_code) {
    CUDA_TRY(solve_occupancy_small(g, &bps));
    rc = grid_for_occupancy(w, g, n_scenes, bps, &grid);
    if (rc) return rc;
  }
  pl->grid = grid; pl->blocks_per_sm = bps; pl->small_code = small_code;
  return TTMPC_OK;
}

static int solve_device_impl(const ttmpc_config *cfg, int n_scenes, const double *d_p, int use_u0,
                             int use_y0, const double *d_c0, const ttmpc_result *res,
                             cudaStream_t st, Slot *host_slot, bool gated);

extern "C" int ttmpc_solve_batch_device(const ttmpc_config *cfg, int n_scenes, const double *d_p,
                                        int use_u0, int use_y0, const double *d_c0,
                                        const ttmpc_result *res, void *stream) {
  return solve_device_impl(cfg, n_scenes, d_p, use_u0, use_y0, d_c0, res, (cudaStream_t)stream, nullptr, false);
}

static int solve_device_impl(const ttmpc_config *cfg, int n_scenes, const double *d_p, int use_u0,
                             int use_y0, const double *d_c0, const ttmpc_result *res,
                             cudaStream_t st, Slot *host_slot, bool gated) {
  DevCfg g;
  int rc = make_devcfg(cfg, &g);
  if (rc) return rc;
  if (n_scenes < 0 || !res || !res->u || (n_scenes > 0 && !d_p))
    return fail(TTMPC_ERR_BAD_ARG, "n_scenes >= 0, d_p and res->u are required");
  if (n_scenes == 0) return TTMPC_OK;
  // The process-wide lock covers the bookkeeping only (workspace, the stream's slot, growing the
  // slot's scratch buffers); the memsets and launches below run outside it, so several host threads
  // / streams issue their solves concurrently.  One slot is used by one stream (or one host lease).
  Workspace *w;
  Slot *sl = host_slot;
  const int *d_ready = (host_slot && gated) ? host_slot->ready : nullptr;
  SolvePlan plan;
  bool want_order = false;
  {
    std::lock_guard<std::mutex> lk(g_mu);
    rc = get_ws(&w);
    if (rc) return rc;
    // host path: the caller's slot (streamed inputs gated by its `ready` counter); device path:
    // the slot of the stream
    if (!sl) { rc = slot_for_stream(w, st, &sl); if (rc) return rc; }
    rc = plan_solve(w, g, n_scenes, &plan);
    if (rc) return rc;
    const size_t table = (size_t)DYN_FIELDS * g.Ndyn * g.N * sizeof(double);
    rc = ensure_dyn(sl, (table ? table : 8) * (size_t)plan.grid * g.warps_per_block);
    if (rc) return rc;
    // more scenes than resident warps: dispatch the likely-long ones first.  Not on the streamed
    // host path (scenes become available in index order there).
    want_order = !d_ready && n_scenes > (long long)plan.grid * g.warps_per_block;
    if (want_order) {
      rc = ensure_order(sl, 2 * (size_t)n_scenes + 64);
      if (rc) return rc;
    }
  }
  CUDA_TRY(cudaMemsetAsync(sl->work_counter, 0, sizeof(int), st));
  const char *nh = std::getenv("TTMPC_NO_HELPERS");
  SolveArgs A;
  A.eprof = w->stats + 8;  // stats block is 24 x u64: [0..7] counters, [8..17] eval sections
  A.helpers = (nh && nh[0] == '1') ? 0 : 1;  // TTMPC_NO_HELPERS=1 disables the tail helpers
  A.ready = d_ready; A.timeout_flag = d_ready ? sl->ready + 1 : nullptr;
  A.p = d_p; A.c0 = d_c0; A.u = res->u; A.y = res->y; A.cost = res->cost;
  A.last_fpr = res->last_fpr; A.f1_infeas = res->f1_infeas; A.f2_norm = res->f2_norm;
  A.penalty = res->penalty; A.exit_status = res->exit_status; A.outer_iters = res->outer_iters;
  A.inner_iters = res->inner_iters; A.pred_states = res->pred_states; A.evals = res->evals;
  A.dyn_scratch = sl->dyn_scratch; A.work_counter = sl->work_counter; A.stats = w->stats;
  A.run_stats = sl->run_stats;  // [0] evaluations, [1] count of finished scenes of this launch
  // the running average behind the early-helper threshold is per launch (workloads differ by 30x)
  CUDA_TRY(cudaMemsetAsync(A.run_stats, 0, 2 * sizeof(unsigned long long), st));
  A.n_scenes = n_scenes; A.use_u0 = use_u0; A.use_y0 = use_y0;
  A.order = nullptr;
  if (want_order) {
    CUDA_TRY(launch_rank_scenes(g, d_p, n_scenes, sl->order + n_scenes, sl->order, st));
    A.order = sl->order;
  }
  if (plan.small_code) CUDA_TRY(launch_solve_small(g, A, plan.grid, st));
  else CUDA_TRY(launch_solve(g, A, plan.grid, st));
  return TTMPC_OK;
}

// ------------------------------------------------------------------ fleet step
static int fleet_dims(const ttmpc_config *cfg, const ttmpc_fleet *f, FleetDims *d) {
  DevCfg g;
  int rc = make_devcfg(cfg, &g);
  if (rc) return rc;
  if (!f || f->n < 0) return fail(TTMPC_ERR_BAD_ARG, "fleet: null or n < 0");
  if (f->n > 0 && (!f->state || !f->goal || !f->last_u || !f->idx_ref || !f->status || !f->ref_traj ||
                   !f->ref_len || !f->stc))
    return fail(TTMPC_ERR_BAD_ARG, "fleet: state, goal, last_u, idx_ref, status, ref_traj, ref_len, stc are required");
  if (f->action_steps != 1) return fail(TTMPC_ERR_UNSUPPORTED, "fleet: only action_steps = 1 is supported");
  if (f->ref_stride < 1) return fail(TTMPC_ERR_BAD_ARG, "fleet: ref_stride must be >= 1");
  if (f->dyn_cur && (!f->dyn_last || !f->dyn_disp || f->n_dyn_live < 0 || f->n_dyn_live > cfg->Ndynobs))
    return fail(TTMPC_ERR_BAD_ARG, "fleet: dyn_cur needs dyn_last, dyn_disp and 0 <= n_dyn_live <= Ndynobs");
  d->N = cfg->N_hor; d->np = g.np; d->ts = cfg->ts;
  d->n_other = cfg->ns * cfg->N_hor * cfg->Nother;
  d->n_stc = cfg->Nstcobs * cfg->nstcobs;
  d->n_dyn = cfg->Ndynobs * cfg->ndynobs * cfg->N_hor;
  return TTMPC_OK;
}
extern "C" int ttmpc_fleet_pack_device(const ttmpc_config *cfg, const ttmpc_fleet *fleet, double *d_p,
                                       void *stream) {
  FleetDims d;
  int rc = fleet_dims(cfg, fleet, &d);
  if (rc) return rc;
  if (fleet->n == 0) return TTMPC_OK;
  if (!d_p) return fail(TTMPC_ERR_BAD_ARG, "fleet: d_p is required");
  CUDA_TRY(launch_fleet_pack(*fleet, d, d_p, (cudaStream_t)stream));
  return TTMPC_OK;
}
extern "C" int ttmpc_fleet_advance_device(const ttmpc_config *cfg, const ttmpc_fleet *fleet,
                                          const double *d_u, const int *d_exit_status, void *stream) {
  FleetDims d;
  int rc = fleet_dims(cfg, fleet, &d);
  if (rc) return rc;
  if (fleet->n == 0) return TTMPC_OK;
  if (!d_u) return fail(TTMPC_ERR_BAD_ARG, "fleet: d_u is required");
  CUDA_TRY(launch_fleet_advance(*fleet, d, d_u, d_exit_status, (cudaStream_t)stream));
  return TTMPC_OK;
}
extern "C" int ttmpc_fleet_step_device(const ttmpc_config *cfg, const ttmpc_fleet *fleet, double *d_p,
                                       int use_y0, const ttmpc_result *res, void *stream) {
  if (!res || !res->u || !res->exit_status)
    return fail(TTMPC_ERR_BAD_ARG, "fleet: res->u and res->exit_status are required");
  int rc = ttmpc_fleet_pack_device(cfg, fleet, d_p, stream);
  if (rc) return rc;
  rc = ttmpc_solve_batch_device(cfg, fleet->n, d_p, 0, use_y0, nullptr, res, stream);
  if (rc) return rc;
  return ttmpc_fleet_advance_device(cfg, fleet, res->u, res->exit_status, stream);
}

// Cumulative device-side counters since the last reset:
// [0] cost-only evaluations [1] cost+gradient evaluations [2] dynamic-obstacle
// bodies executed [3] PANOC iterations; the TTMPC_PROFILE builds fill the rest of the
// 24 counters.  Reads the first `count`, resets all 24.  Synchronises the device.
static int read_stats(unsigned long long *out, int count, int reset) {
  std::lock_guard<std::mutex> lk(g_mu);
  Workspace *w;
  int rc = get_ws(&w);
  if (rc) return rc;
  CUDA_TRY(cudaDeviceSynchronize());
  CUDA_TRY(cudaMemcpy(out, w->stats, count * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
  if (reset) CUDA_TRY(cudaMemset(w->stats, 0, 192));
  return TTMPC_OK;
}
extern "C" int ttmpc_read_stats(unsigned long long out[4], int reset) { return read_stats(out, 4, reset); }
extern "C" int ttmpc_read_stats8(unsigned long long out[8], int reset) { return read_stats(out, 8, reset); }
extern "C" int ttmpc_read_stats24(unsigned long long out[24], int reset) { return read_stats(out, 24, reset); }

// Launch geometry the solve of an n_scenes batch would use, of the build that would run it (for
// DESIGN/bench reporting).
extern "C" int ttmpc_launch_info(const ttmpc_config *cfg, int n_scenes, int *grid, int *block,
                                 int *smem_bytes, int *blocks_per_sm, int *sm_count) {
  DevCfg g;
  int rc = make_devcfg(cfg, &g);
  if (rc) return rc;
  std::lock_guard<std::mutex> lk(g_mu);
  Workspace *w;
  rc = get_ws(&w);
  if (rc) return rc;
  SolvePlan plan;
  rc = plan_solve(w, g, n_scenes, &plan);
  if (rc) return rc;
  if (grid) *grid = plan.grid;
  if (block) *block = g.warps_per_block * 32;
  if (smem_bytes) *smem_bytes = g.smem_per_warp * g.warps_per_block;
  if (blocks_per_sm) *blocks_per_sm = plan.blocks_per_sm;
  if (sm_count) *sm_count = w->sm_count;
  return TTMPC_OK;
}

namespace {
struct Carver {
  char *d, *h; size_t off = 0;
  template <class T> void take(size_t n, T **dp, T **hp) {
    off = (off + 255) / 256 * 256;
    *dp = reinterpret_cast<T *>(d + off);
    *hp = reinterpret_cast<T *>(h + off);
    off += n * sizeof(T);
  }
};
}  // namespace

extern "C" int ttmpc_solve_batch_host(const ttmpc_config *cfg, int n, const double *h_p,
                                      int use_u0, int use_y0, const double *h_c0,
                                      const ttmpc_result *res) {
  DevCfg g;
  int rc = make_devcfg(cfg, &g);
  if (rc) return rc;
  if (n < 0 || !res || !res->u || (n > 0 && !h_p))
    return fail(TTMPC_ERR_BAD_ARG, "n >= 0, h_p and res->u are required");
  if (n == 0) return TTMPC_OK;
  const size_t nn = (size_t)n, nu = 2 * (size_t)g.N;
  size_t total = 4096 + 256 * 16 + sizeof(double) * (nn * g.np + nn + 2 * nn * nu + 5 * nn + nn * g.N * 3) +
                 sizeof(int) * 3 * nn + sizeof(long long) * 4 * nn;
  // every call owns a slot (staging buffers, two streams, `ready` counter) until it returns:
  // calls from several host threads overlap on the GPU
  Workspace *ws;
  Slot *w = nullptr;
  int busy_calls = 1;
  rc = acquire_host_slot(&ws, &w, &busy_calls);
  HostSlotLease lease{w};
  if (rc) return rc;
  rc = ensure_staging(w, total);
  if (rc) return rc;
  Carver cv{(char *)w->dbuf, (char *)w->hbuf};
  double *dp, *hp, *dc0, *hc0, *du, *hu, *dy, *hy, *dcost, *hcost, *dfpr, *hfpr, *df1, *hf1, *df2,
      *hf2, *dpen, *hpen, *dps, *hps;
  int *dex, *hex, *dout, *hout, *din, *hin;
  long long *dev, *hev;
  cv.take(nn * g.np, &dp, &hp);
  cv.take(nn, &dc0, &hc0);
  cv.take(nn * nu, &du, &hu);
  cv.take(nn * nu, &dy, &hy);
  cv.take(nn, &dcost, &hcost);
  cv.take(nn, &dfpr, &hfpr);
  cv.take(nn, &df1, &hf1);
  cv.take(nn, &df2, &hf2);
  cv.take(nn, &dpen, &hpen);
  cv.take(nn * g.N * 3, &dps, &hps);
  cv.take(nn, &dex, &hex);
  cv.take(nn, &dout, &hout);
  cv.take(nn, &din, &hin);
  cv.take(4 * nn, &dev, &hev);
  // Inputs stream in while the kernel already runs: small inputs first, then the parameter
  // block in chunks (host memcpy into pinned staging -> async H2D -> bump the device-side
  // `ready` counter); the persistent kernel waits on `ready` before it stages a scene.
  cudaStream_t cs = w->copy_stream, st = w->exec_stream;
  CUDA_TRY(cudaMemsetAsync(w->ready, 0, 2 * sizeof(int), cs));  // [0] ready count, [1] timeout flag
  if (h_c0) {
    std::memcpy(hc0, h_c0, sizeof(double) * nn);
    CUDA_TRY(cudaMemcpyAsync(dc0, hc0, sizeof(double) * nn, cudaMemcpyHostToDevice, cs));
  }
  if (use_u0) {
    std::memcpy(hu, res->u, sizeof(double) * nn * nu);
    CUDA_TRY(cudaMemcpyAsync(du, hu, sizeof(double) * nn * nu, cudaMemcpyHostToDevice, cs));
  }
  if (use_y0 && res->y) {
    std::memcpy(hy, res->y, sizeof(double) * nn * nu);
    CUDA_TRY(cudaMemcpyAsync(dy, hy, sizeof(double) * nn * nu, cudaMemcpyHostToDevice, cs));
  }
  CUDA_TRY(cudaEventRecord(w->ev_inputs, cs));
  CUDA_TRY(cudaStreamWaitEvent(st, w->ev_inputs, 0));
  ttmpc_result dres;
  std::memset(&dres, 0, sizeof(dres));
  dres.u = du; dres.y = res->y ? dy : nullptr; dres.cost = dcost; dres.exit_status = dex;
  dres.outer_iters = dout; dres.inner_iters = din; dres.last_fpr = dfpr; dres.f1_infeas = df1;
  dres.f2_norm = df2; dres.penalty = dpen; dres.pred_states = res->pred_states ? dps : nullptr;
  dres.evals = dev;
  // Streaming the parameters in behind the running kernel gives ONE call its lowest latency (the
  // kernel starts on the first chunk) but costs the dispatch order (scenes become available in
  // index order, the likely-long ones cannot go first).  When other host calls are already in
  // flight the GPU is busy anyway: copy everything, then launch with the dispatch order
  // (measured with six calls in flight: 511 k -> 528 k solves/s end to end; one call alone 21.2 ms
  // streamed, 22.3 ms unstreamed).  CUDA_LAUNCH_BLOCKING=1 turns streaming off, and is the only
  // switch that does.  It is not a tuning option: with launches serialised (launch-blocking
  // debugging, or a profiler that serialises kernels -- set it there too) no chunk is copied while
  // the gated kernel runs, and the kernel would wait out its 2 s time-out before the unstreamed re-run.
  const char *lb = std::getenv("CUDA_LAUNCH_BLOCKING");
  const bool stream_in = busy_calls <= 1 && !(lb && lb[0] == '1');
  if (stream_in) {
    rc = solve_device_impl(cfg, n, dp, use_u0, use_y0 && res->y, h_c0 ? dc0 : nullptr, &dres, st, w, true);
    if (rc) return rc;
  }
  // Pinned (page-locked) caller memory is copied from directly; pageable memory goes through the
  // slot's pinned staging buffer first (a host memcpy, ~10 GB/s per thread).
  cudaPointerAttributes at;
  const bool pinned_in = cudaPointerGetAttributes(&at, h_p) == cudaSuccess ? at.type == cudaMemoryTypeHost
                                                                           : (cudaGetLastError(), false);
  {
    int chunk = 256;
    while ((n + chunk - 1) / chunk > 4096) chunk *= 2;
    const int n_chunks = (n + chunk - 1) / chunk;
    // chunk ci: scenes up to s1, `cnt` parameters from element `off` of the block
    struct Chunk { int s1; size_t off, cnt; };
    auto chunk_at = [&](int ci) {
      const int s0 = ci * chunk, s1 = std::min(s0 + chunk, n);
      return Chunk{s1, (size_t)s0 * g.np, (size_t)(s1 - s0) * g.np};
    };
    // The copy into pinned staging is host-memory bound and the kernel cannot run ahead of it: a
    // few worker threads stage the chunks (chunk i by thread i mod T), this thread issues the H2D
    // copies in order as the chunks become ready.  The team shrinks when several calls are in
    // flight (TTMPC_HOST_THREADS = thread budget of this process, default half the cores).
    const unsigned hw = std::thread::hardware_concurrency();
    int budget = (int)(hw ? hw / 2 : 1);
    if (const char *e = std::getenv("TTMPC_HOST_THREADS")) { const int v = std::atoi(e); if (v >= 1) budget = v; }
    const int T = pinned_in ? 1 : std::max(1, std::min({8, budget / std::max(1, busy_calls), n_chunks}));
    const double *src = pinned_in ? h_p : hp;
    std::vector<std::atomic<int>> staged(n_chunks);
    for (auto &f : staged) f.store(pinned_in ? 1 : 0, std::memory_order_relaxed);
    auto stage = [&](int ci) {
      const Chunk c = chunk_at(ci);
      std::memcpy(hp + c.off, h_p + c.off, sizeof(double) * c.cnt);
      staged[ci].store(1, std::memory_order_release);
    };
    std::vector<std::thread> workers;
    for (int t = 1; t < T; t++)
      workers.emplace_back([&, t] { for (int ci = t; ci < n_chunks; ci += T) stage(ci); });
    int rc_copy = TTMPC_OK;
    int mine = 0;  // next chunk this thread stages itself (thread 0's share)
    for (int ci = 0; ci < n_chunks; ci++) {
      while (!staged[ci].load(std::memory_order_acquire)) {
        if (mine < n_chunks) { stage(mine); mine += T; }  // do own share while waiting
        else std::this_thread::yield();
      }
      if (rc_copy != TTMPC_OK) continue;
      const Chunk c = chunk_at(ci);
      w->h_ready[ci] = c.s1;
      if (cudaMemcpyAsync(dp + c.off, src + c.off, sizeof(double) * c.cnt, cudaMemcpyHostToDevice, cs) != cudaSuccess ||
          cudaMemcpyAsync(w->ready, w->h_ready + ci, sizeof(int), cudaMemcpyHostToDevice, cs) != cudaSuccess)
        rc_copy = TTMPC_ERR_CUDA;
    }
    for (auto &th : workers) th.join();
    if (rc_copy != TTMPC_OK) return fail(TTMPC_ERR_CUDA, "host path: asynchronous copy of the parameter block failed");
  }
  int timed_out = 0;
  if (stream_in) {
    rc = wait_stream(w, st, n);
    if (rc) return rc;
    CUDA_TRY(cudaMemcpy(&timed_out, w->ready + 1, sizeof(int), cudaMemcpyDeviceToHost));
  }
  if (!stream_in || timed_out) {  // unstreamed (re-)run: all inputs are resident now
    rc = wait_stream(w, cs, n);
    if (rc) return rc;
    if (use_u0) CUDA_TRY(cudaMemcpyAsync(du, hu, sizeof(double) * nn * nu, cudaMemcpyHostToDevice, st));
    if (use_y0 && res->y) CUDA_TRY(cudaMemcpyAsync(dy, hy, sizeof(double) * nn * nu, cudaMemcpyHostToDevice, st));
    rc = solve_device_impl(cfg, n, dp, use_u0, use_y0 && res->y, h_c0 ? dc0 : nullptr, &dres, st, w, false);
    if (rc) return rc;
  }
  // one contiguous D2H of everything after the inputs
  const size_t out_begin = (size_t)((char *)du - (char *)w->dbuf);
  CUDA_TRY(cudaMemcpyAsync((char *)w->hbuf + out_begin, (char *)w->dbuf + out_begin, cv.off - out_begin,
                           cudaMemcpyDeviceToHost, st));
  rc = wait_stream(w, st, n);
  if (rc) return rc;
  std::memcpy(res->u, hu, sizeof(double) * nn * nu);
  if (res->y) std::memcpy(res->y, hy, sizeof(double) * nn * nu);
  if (res->cost) std::memcpy(res->cost, hcost, sizeof(double) * nn);
  if (res->last_fpr) std::memcpy(res->last_fpr, hfpr, sizeof(double) * nn);
  if (res->f1_infeas) std::memcpy(res->f1_infeas, hf1, sizeof(double) * nn);
  if (res->f2_norm) std::memcpy(res->f2_norm, hf2, sizeof(double) * nn);
  if (res->penalty) std::memcpy(res->penalty, hpen, sizeof(double) * nn);
  if (res->pred_states) std::memcpy(res->pred_states, hps, sizeof(double) * nn * g.N * 3);
  if (res->exit_status) std::memcpy(res->exit_status, hex, sizeof(int) * nn);
  if (res->outer_iters) std::memcpy(res->outer_iters, hout, sizeof(int) * nn);
  if (res->inner_iters) std::memcpy(res->inner_iters, hin, sizeof(int) * nn);
  if (res->evals) std::memcpy(res->evals, hev, sizeof(long long) * 4 * nn);
  lease.clean = true;
  return TTMPC_OK;
}

extern "C" int ttmpc_eval_batch_device(const ttmpc_config *cfg, int n, const double *d_p,
                                       const double *d_u, const double *d_c, const double *d_y,
                                       double *d_f, double *d_F1, double *d_F2, double *d_psi,
                                       double *d_grad, void *stream) {
  DevCfg g;
  int rc = make_devcfg(cfg, &g);
  if (rc) return rc;
  if (n < 0 || (n > 0 && (!d_p || !d_u))) return fail(TTMPC_ERR_BAD_ARG, "d_p and d_u are required");
  if (n == 0) return TTMPC_OK;
  std::lock_guard<std::mutex> lk(g_mu);
  Workspace *w;
  rc = get_ws(&w);
  if (rc) return rc;
  int grid;
  rc = grid_for(w, g, n, &grid);
  if (rc) return rc;
  const size_t table = (size_t)DYN_FIELDS * g.Ndyn * g.N * sizeof(double);
  Slot *sl;
  rc = slot_for_stream(w, (cudaStream_t)stream, &sl);
  if (rc) return rc;
  rc = ensure_dyn(sl, (table ? table : 8) * (size_t)grid * g.warps_per_block);
  if (rc) return rc;
  EvalArgs A;
  A.p = d_p; A.u = d_u; A.c = d_c; A.y = d_y; A.f = d_f; A.F1 = d_F1; A.F2 = d_F2; A.psi = d_psi;
  A.grad = d_grad; A.dyn_scratch = sl->dyn_scratch; A.n_scenes = n;
  CUDA_TRY(launch_eval(g, A, grid, (cudaStream_t)stream));
  return TTMPC_OK;
}

extern "C" int ttmpc_eval_batch_host(const ttmpc_config *cfg, int n, const double *h_p,
                                     const double *h_u, const double *h_c, const double *h_y,
                                     double *h_f, double *h_F1, double *h_F2, double *h_psi,
                                     double *h_grad) {
  DevCfg g;
  int rc = make_devcfg(cfg, &g);
  if (rc) return rc;
  if (n < 0 || (n > 0 && (!h_p || !h_u))) return fail(TTMPC_ERR_BAD_ARG, "h_p and h_u are required");
  if (n == 0) return TTMPC_OK;
  const size_t nn = (size_t)n, nu = 2 * (size_t)g.N;
  double *dp = nullptr, *du = nullptr, *dc = nullptr, *dy = nullptr, *df = nullptr, *dF1 = nullptr,
         *dF2 = nullptr, *dpsi = nullptr, *dgrad = nullptr;
  auto cleanup = [&]() {
    cudaFree(dp); cudaFree(du); cudaFree(dc); cudaFree(dy); cudaFree(df); cudaFree(dF1);
    cudaFree(dF2); cudaFree(dpsi); cudaFree(dgrad);
  };
#define TRY_OR_CLEAN(x) do { cudaError_t e__ = (x); if (e__ != cudaSuccess) { cleanup(); return fail(TTMPC_ERR_CUDA, std::string(#x) + ": " + cudaGetErrorString(e__)); } } while (0)
  TRY_OR_CLEAN(cudaMalloc(&dp, sizeof(double) * nn * g.np));
  TRY_OR_CLEAN(cudaMalloc(&du, sizeof(double) * nn * nu));
  TRY_OR_CLEAN(cudaMalloc(&dc, sizeof(double) * nn));
  TRY_OR_CLEAN(cudaMalloc(&dy, sizeof(double) * nn * nu));
  TRY_OR_CLEAN(cudaMalloc(&df, sizeof(double) * nn));
  TRY_OR_CLEAN(cudaMalloc(&dF1, sizeof(double) * nn * nu));
  TRY_OR_CLEAN(cudaMalloc(&dF2, sizeof(double) * nn * (g.Ndyn > 0 ? g.Ndyn : 1)));
  TRY_OR_CLEAN(cudaMalloc(&dpsi, sizeof(double) * nn));
  TRY_OR_CLEAN(cudaMalloc(&dgrad, sizeof(double) * nn * nu));
  TRY_OR_CLEAN(cudaMemcpy(dp, h_p, sizeof(double) * nn * g.np, cudaMemcpyHostToDevice));
  TRY_OR_CLEAN(cudaMemcpy(du, h_u, sizeof(double) * nn * nu, cudaMemcpyHostToDevice));
  if (h_c) TRY_OR_CLEAN(cudaMemcpy(dc, h_c, sizeof(double) * nn, cudaMemcpyHostToDevice));
  if (h_y) TRY_OR_CLEAN(cudaMemcpy(dy, h_y, sizeof(double) * nn * nu, cudaMemcpyHostToDevice));
  rc = ttmpc_eval_batch_device(cfg, n, dp, du, h_c ? dc : nullptr, h_y ? dy : nullptr, df, dF1, dF2,
                               dpsi, dgrad, 0);
  if (rc) { cleanup(); return rc; }
  TRY_OR_CLEAN(cudaDeviceSynchronize());
  if (h_f) TRY_OR_CLEAN(cudaMemcpy(h_f, df, sizeof(double) * nn, cudaMemcpyDeviceToHost));
  if (h_F1) TRY_OR_CLEAN(cudaMemcpy(h_F1, dF1, sizeof(double) * nn * nu, cudaMemcpyDeviceToHost));
  if (h_F2 && g.Ndyn) TRY_OR_CLEAN(cudaMemcpy(h_F2, dF2, sizeof(double) * nn * g.Ndyn, cudaMemcpyDeviceToHost));
  if (h_psi) TRY_OR_CLEAN(cudaMemcpy(h_psi, dpsi, sizeof(double) * nn, cudaMemcpyDeviceToHost));
  if (h_grad) TRY_OR_CLEAN(cudaMemcpy(h_grad, dgrad, sizeof(double) * nn * nu, cudaMemcpyDeviceToHost));
  cleanup();
  return TTMPC_OK;
}

// Latency probe (diagnostics): h_p = one scene's parameters (host); out[8] cycles of
// {cost eval, grad eval, wsum, lbfgs apply (mem pairs), div, sqrt, dfma, checksum}.
extern "C" int ttmpc_probe_latency(const ttmpc_config *cfg, const double *h_p, long long out[8], int reps) {
  DevCfg g;
  int rc = make_devcfg(cfg, &g);
  if (rc) return rc;
  double *dp = nullptr, *dyn = nullptr; long long *dout = nullptr;
  CUDA_TRY(cudaMalloc(&dp, sizeof(double) * g.np));
  CUDA_TRY(cudaMalloc(&dyn, sizeof(double) * DYN_FIELDS * (g.Ndyn > 0 ? g.Ndyn : 1) * g.N));
  CUDA_TRY(cudaMalloc(&dout, 64));
  CUDA_TRY(cudaMemcpy(dp, h_p, sizeof(double) * g.np, cudaMemcpyHostToDevice));
  CUDA_TRY(launch_probe(g, dp, dyn, dout, reps, 0));
  CUDA_TRY(cudaDeviceSynchronize());
  CUDA_TRY(cudaMemcpy(out, dout, 64, cudaMemcpyDeviceToHost));
  cudaFree(dp); cudaFree(dyn); cudaFree(dout);
  return TTMPC_OK;
}

extern "C" int ttmpc_measure_fp64_peak(double *tflops, void *stream) {
  if (!tflops) return fail(TTMPC_ERR_BAD_ARG, "null output");
  int dev = 0, sms = 0;
  CUDA_TRY(cudaGetDevice(&dev));
  CUDA_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  const int threads = 256, blocks = sms * 8, iters = 1 << 15;
  double *out = nullptr;
  CUDA_TRY(cudaMalloc(&out, sizeof(double) * threads * blocks));
  cudaStream_t st = (cudaStream_t)stream;
  cudaEvent_t e0, e1;
  CUDA_TRY(cudaEventCreate(&e0));
  CUDA_TRY(cudaEventCreate(&e1));
  double best = 0.0;
  for (int rep = 0; rep < 4; rep++) {
    CUDA_TRY(cudaEventRecord(e0, st));
    CUDA_TRY(launch_fp64_peak(out, blocks, threads, iters, st));
    CUDA_TRY(cudaEventRecord(e1, st));
    CUDA_TRY(cudaEventSynchronize(e1));
    float ms = 0;
    CUDA_TRY(cudaEventElapsedTime(&ms, e0, e1));
    double fl = 2.0 * 8.0 * (double)iters * threads * blocks;
    double tf = fl / (ms * 1e-3) / 1e12;
    if (rep > 0 && tf > best) best = tf;
  }
  cudaEventDestroy(e0); cudaEventDestroy(e1); cudaFree(out);
  *tflops = best;
  return TTMPC_OK;
}
