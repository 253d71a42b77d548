// c_api.cu -- the extern "C" surface declared in include/rbg_b200.h:
// argument validation, error reporting, launch sequencing, and the
// host-buffer variants (pipelined H2D -> kernels -> D2H over env slices).
#include <stdarg.h>
#include <stdio.h>
#include <string.h>

#include <atomic>
#include <chrono>
#include <mutex>
#include <unordered_map>
#include <vector>

#include "rbg_host.h"

namespace rbg {

static thread_local char g_err[512] = "";
static std::atomic<long long> g_launches{0};

int set_error(int code, const char *fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}

int set_cuda_error(cudaError_t e, const char *what) {
  return set_error(RBG_ECUDA, "%s: %s", what, cudaGetErrorString(e));
}

int check_launch(const char *what) {
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return set_cuda_error(e, what);
  return RBG_OK;
}

// ---- device properties, cached per device ---------------------------------
struct DevProps {
  int sms = 0;
  size_t smem_per_sm = 0;
};
static DevProps g_devprops[64];
static const DevProps &dev_props() {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) dev = 0;
  DevProps &d = g_devprops[dev];
  if (d.sms == 0) {
    int v = 0;
    d.sms = (cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess && v > 0) ? v : 148;
    d.smem_per_sm = (cudaDeviceGetAttribute(&v, cudaDevAttrMaxSharedMemoryPerMultiprocessor, dev) == cudaSuccess && v > 0) ? (size_t)v : (size_t)228 * 1024;
  }
  return d;
}
int device_sm_count() { return dev_props().sms; }
size_t device_smem_per_sm() { return dev_props().smem_per_sm; }

bool stream_capturing(cudaStream_t stream) {
  cudaStreamCaptureStatus st = cudaStreamCaptureStatusNone;
  if (cudaStreamGetCaptureInfo(stream, &st) != cudaSuccess) {
    cudaGetLastError();  // (the legacy stream beside a capturing blocking stream): not ours to report here
    return false;
  }
  return st == cudaStreamCaptureStatusActive;
}

// ---- per-kernel event timing (rbg_kernel_timing / rbg_kernel_time) --------
struct EventPair {
  cudaEvent_t a, b;
};
static std::atomic<int> g_timing{0};
static std::mutex g_timing_mu;
static std::vector<EventPair> g_events[RBG_K_COUNT];

bool kernel_timing_on() { return g_timing.load(std::memory_order_relaxed) != 0; }

LaunchScope::LaunchScope(int kernel_id, cudaStream_t s) : id(kernel_id), stream(s), rec(nullptr) {
  g_launches.fetch_add(1, std::memory_order_relaxed);
  if (!g_timing.load(std::memory_order_relaxed) || id < 0 || id >= RBG_K_COUNT) return;
  EventPair *ep = new EventPair;
  if (cudaEventCreate(&ep->a) != cudaSuccess || cudaEventCreate(&ep->b) != cudaSuccess) {
    delete ep;
    return;
  }
  cudaEventRecord(ep->a, stream);
  rec = ep;
}

LaunchScope::~LaunchScope() {
  if (!rec) return;
  EventPair *ep = static_cast<EventPair *>(rec);
  cudaEventRecord(ep->b, stream);
  std::lock_guard<std::mutex> lock(g_timing_mu);
  g_events[id].push_back(*ep);
  delete ep;
}

static int check_dims(int64_t B, int G, int N, int need_cells_per_agent) {
  if (B < 0) return set_error(RBG_EINVAL, "B=%lld must be >= 0", (long long)B);
  if (B > 0x3fffffffLL) return set_error(RBG_EINVAL, "B=%lld too large (max 2^30-1 per call)", (long long)B);
  if (G < 2 || G > RBG_MAX_G) return set_error(RBG_EINVAL, "grid size G=%d outside [2,%d]", G, RBG_MAX_G);
  if (N < 1 || N > RBG_MAX_N) return set_error(RBG_EINVAL, "num_agents N=%d outside [1,%d]", N, RBG_MAX_N);
  if ((int64_t)need_cells_per_agent * N > (int64_t)G * G)
    return set_error(RBG_EINVAL, "N=%d agents need %d cells on a %dx%d grid (choice(replace=False) would raise)",
                     N, need_cells_per_agent * N, G, G);
  return RBG_OK;
}

static bool aligned16(const void *p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }
static bool aligned8(const void *p) { return (reinterpret_cast<uintptr_t>(p) & 7u) == 0; }

// 16-byte alignment of the bulk arrays is needed by the 128-bit path only, i.e. when G*G % 4 == 0 (otherwise the
// kernels use scalar accesses, and e.g. the step slices of a stacked rollout are legitimately unaligned)
static int check_state(const rbg_state *s, const char *name, int G) {
  if (!s) return set_error(RBG_EINVAL, "%s is NULL", name);
  if (!s->grid || !s->step_count || !s->agent_id || !s->start || !s->target || !s->position || !s->key)
    return set_error(RBG_EINVAL, "%s has a NULL field", name);
  if ((G * G) % 4 == 0 && !aligned16(s->grid)) return set_error(RBG_EALIGN, "%s.grid not 16-byte aligned", name);
  if (!aligned8(s->start) || !aligned8(s->target) || !aligned8(s->position))
    return set_error(RBG_EALIGN, "%s.start/target/position not 8-byte aligned", name);
  return RBG_OK;
}

static int check_timestep(const rbg_timestep *t, int G) {
  if (!t) return set_error(RBG_EINVAL, "timestep is NULL");
  if (!t->obs_grid || !t->action_mask || !t->obs_step_count || !t->reward || !t->discount || !t->step_type ||
      !t->num_connections || !t->ratio_connections || !t->total_path_length)
    return set_error(RBG_EINVAL, "timestep has a NULL field");
  if ((G * G) % 4 == 0 && !aligned16(t->obs_grid)) return set_error(RBG_EALIGN, "timestep.obs_grid not 16-byte aligned");
  return RBG_OK;
}

static int check_metrics(const rbg_episode_metrics *m, const char *name) {
  if (!m) return set_error(RBG_EINVAL, "%s is NULL", name);
  if (!m->episode_return || !m->episode_length || !m->num_connections || !m->ratio_connections || !m->total_path_length)
    return set_error(RBG_EINVAL, "%s has a NULL field", name);
  return RBG_OK;
}

static int check_dataset(const rbg_env_params *params) {
  if (!params->dataset_heads || !params->dataset_targets)
    return set_error(RBG_EINVAL, "autoreset_kind RBG_GEN_DATASET needs params->dataset_heads / dataset_targets (device int32[K,2,N])");
  if (params->dataset_K < 1 || params->dataset_K > 0x7fffffffLL)
    return set_error(RBG_EINVAL, "autoreset_kind RBG_GEN_DATASET: number of boards dataset_K=%lld", (long long)params->dataset_K);
  return RBG_OK;
}

static int debug_flags() {
  static int v = -1;
  if (v < 0) {
    const char *e = getenv("RBG_DEBUG_FLAGS");
    v = e ? atoi(e) : 0;
  }
  return v;
}

// ---- auto-reset workspace ------------------------------------------------------
// VmapAutoResetWrapper regenerates a board whenever an env finishes.  The reset key
// of an episode is known as soon as the episode starts (split(state.key)[0]), so the
// NEXT episode of every env that just reset is generated ahead of time ("refill")
// into a per-env cache; when the env finishes, env_warp_kernel swaps the
// cached episode in.  Only envs whose cache entry is not ready (first episode, or two
// terminations in consecutive steps) take the synchronous reset kernel.  Results are
// identical either way: a board is a pure function of its key.
struct WsLayout {
  size_t sync_list, refill_list[2], refill_keys[2], cache_tag, cache_key, cache_pins, group_done, group_pending, total;
};
static WsLayout ws_layout(int64_t B, int N) {
  auto up = [](size_t x) { return (x + 255) & ~(size_t)255; };
  WsLayout w;
  size_t off = 512;  // counters: sync @0, refill[0] @64, refill[1] @128; persistent rollout: 16 sets of 4 ints @256
  const size_t b = (size_t)(B > 0 ? B : 0);
  w.sync_list = off;
  off = up(off + 4 * b);
  for (int i = 0; i < 2; ++i) {
    w.refill_list[i] = off;
    off = up(off + 4 * b);
    w.refill_keys[i] = off;
    off = up(off + 8 * b);
  }
  w.cache_tag = off;
  off = up(off + 8 * b);
  w.cache_key = off;
  off = up(off + 8 * b);
  w.cache_pins = off;
  off = up(off + 4 * b * (size_t)N);
  w.group_done = off;  // persistent rollout: per env group, the last launch that wrote it / its requests in flight
  off = up(off + 4 * b);
  w.group_pending = off;
  off = up(off + 4 * b);
  w.total = off;
  return w;
}

// A ParallelRandomWalk / Uniform generation (kind) of the boards that follow `keys`, after `extra_split` leading
// split()[0]: PRWG:52 key, pos_key = split(key): the board uses split(key)[0]; UG:76 the uniform generator consumes the
// split itself (both halves).  With `cache_ws` the boards go to the next-episode cache of that auto-reset workspace.
static PrwParams prw_params(int kind, const uint32_t *keys, int64_t B, int G, int N, int extra_split, uint8_t *cache_ws = nullptr) {
  PrwParams p;
  memset(&p, 0, sizeof(p));
  p.keys = keys;
  p.B = B;
  p.G = G;
  p.N = N;
  p.mode = kind == RBG_GEN_PRW ? PRW_MODE_STATE : PRW_MODE_UNIFORM;
  p.extra_split = (kind == RBG_GEN_PRW ? 1 : 0) + extra_split;
  p.debug = debug_flags();
  if (cache_ws) {
    const WsLayout wl = ws_layout(B, N);
    p.to_cache = 1;
    p.cache_tag = reinterpret_cast<unsigned long long *>(cache_ws + wl.cache_tag);
    p.cache_key = reinterpret_cast<uint2 *>(cache_ws + wl.cache_key);
    p.cache_pins = reinterpret_cast<uint32_t *>(cache_ws + wl.cache_pins);
  }
  return p;
}

static int generator_state_impl(int kind, const uint32_t *keys, int64_t B, int G, int N, const rbg_state *out,
                                const rbg_timestep *ts, int extra_split, const int32_t *list,
                                const int32_t *list_count, cudaStream_t stream) {
  if (kind == RBG_GEN_PRW || kind == RBG_GEN_UNIFORM) {
    PrwParams p = prw_params(kind, keys, B, G, N, extra_split);
    p.st = *out;
    if (ts) {
      p.ts = *ts;
      p.observe = 1;
    }
    p.list = list;
    p.list_count = list_count;
    return launch_prw(p, B, stream);
  }
  if (kind == RBG_GEN_SEEDEXT) {
    SeedExtParams p;
    memset(&p, 0, sizeof(p));
    p.keys = keys;
    p.B = B;
    p.G = G;
    p.N = N;
    p.randomness = 0.0f;  // RSG:30 jit(generate_starts_ends) with the defaults
    p.two_sided = 1;
    p.iterations = 1;
    p.ext_steps = -1;
    p.extra_split = 1 + extra_split;  // RSG:34 key, pos_key = split(key)
    p.mode = GEN_MODE_STATE;
    p.st = *out;
    if (ts) {
      p.ts = *ts;
      p.observe = 1;
    }
    p.list = list;
    p.list_count = list_count;
    return launch_seedext(p, B, stream);
  }
  if (kind == RBG_GEN_SEQRW) {
    SeqRwParams p;
    memset(&p, 0, sizeof(p));
    p.keys = keys;
    p.B = B;
    p.G = G;
    p.N = N;
    p.extra_split = 1 + extra_split;  // sequential_random_walk_generator.py:42 key, pos_key = split(key)
    p.mode = GEN_MODE_STATE;
    p.st = *out;
    if (ts) {
      p.ts = *ts;
      p.observe = 1;
    }
    p.list = list;
    p.list_count = list_count;
    return launch_seqrw(p, B, stream);
  }
  return set_error(RBG_EINVAL, "unknown generator kind %d", kind);
}

struct AutoResetCtx {
  int64_t B = 0;
  int G = 0, N = 0, kind = -1;
  uint64_t step = 0;
  int persist_epoch = 0;  // launches of the persistent rollout on this workspace
  cudaStream_t last_stream = nullptr;  // the stream the workspace was last used on
  bool tail_valid = false;
};
static std::mutex g_ar_mu;
static std::unordered_map<void *, AutoResetCtx> g_ar;

// The next speculative call on `workspace` must adopt it afresh (counters zeroed, cache warm-started):
// its contents are no longer what the recorded context left there.
static void invalidate_workspace(void *workspace) {
  std::lock_guard<std::mutex> lock(g_ar_mu);
  auto it = g_ar.find(workspace);
  if (it != g_ar.end()) it->second.B = 0;
}

// The workspace moves to another stream (rare): its work on the old stream is awaited on the host.  Events per call
// would do, but an event record between two launches stops the second from starting under the first's tail.  A stream
// that is being captured is only recorded: a graph's replays are ordered against other streams by whoever launches them.
static int workspace_follow_stream(AutoResetCtx *ctx, cudaStream_t stream) {
  if (ctx->tail_valid && ctx->last_stream != stream && !stream_capturing(stream)) {
    cudaStreamSynchronize(ctx->last_stream);
    cudaGetLastError();  // (the old stream may be gone)
  }
  ctx->last_stream = stream;
  ctx->tail_valid = true;
  return RBG_OK;
}

// A speculative call on `ws` for another batch than the recorded one (or the first call): nothing is cached yet.  The
// counters are zeroed, and the cache is warm-started with the next episode of EVERY env, one bulk generation keyed by
// the current State.key `keys` (a cold cache would send each env's first reset down the synchronous path).
// Adoption is host-side bookkeeping that a replay would not redo, so it is refused while `stream` is capturing.
static int adopt_workspace(AutoResetCtx *ctx, uint8_t *ws, int kind, const uint32_t *keys, int64_t B, int G, int N, cudaStream_t stream) {
  if (ctx->B == B && ctx->G == G && ctx->N == N && ctx->kind == kind) return RBG_OK;
  if (stream_capturing(stream))
    return set_error(RBG_EINVAL, "the auto-reset workspace is new to this batch (or was re-initialised): step once outside the capture before capturing a step");
  cudaError_t e;
  int rc;
  if ((e = cudaMemsetAsync(ws, 0, 256, stream)) != cudaSuccess) return set_cuda_error(e, "cudaMemsetAsync(counters)");
  if ((rc = launch_prw(prw_params(kind, keys, B, G, N, 1, ws), B, stream))) return rc;
  ctx->B = B;
  ctx->G = G;
  ctx->N = N;
  ctx->kind = kind;
  ctx->step = 0;
  ctx->persist_epoch = 0;
  return RBG_OK;
}

// A Connector step (ENV_MODE_STEP under `env`) or observation (ENV_MODE_OBSERVE, env NULL) of B envs from `in` into `out`
static EnvParams env_params(int mode, const rbg_state &in, const rbg_state &out, int64_t B, int G, int N, const rbg_env_params *env) {
  EnvParams p;
  memset(&p, 0, sizeof(p));
  p.in = in;
  p.out = out;
  p.B = B;
  p.G = G;
  p.N = N;
  p.mode = mode;
  if (env)
    p.env = *env;
  else
    p.env.autoreset_kind = -1;
  return p;
}

// Per-step auto-reset with the cache (ParallelRandomWalk / Uniform): everything runs on the caller's stream.  The
// synchronous resets of step t and the cache refill are one kernel (prw_pair_kernel) that says launch_dependents
// between the two, and the env kernel of step t + 1 is launched with programmatic stream serialization, so the refill
// of step t overlaps the env kernel of step t + 1 by construction and nothing else moves.  While kernel timing is on,
// the env kernel waits for the whole of prw_pair_kernel, so that each event pair times one kernel.
static int connector_step_impl(const rbg_state *in, const rbg_state *out, const int32_t *action, int32_t *action_out,
                               int random_policy, int64_t B, int G, int N, const rbg_env_params *params,
                               const rbg_timestep *ts, void *workspace, cudaStream_t stream) {
  int rc;
  if ((rc = check_dims(B, G, N, 1))) return rc;
  if (B == 0) return RBG_OK;  // an empty batch has no buffers to check
  if ((rc = check_state(in, "state_in", G))) return rc;
  if ((rc = check_state(out, "state_out", G))) return rc;
  if ((rc = check_timestep(ts, G))) return rc;
  if (!params) return set_error(RBG_EINVAL, "params is NULL");
  if (!random_policy && !action) return set_error(RBG_EINVAL, "action is NULL");
  const bool autoreset = params->autoreset_kind >= 0;
  const bool dataset = params->autoreset_kind == RBG_GEN_DATASET;
  if (autoreset && !dataset && !workspace) return set_error(RBG_EINVAL, "auto-reset needs a workspace (rbg_step_workspace_bytes)");
  if (autoreset && params->autoreset_kind > RBG_GEN_SEQRW)
    return set_error(RBG_EINVAL, "unknown autoreset generator kind %d", params->autoreset_kind);
  if (dataset && (rc = check_dataset(params))) return rc;
  EnvParams p = env_params(ENV_MODE_STEP, *in, *out, B, G, N, params);
  p.ts = *ts;
  p.action = action;
  p.action_out = action_out;
  p.random_policy = random_policy;
  if (!autoreset || dataset) return launch_env(p, stream);  // dataset resets are a lookup inside the kernel

  uint8_t *ws = reinterpret_cast<uint8_t *>(workspace);
  if (!aligned16(ws)) return set_error(RBG_EALIGN, "workspace not 16-byte aligned");
  const WsLayout wl = ws_layout(B, N);
  const int kind = params->autoreset_kind;
  int32_t *sync_count = reinterpret_cast<int32_t *>(ws);
  int32_t *sync_list = reinterpret_cast<int32_t *>(ws + wl.sync_list);
  p.list = sync_list;
  p.list_count = sync_count;
  // VmapAutoResetWrapper._auto_reset: key, _ = split(state.key); reset(key):
  // one more leading split()[0] than a plain generator call.
  if (kind != RBG_GEN_PRW && kind != RBG_GEN_UNIFORM) {
    cudaError_t e;
    if ((e = cudaMemsetAsync(ws, 0, 64, stream)) != cudaSuccess) return set_cuda_error(e, "cudaMemsetAsync(reset counter)");
    // This path leaves its reset count in the counter.  If the same workspace has served (or will
    // serve) a speculative batch, that batch must adopt it afresh: its kernels rely on counters
    // that are zero between steps.
    invalidate_workspace(workspace);
    if ((rc = launch_env(p, stream))) return rc;
    return generator_state_impl(kind, out->key, B, G, N, out, ts, 1, sync_list, sync_count, stream);
  }
  // speculative: the counters were zeroed once when the workspace was adopted, and the list kernels clear their own
  // counter when they finish (prw_kernel list_ticket)
  AutoResetCtx *ctx;
  {
    std::lock_guard<std::mutex> lock(g_ar_mu);
    ctx = &g_ar[workspace];
    if ((rc = workspace_follow_stream(ctx, stream))) return rc;
    if ((rc = adopt_workspace(ctx, ws, kind, in->key, B, G, N, stream))) return rc;
    // the refill lists alternate between two buffers: this step's env kernel runs under the previous step's refill
    const int par = (int)(ctx->step & 1);
    p.cache_tag = reinterpret_cast<const unsigned long long *>(ws + wl.cache_tag);
    p.cache_key = reinterpret_cast<const uint2 *>(ws + wl.cache_key);
    p.cache_pins = reinterpret_cast<const uint32_t *>(ws + wl.cache_pins);
    p.refill_list = reinterpret_cast<int32_t *>(ws + wl.refill_list[par]);
    p.refill_keys = reinterpret_cast<uint32_t *>(ws + wl.refill_keys[par]);
    p.refill_count = reinterpret_cast<int32_t *>(ws + 64 + 64 * par);
  }
  if ((rc = launch_env(p, stream, !kernel_timing_on()))) return rc;
  // one launch: the synchronous resets (rare misses), launch_dependents, then the cache refill
  PrwParams a = prw_params(kind, out->key, B, G, N, 1);
  a.st = *out;
  a.ts = *ts;
  a.observe = 1;
  a.list = sync_list;
  a.list_count = sync_count;
  a.list_ticket = sync_count + 1;
  PrwParams q = prw_params(kind, p.refill_keys, B, G, N, 1, ws);
  q.keys_compact = 1;
  q.list = p.refill_list;
  q.list_count = p.refill_count;
  q.list_ticket = p.refill_count + 1;
  if ((rc = launch_prw_pair(a, q, B, stream))) return rc;
  ctx->step++;
  return RBG_OK;
}

// ---- device scratch for the _host variants --------------------------------
struct Scratch {
  void *ptr = nullptr;
  size_t bytes = 0;
  int device = -1;
};
static std::mutex g_scratch_mu;
// One scratch, one set of streams and one signature PER DEVICE: a process that drives several GPUs through the
// _host variants (one thread per device, or device switches between calls) keeps each device's workspaces alive.
constexpr int kMaxDevices = 64;
// Who laid the scratch out last (a step variant with auto-reset keeps its workspaces there between
// calls): any other use, shape or base pointer means those workspaces have been overwritten.
struct ScratchSig {
  int fn = 0;
  int64_t B = 0;
  int G = 0, N = 0, kind = -1;
  void *base = nullptr;
  bool operator==(const ScratchSig &o) const { return fn == o.fn && B == o.B && G == o.G && N == o.N && kind == o.kind && base == o.base; }
};
struct HostCtx {
  Scratch scratch;
  cudaStream_t streams[3] = {nullptr, nullptr, nullptr};
  cudaEvent_t slice_ev[16] = {nullptr};
  cudaEvent_t copy_ev[16] = {nullptr};
  cudaEvent_t entry_ev = nullptr;
  uint8_t *stage8 = nullptr;  // pinned host staging of the byte observation (rbg_connector_step_host_io)
  size_t stage8_bytes = 0;
  // thread-count tuning of the byte transport: the first calls of a batch shape try 1/4, 1/2, 3/4 and all of the
  // pool's workers (four calls each, the last three timed; more threads must win by 1 %) and the fastest count stays
  int64_t tune_B = -1;
  int tune_call = 0, tune_best = 0;
  double tune_best_s = 0.0;
  ScratchSig sig;
};
// what the _host variants moved over the bus since the last reset (rbg_host_transfer_stats)
static std::atomic<long long> g_h2d_bytes{0}, g_d2h_bytes{0};
static HostCtx g_host[kMaxDevices];
static thread_local HostCtx *g_hc = &g_host[0];  // the device of the _host call in progress (set by use_device)

static int scratch_get(size_t bytes, int device, void **out) {
  if (g_hc->scratch.ptr && (g_hc->scratch.bytes < bytes || g_hc->scratch.device != device)) {
    cudaFree(g_hc->scratch.ptr);
    g_hc->scratch = Scratch();
  }
  if (!g_hc->scratch.ptr) {
    cudaError_t e = cudaMalloc(&g_hc->scratch.ptr, bytes);
    if (e != cudaSuccess) {
      g_hc->scratch = Scratch();
      return set_cuda_error(e, "cudaMalloc(host-variant scratch)");
    }
    g_hc->scratch.bytes = bytes;
    g_hc->scratch.device = device;
  }
  for (int i = 0; i < 3; ++i)
    if (!g_hc->streams[i]) {
      cudaError_t e = cudaStreamCreateWithFlags(&g_hc->streams[i], cudaStreamNonBlocking);
      if (e != cudaSuccess) return set_cuda_error(e, "cudaStreamCreate");
    }
  *out = g_hc->scratch.ptr;
  return RBG_OK;
}

// Waits for all three streams of the _host variants, also after one of them has failed.
static int sync_streams() {
  int rc = RBG_OK;
  for (int i = 0; i < 3; ++i) {
    cudaError_t e = cudaStreamSynchronize(g_hc->streams[i]);
    if (e != cudaSuccess) rc = set_cuda_error(e, "cudaStreamSynchronize");
  }
  return rc;
}

// A _host call that fails after it has enqueued copies waits for its streams before it returns, so that no copy from
// or into the caller's buffers is in flight once it has returned.  The message stays the failure's.
static int fail_synced(int rc) {
  char msg[sizeof(g_err)];
  memcpy(msg, g_err, sizeof(msg));
  sync_streams();
  memcpy(g_err, msg, sizeof(msg));
  return rc;
}

struct Carver {
  uint8_t *base;
  size_t off = 0;
  template <typename T>
  T *take(size_t n) {
    off = (off + 255) & ~(size_t)255;
    T *p = base ? reinterpret_cast<T *>(base + off) : nullptr;
    off += n * sizeof(T);
    return p;
  }
};

// `layout(Carver &)` takes a call's device buffers in order.  It runs once on a null base to size the scratch and
// once on the scratch itself, so the two passes cannot disagree.
template <typename Layout>
static int scratch_carve(int device, void **base, Layout &&layout) {
  Carver size{nullptr};
  layout(size);
  int rc = scratch_get(size.off + 256, device, base);
  if (rc) return rc;
  Carver c{reinterpret_cast<uint8_t *>(*base)};
  layout(c);
  return RBG_OK;
}

static void carve_state(Carver &c, int64_t B, int G, int N, rbg_state *s) {
  s->grid = c.take<int32_t>((size_t)B * G * G);
  s->step_count = c.take<int32_t>((size_t)B);
  s->agent_id = c.take<int32_t>((size_t)B * N);
  s->start = c.take<int32_t>((size_t)B * N * 2);
  s->target = c.take<int32_t>((size_t)B * N * 2);
  s->position = c.take<int32_t>((size_t)B * N * 2);
  s->key = c.take<uint32_t>((size_t)B * 2);
}
static void carve_timestep(Carver &c, int64_t B, int G, int N, rbg_timestep *t) {
  t->obs_grid = c.take<int32_t>((size_t)B * N * G * G);
  t->action_mask = c.take<uint8_t>((size_t)B * N * 5);
  t->obs_step_count = c.take<int32_t>((size_t)B);
  t->reward = c.take<float>((size_t)B * N);
  t->discount = c.take<float>((size_t)B * N);
  t->step_type = c.take<int8_t>((size_t)B);
  t->num_connections = c.take<int32_t>((size_t)B);
  t->ratio_connections = c.take<float>((size_t)B);
  t->total_path_length = c.take<int32_t>((size_t)B);
}

#define RBG_CPY(dst, src, n, kind, st)                                                    \
  do {                                                                                    \
    cudaError_t e_ = cudaMemcpyAsync((dst), (src), (n), (kind), (st));                    \
    if (e_ != cudaSuccess) return set_cuda_error(e_, "cudaMemcpyAsync " #dst);            \
  } while (0)

static int copy_state(const rbg_state *dst, const rbg_state *src, int64_t off, int64_t n, int G, int N,
                      cudaMemcpyKind kind, int64_t dst_off, cudaStream_t st) {
  const size_t c = (size_t)G * G;
  RBG_CPY(dst->grid + dst_off * c, src->grid + off * c, n * c * 4, kind, st);
  RBG_CPY(dst->step_count + dst_off, src->step_count + off, n * 4, kind, st);
  RBG_CPY(dst->agent_id + dst_off * N, src->agent_id + off * N, n * N * 4, kind, st);
  RBG_CPY(dst->start + dst_off * N * 2, src->start + off * N * 2, n * N * 8, kind, st);
  RBG_CPY(dst->target + dst_off * N * 2, src->target + off * N * 2, n * N * 8, kind, st);
  RBG_CPY(dst->position + dst_off * N * 2, src->position + off * N * 2, n * N * 8, kind, st);
  RBG_CPY(dst->key + dst_off * 2, src->key + off * 2, n * 8, kind, st);
  return RBG_OK;
}
// `with_obs`: false leaves observation.grid (the bulk) out
static int copy_timestep(const rbg_timestep *dst, const rbg_timestep *src, int64_t off, int64_t n, int G, int N,
                         cudaMemcpyKind kind, int64_t dst_off, cudaStream_t st, bool with_obs = true) {
  const size_t c = (size_t)G * G * N;
  if (with_obs) RBG_CPY(dst->obs_grid + dst_off * c, src->obs_grid + off * c, n * c * 4, kind, st);
  RBG_CPY(dst->action_mask + dst_off * N * 5, src->action_mask + off * N * 5, n * N * 5, kind, st);
  RBG_CPY(dst->obs_step_count + dst_off, src->obs_step_count + off, n * 4, kind, st);
  RBG_CPY(dst->reward + dst_off * N, src->reward + off * N, n * N * 4, kind, st);
  RBG_CPY(dst->discount + dst_off * N, src->discount + off * N, n * N * 4, kind, st);
  RBG_CPY(dst->step_type + dst_off, src->step_type + off, n, kind, st);
  RBG_CPY(dst->num_connections + dst_off, src->num_connections + off, n * 4, kind, st);
  RBG_CPY(dst->ratio_connections + dst_off, src->ratio_connections + off, n * 4, kind, st);
  RBG_CPY(dst->total_path_length + dst_off, src->total_path_length + off, n * 4, kind, st);
  return RBG_OK;
}

static rbg_state state_at(const rbg_state &s, int64_t off, int G, int N) {
  rbg_state r;
  r.grid = s.grid + off * G * G;
  r.step_count = s.step_count + off;
  r.agent_id = s.agent_id + off * N;
  r.start = s.start + off * N * 2;
  r.target = s.target + off * N * 2;
  r.position = s.position + off * N * 2;
  r.key = s.key + off * 2;
  return r;
}
static rbg_timestep timestep_at(const rbg_timestep &t, int64_t off, int G, int N) {
  rbg_timestep r;
  r.obs_grid = t.obs_grid + off * N * G * G;
  r.action_mask = t.action_mask + off * N * 5;
  r.obs_step_count = t.obs_step_count + off;
  r.reward = t.reward + off * N;
  r.discount = t.discount + off * N;
  r.step_type = t.step_type + off;
  r.num_connections = t.num_connections + off;
  r.ratio_connections = t.ratio_connections + off;
  r.total_path_length = t.total_path_length + off;
  return r;
}

// slices are multiples of 64 envs so that every slice base keeps the 16-byte
// alignment of the bulk arrays for any (G, N)
static int64_t slice_size(int64_t B, int nslices) {
  int64_t s = (B + nslices - 1) / nslices;
  s = (s + 63) / 64 * 64;
  return s < 64 ? 64 : s;
}

}  // namespace rbg

using namespace rbg;

extern "C" {

int rbg_version(void) { return RBG_VERSION; }
const char *rbg_last_error(void) { return g_err; }

int rbg_device_info(int *sm_arch, int *sm_count) {
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return set_cuda_error(e, "cudaGetDevice");
  cudaDeviceProp prop;
  e = cudaGetDeviceProperties(&prop, dev);
  if (e != cudaSuccess) return set_cuda_error(e, "cudaGetDeviceProperties");
  if (sm_arch) *sm_arch = prop.major * 10 + prop.minor;
  if (sm_count) *sm_count = prop.multiProcessorCount;
  return RBG_OK;
}

int64_t rbg_launch_count(int reset) {
  return reset ? g_launches.exchange(0) : g_launches.load();
}

int rbg_kernel_timing(int enable) {
  g_timing.store(enable ? 1 : 0);
  return RBG_OK;
}

int rbg_kernel_time(int kernel, int64_t *launches, double *total_ms) {
  if (kernel < 0 || kernel >= RBG_K_COUNT) return set_error(RBG_EINVAL, "rbg_kernel_time: unknown kernel id %d", kernel);
  std::vector<EventPair> evs;
  {
    std::lock_guard<std::mutex> lock(g_timing_mu);
    evs.swap(g_events[kernel]);
  }
  double ms = 0.0;
  int rc = RBG_OK;
  for (EventPair &ep : evs) {
    float t = 0.0f;
    cudaError_t e = cudaEventSynchronize(ep.b);
    if (e == cudaSuccess) e = cudaEventElapsedTime(&t, ep.a, ep.b);
    if (e != cudaSuccess) rc = set_cuda_error(e, "rbg_kernel_time");
    ms += t;
    cudaEventDestroy(ep.a);
    cudaEventDestroy(ep.b);
  }
  if (launches) *launches = (int64_t)evs.size();
  if (total_ms) *total_ms = ms;
  return rc;
}

int rbg_split_keys(const uint32_t key[2], int64_t B, int64_t offset, int64_t count, uint32_t *out, void *stream) {
  if (!key || !out) return set_error(RBG_EINVAL, "rbg_split_keys: NULL pointer");
  if (B < 1 || B > 0x7fffffffLL || offset < 0 || count < 0 || offset + count > B)
    return set_error(RBG_EINVAL, "rbg_split_keys: bad slice [%lld,+%lld) of B=%lld", (long long)offset,
                     (long long)count, (long long)B);
  return launch_split_keys(key[0], key[1], B, offset, count, out, (cudaStream_t)stream);
}

int rbg_prw_generate(const uint32_t *keys, int64_t B, int G, int N, int32_t *heads, int32_t *targets,
                     int32_t *solved, int32_t *stats, void *stream) {
  int rc;
  if ((rc = check_dims(B, G, N, 1))) return rc;
  if (B == 0) return RBG_OK;  // an empty batch has no buffers to check
  if (!keys || !heads || !targets || !solved) return set_error(RBG_EINVAL, "rbg_prw_generate: NULL pointer");
  if (!aligned16(solved)) return set_error(RBG_EALIGN, "rbg_prw_generate: solved not 16-byte aligned");
  PrwParams p;
  memset(&p, 0, sizeof(p));
  p.keys = keys;
  p.B = B;
  p.G = G;
  p.N = N;
  p.mode = PRW_MODE_BOARD;
  p.debug = debug_flags();
  p.heads = heads;
  p.targets = targets;
  p.solved = solved;
  p.stats = stats;
  return launch_prw(p, B, (cudaStream_t)stream);
}

int rbg_generator_state(int kind, const uint32_t *keys, int64_t B, int G, int N, const rbg_state *out, void *stream) {
  int rc;
  // (the sequential random walk has no choice(replace=False) over the agents: more agents than cells is a failed generation)
  if ((rc = check_dims(B, G, N, kind == RBG_GEN_UNIFORM ? 2 : kind == RBG_GEN_SEQRW ? 0 : 1))) return rc;
  if (B == 0) return RBG_OK;  // an empty batch has no buffers to check
  if (!keys) return set_error(RBG_EINVAL, "keys is NULL");
  if ((rc = check_state(out, "state", G))) return rc;
  return generator_state_impl(kind, keys, B, G, N, out, nullptr, 0, nullptr, nullptr, (cudaStream_t)stream);
}

int rbg_dataset_state(const uint32_t *keys, int64_t B, int G, int N, const int32_t *heads, const int32_t *targets, int64_t K,
                      const rbg_state *out, void *stream) {
  int rc;
  if ((rc = check_dims(B, G, N, 1))) return rc;
  if (B == 0) return RBG_OK;
  if (!keys || !heads || !targets) return set_error(RBG_EINVAL, "rbg_dataset_state: NULL pointer");
  if (K < 1 || K > 0x7fffffffLL) return set_error(RBG_EINVAL, "rbg_dataset_state: number of boards K=%lld", (long long)K);
  if ((rc = check_state(out, "state", G))) return rc;
  return launch_dataset_state(keys, B, G, N, heads, targets, K, *out, (cudaStream_t)stream);
}

int rbg_seedext_solved(const uint32_t *keys, int64_t B, int G, int N, float randomness, int two_sided,
                       int iterations, int64_t extension_steps, int32_t *solved, void *stream) {
  int rc;
  if ((rc = check_dims(B, G, N, 1))) return rc;
  if (B == 0) return RBG_OK;  // an empty batch has no buffers to check
  if (!keys || !solved) return set_error(RBG_EINVAL, "rbg_seedext_solved: NULL pointer");
  if (!aligned16(solved)) return set_error(RBG_EALIGN, "rbg_seedext_solved: solved not 16-byte aligned");
  SeedExtParams p;
  memset(&p, 0, sizeof(p));
  p.keys = keys;
  p.B = B;
  p.G = G;
  p.N = N;
  p.randomness = randomness;
  p.two_sided = two_sided;
  p.iterations = iterations;
  p.ext_steps = extension_steps;
  p.mode = GEN_MODE_BOARD;
  p.solved = solved;
  return launch_seedext(p, B, (cudaStream_t)stream);
}

int rbg_seedext_starts_ends(const uint32_t *keys, int64_t B, int G, int N, float randomness, int two_sided,
                            int iterations, int64_t extension_steps, int32_t *starts, int32_t *ends, void *stream) {
  int rc;
  if ((rc = check_dims(B, G, N, 1))) return rc;
  if (B == 0) return RBG_OK;  // an empty batch has no buffers to check
  if (!keys || !starts || !ends) return set_error(RBG_EINVAL, "rbg_seedext_starts_ends: NULL pointer");
  SeedExtParams p;
  memset(&p, 0, sizeof(p));
  p.keys = keys;
  p.B = B;
  p.G = G;
  p.N = N;
  p.randomness = randomness;
  p.two_sided = two_sided;
  p.iterations = iterations;
  p.ext_steps = extension_steps;
  p.mode = GEN_MODE_STARTS_ENDS;
  p.starts = starts;
  p.ends = ends;
  return launch_seedext(p, B, (cudaStream_t)stream);
}

int rbg_seqrw_generate(const uint32_t *keys, int64_t B, int G, int N, void *board, int as_float32, int32_t *stats, void *stream) {
  int rc;
  if ((rc = check_dims(B, G, N, 0))) return rc;
  if (B == 0) return RBG_OK;
  if (G < 3) return set_error(RBG_EINVAL, "SequentialRandomWalk: rows=%d (available_cells pads with jnp.full(rows - 3, -1): rows >= 3)", G);
  if (!keys || !board) return set_error(RBG_EINVAL, "rbg_seqrw_generate: NULL argument");
  if (!aligned16(board)) return set_error(RBG_EALIGN, "board not 16-byte aligned");
  SeqRwParams p;
  memset(&p, 0, sizeof(p));
  p.keys = keys;
  p.B = B;
  p.G = G;
  p.N = N;
  p.mode = GEN_MODE_BOARD;
  p.float_board = as_float32 ? 1 : 0;
  p.board = reinterpret_cast<int32_t *>(board);
  p.stats = stats;
  return launch_seqrw(p, B, (cudaStream_t)stream);
}

int rbg_seqrw_starts_ends(const uint32_t *keys, int64_t B, int G, int N, int32_t *starts, int32_t *ends, void *stream) {
  int rc;
  if ((rc = check_dims(B, G, N, 0))) return rc;
  if (B == 0) return RBG_OK;
  if (!keys || !starts || !ends) return set_error(RBG_EINVAL, "rbg_seqrw_starts_ends: NULL argument");
  SeqRwParams p;
  memset(&p, 0, sizeof(p));
  p.keys = keys;
  p.B = B;
  p.G = G;
  p.N = N;
  p.mode = GEN_MODE_STARTS_ENDS;
  p.starts = starts;
  p.ends = ends;
  return launch_seqrw(p, B, (cudaStream_t)stream);
}

int rbg_connector_observe(const rbg_state *state, int64_t B, int G, int N, const rbg_timestep *ts, void *stream) {
  int rc;
  if ((rc = check_dims(B, G, N, 1))) return rc;
  if (B == 0) return RBG_OK;  // an empty batch has no buffers to check
  if ((rc = check_state(state, "state", G))) return rc;
  if ((rc = check_timestep(ts, G))) return rc;
  EnvParams p = env_params(ENV_MODE_OBSERVE, *state, *state, B, G, N, nullptr);
  p.ts = *ts;
  return launch_env(p, (cudaStream_t)stream);
}

int rbg_connector_reset(int kind, const uint32_t *keys, int64_t B, int G, int N, const rbg_state *state,
                        const rbg_timestep *ts, void *stream) {
  int rc = rbg_generator_state(kind, keys, B, G, N, state, stream);
  if (rc) return rc;
  return rbg_connector_observe(state, B, G, N, ts, stream);
}

int rbg_connector_reset_dataset(const uint32_t *keys, int64_t B, int G, int N, const int32_t *heads, const int32_t *targets,
                                int64_t K, const rbg_state *state, const rbg_timestep *ts, void *stream) {
  int rc = rbg_dataset_state(keys, B, G, N, heads, targets, K, state, stream);
  if (rc) return rc;
  return rbg_connector_observe(state, B, G, N, ts, stream);
}

int rbg_split_each(const uint32_t *keys, int64_t B, int num, uint32_t *out, void *stream) {
  if (B < 0 || B > 0x3fffffffLL) return set_error(RBG_EINVAL, "rbg_split_each: B=%lld", (long long)B);
  if (num < 1 || num > 65536) return set_error(RBG_EINVAL, "rbg_split_each: num=%d outside [1,65536]", num);
  if (B == 0) return RBG_OK;
  if (!keys || !out) return set_error(RBG_EINVAL, "rbg_split_each: NULL pointer");
  return launch_split_each(keys, B, num, out, (cudaStream_t)stream);
}

int64_t rbg_step_workspace_bytes(int64_t B, int G, int N) {
  (void)G;
  return (int64_t)ws_layout(B, N).total;
}

int rbg_workspace_release(void *workspace) {
  std::lock_guard<std::mutex> lock(g_ar_mu);
  auto it = g_ar.find(workspace);
  if (it == g_ar.end()) return RBG_OK;
  if (it->second.tail_valid) {
    cudaStreamSynchronize(it->second.last_stream);
    cudaGetLastError();
  }
  g_ar.erase(it);
  return RBG_OK;
}

int rbg_connector_step(const rbg_state *in, const rbg_state *out, const int32_t *action, int64_t B, int G, int N,
                       const rbg_env_params *params, const rbg_timestep *ts, void *workspace, void *stream) {
  return connector_step_impl(in, out, action, nullptr, 0, B, G, N, params, ts, workspace, (cudaStream_t)stream);
}

int rbg_connector_step_random(const rbg_state *in, const rbg_state *out, int32_t *action_out, int64_t B, int G, int N,
                              const rbg_env_params *params, const rbg_timestep *ts, void *workspace, void *stream) {
  return connector_step_impl(in, out, nullptr, action_out, 1, B, G, N, params, ts, workspace, (cudaStream_t)stream);
}

// Steps per launch of the fused rollout kernels: the reference's n_steps (agent_training/configs/env/connector.yaml:27)
constexpr int kRolloutChunk = 20;

// Fused rollout, one launch per chunk of steps: rollout_warp_kernel for the dataset (resets are a table lookup inside
// the kernel: no cache, no workspace), rollout_persist_kernel for ParallelRandomWalk / Uniform (the kernel's generator
// warps keep the next-episode cache filled; consecutive launches on the stream overlap head to tail).
static int rollout_fused(const rbg_state *state, int32_t *action_out, int64_t T, int64_t B, int G, int N,
                         const rbg_env_params *params, const rbg_timestep *ts, void *workspace, cudaStream_t stream) {
  uint8_t *ws = reinterpret_cast<uint8_t *>(workspace);
  const WsLayout wl = ws_layout(B, N);
  const int kind = params->autoreset_kind;
  const bool dataset = kind == RBG_GEN_DATASET;
  cudaError_t e;
  int rc;
  EnvParams p = env_params(ENV_MODE_STEP, *state, *state, B, G, N, params);
  p.random_policy = 1;
  AutoResetCtx *ctx = nullptr;
  if (!dataset) {
    {
      std::lock_guard<std::mutex> lock(g_ar_mu);
      ctx = &g_ar[workspace];
    }
    if ((rc = workspace_follow_stream(ctx, stream))) return rc;
    if ((rc = adopt_workspace(ctx, ws, kind, state->key, B, G, N, stream))) return rc;
    p.cache_tag = reinterpret_cast<const unsigned long long *>(ws + wl.cache_tag);
    p.cache_key = reinterpret_cast<const uint2 *>(ws + wl.cache_key);
    p.cache_pins = reinterpret_cast<const uint32_t *>(ws + wl.cache_pins);
  }
  for (int64_t t0 = 0; t0 < T; t0 += kRolloutChunk) {
    const int n = (int)((T - t0) < kRolloutChunk ? (T - t0) : kRolloutChunk);
    int32_t *acts = action_out ? action_out + t0 * B * N : nullptr;
    p.ts = timestep_at(*ts, t0 * B, G, N);
    if (dataset) {
      if ((rc = launch_rollout(p, n, acts, stream))) return rc;
      continue;
    }
    if (ctx->persist_epoch == 0 || ctx->persist_epoch > 0x3fffffff) {  // flags start at 0 = "written by launch 0"
      if ((e = cudaMemsetAsync(ws + wl.group_done, 0, (wl.group_pending - wl.group_done) + 4 * (size_t)B, stream)) != cudaSuccess) return set_cuda_error(e, "cudaMemsetAsync(group flags)");
      if ((e = cudaMemsetAsync(ws + 256, 0, 256, stream)) != cudaSuccess) return set_cuda_error(e, "cudaMemsetAsync(persist counters)");
      ctx->persist_epoch = 0;
    }
    const int epoch = ++ctx->persist_epoch;
    const bool overlap = epoch > 1 && !kernel_timing_on();  // event pairs must time one kernel at a time
    if ((rc = launch_rollout_persist(p, kind, n, acts, reinterpret_cast<int32_t *>(ws + 256),
                                     reinterpret_cast<int32_t *>(ws + wl.group_done), reinterpret_cast<int32_t *>(ws + wl.group_pending), epoch, overlap,
                                     reinterpret_cast<uint64_t *>(ws + wl.cache_tag), reinterpret_cast<uint2 *>(ws + wl.cache_key),
                                     reinterpret_cast<uint32_t *>(ws + wl.cache_pins), stream)))
      return rc;
  }
  return RBG_OK;
}

int rbg_connector_rollout_random(const rbg_state *state, int32_t *action_out, int64_t T, int64_t B, int G, int N,
                                 const rbg_env_params *params, const rbg_timestep *ts, void *workspace, void *stream) {
  int rc;
  if (T < 0) return set_error(RBG_EINVAL, "rollout length T=%lld", (long long)T);
  if ((rc = check_dims(B, G, N, 1))) return rc;
  if (B == 0 || T == 0) return RBG_OK;  // an empty batch has no buffers to check
  if (stream_capturing((cudaStream_t)stream))
    return set_error(RBG_EINVAL, "rbg_connector_rollout_random cannot be captured into a CUDA graph: its persistent kernel takes host-side "
                                 "epochs that every replay would reuse (capture rbg_connector_step_random instead)");
  // (when G*G % 4 == 0 every step slice of the stacked arrays keeps the 16-byte alignment the
  // vector path needs; otherwise the kernels use scalar accesses)
  if ((rc = check_state(state, "state", G))) return rc;
  if ((rc = check_timestep(ts, G))) return rc;
  if (!params) return set_error(RBG_EINVAL, "params is NULL");
  const int kind = params->autoreset_kind;
  if (kind > RBG_GEN_SEQRW) return set_error(RBG_EINVAL, "unknown autoreset generator kind %d", kind);
  if (kind < 0) return set_error(RBG_EINVAL, "rollout needs an auto-reset generator kind (params->autoreset_kind >= 0)");
  // few agents on a big board: a fused CTA's grids, staging and generator scratch do not fit its shared memory; the
  // step-wise loop below computes the same steps
  const bool fused = (kind == RBG_GEN_DATASET || kind == RBG_GEN_PRW || kind == RBG_GEN_UNIFORM) && rollout_smem(kind, G, N) <= kRolloutMaxSmem;
  if (fused) {
    if (kind == RBG_GEN_DATASET) {
      if ((rc = check_dataset(params))) return rc;
    } else {
      if (!workspace) return set_error(RBG_EINVAL, "auto-reset needs a workspace (rbg_step_workspace_bytes)");
      if (!aligned16(workspace)) return set_error(RBG_EALIGN, "workspace not 16-byte aligned");
    }
    return rollout_fused(state, action_out, T, B, G, N, params, ts, workspace, (cudaStream_t)stream);
  }
  for (int64_t t = 0; t < T; ++t) {  // step-wise: SeedExtension / SequentialRandomWalk resets, and shapes too big to fuse
    const rbg_timestep tt = timestep_at(*ts, t * B, G, N);
    rc = connector_step_impl(state, state, nullptr, action_out ? action_out + t * B * N : nullptr, 1, B, G, N, params, &tt, workspace,
                             (cudaStream_t)stream);
    if (rc) return rc;
  }
  return RBG_OK;
}

int rbg_connector_episodes_random(const rbg_state *start, int64_t B, int G, int N, const rbg_env_params *params, const rbg_episode_metrics *out,
                                  const rbg_state *final_state, void *stream) {
  int rc;
  if ((rc = check_dims(B, G, N, 1))) return rc;
  if (B == 0) return RBG_OK;  // an empty batch has no buffers to check
  if ((rc = check_state(start, "start", G))) return rc;
  if (!params) return set_error(RBG_EINVAL, "params is NULL");
  if (params->autoreset_kind >= 0)
    return set_error(RBG_EINVAL, "episodes end at their first LAST step: params->autoreset_kind must be < 0 (got %d)", params->autoreset_kind);
  if ((rc = check_metrics(out, "metrics"))) return rc;
  if (final_state && (rc = check_state(final_state, "final_state", G))) return rc;
  return launch_episodes(*start, final_state, *out, B, G, N, *params, (cudaStream_t)stream);
}

int rbg_connector_eval_step(const rbg_state *state, const int32_t *action, uint8_t *live, int32_t *live_count, int64_t B, int G, int N,
                            const rbg_env_params *params, const rbg_timestep *ts, const rbg_episode_metrics *acc, void *stream) {
  int rc;
  if ((rc = check_dims(B, G, N, 1))) return rc;
  if (B == 0) return RBG_OK;  // an empty batch has no buffers to check
  if ((rc = check_state(state, "state", G))) return rc;
  if (!action) return set_error(RBG_EINVAL, "action is NULL");
  if (!live) return set_error(RBG_EINVAL, "live is NULL");
  if (!live_count) return set_error(RBG_EINVAL, "live_count is NULL");
  if (!params) return set_error(RBG_EINVAL, "params is NULL");
  if (params->autoreset_kind >= 0)
    return set_error(RBG_EINVAL, "an evaluation step ends an episode at its first LAST step: params->autoreset_kind must be < 0 (got %d)",
                     params->autoreset_kind);
  if ((rc = check_timestep(ts, G))) return rc;
  if ((rc = check_metrics(acc, "acc"))) return rc;
  return launch_eval_step(*state, action, live, live_count, B, G, N, *params, *ts, *acc, (cudaStream_t)stream);
}

int rbg_connector_eval_step_live(const rbg_state *state, const int32_t *action, const int32_t *order_in, int64_t L, int32_t *order_out,
                                 int32_t *count_out, int64_t B, int G, int N, const rbg_env_params *params, const rbg_timestep *ts,
                                 const rbg_episode_metrics *acc, void *stream) {
  int rc;
  if ((rc = check_dims(B, G, N, 1))) return rc;
  if (L < 0 || L > B) return set_error(RBG_EINVAL, "list length L=%lld outside [0, B=%lld]", (long long)L, (long long)B);
  if (L == 0) return RBG_OK;  // an empty list has no buffers to check
  if ((rc = check_state(state, "state", G))) return rc;
  if (!action) return set_error(RBG_EINVAL, "action is NULL");
  if (!order_in) return set_error(RBG_EINVAL, "order_in is NULL");
  if (!order_out) return set_error(RBG_EINVAL, "order_out is NULL");
  if (!count_out) return set_error(RBG_EINVAL, "count_out is NULL");
  if (order_in < order_out + L && order_out < order_in + L) return set_error(RBG_EINVAL, "order_in and order_out overlap");
  if (!params) return set_error(RBG_EINVAL, "params is NULL");
  if (params->autoreset_kind >= 0)
    return set_error(RBG_EINVAL, "an evaluation step ends an episode at its first LAST step: params->autoreset_kind must be < 0 (got %d)",
                     params->autoreset_kind);
  if (!ts) return set_error(RBG_EINVAL, "timestep is NULL");
  if (!ts->obs_grid || !ts->action_mask || !ts->obs_step_count) return set_error(RBG_EINVAL, "timestep has a NULL observation field");
  if ((G * G) % 4 == 0 && !aligned16(ts->obs_grid)) return set_error(RBG_EALIGN, "timestep.obs_grid not 16-byte aligned");
  if ((rc = check_metrics(acc, "acc"))) return rc;
  return launch_eval_step_live(*state, action, order_in, L, order_out, count_out, B, G, N, *params, *ts, *acc, (cudaStream_t)stream);
}

// ---- device-side evaluation loop: a graph whose one node is a WHILE loop around a captured body
struct EvalLoop {
  cudaGraph_t graph = nullptr;
  cudaGraphExec_t exec = nullptr;
  cudaGraphConditionalHandle cond = 0;
};

int rbg_eval_loop_create(void **loop, uint64_t *cond) {
  if (!loop || !cond) return set_error(RBG_EINVAL, "rbg_eval_loop_create: NULL pointer");
  *loop = nullptr;
  EvalLoop *l = new EvalLoop;
  cudaError_t e = cudaGraphCreate(&l->graph, 0);
  if (e == cudaSuccess) e = cudaGraphConditionalHandleCreate(&l->cond, l->graph, 1, cudaGraphCondAssignDefault);
  if (e != cudaSuccess) {
    if (l->graph) cudaGraphDestroy(l->graph);
    delete l;
    return set_cuda_error(e, "rbg_eval_loop_create");
  }
  *loop = l;
  *cond = (uint64_t)l->cond;
  return RBG_OK;
}

int rbg_eval_loop_condition(uint64_t cond, const int32_t *live_count, int32_t *steps, int max_steps, void *stream) {
  if (!live_count || !steps) return set_error(RBG_EINVAL, "rbg_eval_loop_condition: NULL pointer");
  if (max_steps < 1) return set_error(RBG_EINVAL, "rbg_eval_loop_condition: max_steps=%d must be >= 1", max_steps);
  return launch_eval_loop_cond((unsigned long long)cond, live_count, steps, max_steps, (cudaStream_t)stream);
}

int rbg_eval_loop_finalize(void *loop, void *body_graph) {
  if (!loop || !body_graph) return set_error(RBG_EINVAL, "rbg_eval_loop_finalize: NULL pointer");
  EvalLoop *l = static_cast<EvalLoop *>(loop);
  if (l->exec) return set_error(RBG_EINVAL, "rbg_eval_loop_finalize: the loop is already finalized");
  cudaGraphNodeParams np = {};
  np.type = cudaGraphNodeTypeConditional;
  np.conditional.handle = l->cond;
  np.conditional.type = cudaGraphCondTypeWhile;
  np.conditional.size = 1;
  cudaGraphNode_t node, child;
  cudaError_t e = cudaGraphAddNode(&node, l->graph, nullptr, 0, &np);
  if (e != cudaSuccess) return set_cuda_error(e, "rbg_eval_loop_finalize: WHILE node");
  if ((e = cudaGraphAddChildGraphNode(&child, np.conditional.phGraph_out[0], nullptr, 0, static_cast<cudaGraph_t>(body_graph))) != cudaSuccess) {
    cudaGraphDestroyNode(node);
    return set_cuda_error(e, "rbg_eval_loop_finalize: body");
  }
  if ((e = cudaGraphInstantiate(&l->exec, l->graph, 0)) != cudaSuccess) {
    l->exec = nullptr;
    cudaGraphDestroyNode(node);
    return set_cuda_error(e, "rbg_eval_loop_finalize: cudaGraphInstantiate");
  }
  return RBG_OK;
}

int rbg_eval_loop_launch(void *loop, void *stream) {
  if (!loop) return set_error(RBG_EINVAL, "rbg_eval_loop_launch: NULL loop");
  EvalLoop *l = static_cast<EvalLoop *>(loop);
  if (!l->exec) return set_error(RBG_EINVAL, "rbg_eval_loop_launch: the loop has not been finalized (rbg_eval_loop_finalize)");
  const cudaError_t e = cudaGraphLaunch(l->exec, (cudaStream_t)stream);
  return e == cudaSuccess ? RBG_OK : set_cuda_error(e, "rbg_eval_loop_launch: cudaGraphLaunch");
}

int rbg_eval_loop_destroy(void *loop) {
  if (!loop) return set_error(RBG_EINVAL, "rbg_eval_loop_destroy: NULL loop");
  EvalLoop *l = static_cast<EvalLoop *>(loop);
  if (l->exec) cudaGraphExecDestroy(l->exec);
  if (l->graph) cudaGraphDestroy(l->graph);
  delete l;
  return RBG_OK;
}

int rbg_random_actions(const rbg_state *state, int64_t B, int G, int N, int32_t *action, void *stream) {
  int rc;
  if ((rc = check_dims(B, G, N, 1))) return rc;
  if (B == 0) return RBG_OK;  // an empty batch has no buffers to check
  if ((rc = check_state(state, "state", G))) return rc;
  if (!action) return set_error(RBG_EINVAL, "action is NULL");
  return launch_random_actions(*state, B, G, N, action, (cudaStream_t)stream);
}

int rbg_validate(const int32_t *boards, int64_t B, int G, int N, int32_t *flags, void *stream) {
  int rc;
  if ((rc = check_dims(B, G, N, 0))) return rc;
  if (B == 0) return RBG_OK;  // an empty batch has no buffers to check
  if (!boards || !flags) return set_error(RBG_EINVAL, "rbg_validate: NULL pointer");
  return launch_validate(boards, B, G, N, flags, (cudaStream_t)stream);
}

int rbg_board_statistics(const int32_t *boards, int64_t B, int G, int count_current_wire, int32_t *scored, int32_t *detours, int32_t *diversity,
                         void *stream) {
  int rc;
  if ((rc = check_dims(B, G, 1, 0))) return rc;
  if (B == 0) return RBG_OK;
  if (!boards || !detours || !diversity) return set_error(RBG_EINVAL, "rbg_board_statistics: NULL pointer");
  return launch_board_stats(boards, B, G, count_current_wire, scored, detours, diversity, (cudaStream_t)stream);
}

// ---------------------------------------------------------------- _host
void *rbg_host_alloc(int64_t bytes) {
  void *p = nullptr;
  if (cudaMallocHost(&p, (size_t)bytes) != cudaSuccess) {
    set_error(RBG_ENOMEM, "cudaMallocHost(%lld) failed", (long long)bytes);
    return nullptr;
  }
  return p;
}
void rbg_host_free(void *p) {
  if (p) cudaFreeHost(p);
}

static int use_device(int device, int *cur) {
  cudaError_t e = cudaGetDevice(cur);
  if (e != cudaSuccess) return set_cuda_error(e, "cudaGetDevice (no CUDA device: this library has no CPU path)");
  if (device >= 0 && device != *cur) {
    e = cudaSetDevice(device);
    if (e != cudaSuccess) return set_cuda_error(e, "cudaSetDevice");
    *cur = device;
  }
  if (*cur < 0 || *cur >= kMaxDevices) return set_error(RBG_EINVAL, "device %d out of range", *cur);
  g_hc = &g_host[*cur];
  return RBG_OK;
}

// A host-variant call is about to use the scratch as `sig` describes.  If that is not how it was
// used last, the auto-reset workspaces a step variant keeps in it (`nws` of them, `stride` bytes
// apart from `ws`) hold someone else's bytes: their contexts are invalidated.
static void scratch_claim(const ScratchSig &sig, uint8_t *ws, size_t stride, int64_t nws) {
  if (g_hc->sig == sig) return;
  g_hc->sig = sig;
  for (int64_t i = 0; i < nws; ++i) invalidate_workspace(ws + (size_t)i * stride);
}

int rbg_prw_generate_host(const uint32_t *keys, int64_t B, int G, int N, int32_t *heads, int32_t *targets,
                          int32_t *solved, int device) {
  int rc, dev;
  if ((rc = check_dims(B, G, N, 1))) return rc;
  if (B == 0) return RBG_OK;  // an empty batch has no buffers to check
  if (!keys || !heads || !targets || !solved) return set_error(RBG_EINVAL, "rbg_prw_generate_host: NULL pointer");
  if ((rc = use_device(device, &dev))) return rc;
  std::lock_guard<std::mutex> lock(g_scratch_mu);
  uint32_t *dk;
  int32_t *dh, *dt, *ds;
  void *base;
  rc = scratch_carve(dev, &base, [&](Carver &c) {
    dk = c.take<uint32_t>((size_t)B * 2);
    dh = c.take<int32_t>((size_t)B * 2 * N);
    dt = c.take<int32_t>((size_t)B * 2 * N);
    ds = c.take<int32_t>((size_t)B * G * G);
  });
  if (rc) return rc;
  scratch_claim(ScratchSig{1, B, G, N, -1, base}, nullptr, 0, 0);
  const int nsl = B >= 4096 ? 4 : 1;
  const int64_t sl = slice_size(B, nsl);
  rc = [&]() -> int {
    int si = 0;
    for (int64_t off = 0; off < B; off += sl, ++si) {
      const int64_t n = (B - off) < sl ? (B - off) : sl;
      cudaStream_t st = g_hc->streams[si % 3];
      RBG_CPY(dk + off * 2, keys + off * 2, n * 8, cudaMemcpyHostToDevice, st);
      int r = rbg_prw_generate(dk + off * 2, n, G, N, dh + off * 2 * N, dt + off * 2 * N, ds + off * G * G, nullptr, st);
      if (r) return r;
      RBG_CPY(heads + off * 2 * N, dh + off * 2 * N, n * 2 * N * 4, cudaMemcpyDeviceToHost, st);
      RBG_CPY(targets + off * 2 * N, dt + off * 2 * N, n * 2 * N * 4, cudaMemcpyDeviceToHost, st);
      RBG_CPY(solved + off * G * G, ds + off * G * G, n * G * G * 4, cudaMemcpyDeviceToHost, st);
    }
    return RBG_OK;
  }();
  return rc ? fail_synced(rc) : sync_streams();
}

// The generator kinds rbg_connector_reset_host can run (the dataset kind needs its boards: rbg_connector_reset_dataset),
// and the auto-reset kinds of the step variants; checked before any CUDA call.
static int check_host_reset_kind(int kind) {
  if (kind == RBG_GEN_DATASET)
    return set_error(RBG_EINVAL, "rbg_connector_reset_host: RBG_GEN_DATASET needs the dataset's boards (rbg_connector_reset_dataset)");
  if (kind < RBG_GEN_PRW || kind > RBG_GEN_SEQRW) return set_error(RBG_EINVAL, "rbg_connector_reset_host: unknown generator kind %d", kind);
  return RBG_OK;
}
static int check_host_params(const rbg_env_params *params) {
  if (params->autoreset_kind > RBG_GEN_SEQRW) return set_error(RBG_EINVAL, "unknown autoreset generator kind %d", params->autoreset_kind);
  return params->autoreset_kind == RBG_GEN_DATASET ? check_dataset(params) : RBG_OK;
}

int rbg_connector_reset_host(int kind, const uint32_t *keys, int64_t B, int G, int N, const rbg_state *state,
                             const rbg_timestep *ts, int device) {
  int rc, dev;
  if ((rc = check_dims(B, G, N, kind == RBG_GEN_UNIFORM ? 2 : 1))) return rc;
  if (B == 0) return RBG_OK;  // an empty batch has no buffers to check
  if (!keys || !state || !ts) return set_error(RBG_EINVAL, "rbg_connector_reset_host: NULL pointer");
  if ((rc = check_host_reset_kind(kind))) return rc;
  if ((rc = use_device(device, &dev))) return rc;
  std::lock_guard<std::mutex> lock(g_scratch_mu);
  uint32_t *dk;
  rbg_state ds;
  rbg_timestep dt;
  void *base;
  rc = scratch_carve(dev, &base, [&](Carver &c) {
    dk = c.take<uint32_t>((size_t)B * 2);
    carve_state(c, B, G, N, &ds);
    carve_timestep(c, B, G, N, &dt);
  });
  if (rc) return rc;
  scratch_claim(ScratchSig{2, B, G, N, kind, base}, nullptr, 0, 0);
  const int nsl = B >= 4096 ? 4 : 1;
  const int64_t sl = slice_size(B, nsl);
  rc = [&]() -> int {
    int si = 0, r;
    for (int64_t off = 0; off < B; off += sl, ++si) {
      const int64_t n = (B - off) < sl ? (B - off) : sl;
      cudaStream_t st = g_hc->streams[si % 3];
      RBG_CPY(dk + off * 2, keys + off * 2, n * 8, cudaMemcpyHostToDevice, st);
      rbg_state dss = state_at(ds, off, G, N);
      rbg_timestep dts = timestep_at(dt, off, G, N);
      if ((r = rbg_connector_reset(kind, dk + off * 2, n, G, N, &dss, &dts, st))) return r;
      if ((r = copy_state(state, &ds, off, n, G, N, cudaMemcpyDeviceToHost, off, st))) return r;
      if ((r = copy_timestep(ts, &dt, off, n, G, N, cudaMemcpyDeviceToHost, off, st))) return r;
    }
    return RBG_OK;
  }();
  return rc ? fail_synced(rc) : sync_streams();
}

int rbg_connector_step_host(const rbg_state *in, const rbg_state *out, const int32_t *action, int64_t B, int G,
                            int N, const rbg_env_params *params, const rbg_timestep *ts, int device) {
  int rc, dev;
  if ((rc = check_dims(B, G, N, 1))) return rc;
  if (B == 0) return RBG_OK;  // an empty batch has no buffers to check
  if (!in || !out || !action || !params || !ts) return set_error(RBG_EINVAL, "rbg_connector_step_host: NULL pointer");
  if ((rc = check_host_params(params))) return rc;
  if ((rc = use_device(device, &dev))) return rc;
  std::lock_guard<std::mutex> lock(g_scratch_mu);
  const int nsl = B >= 4096 ? 8 : 1;
  const int64_t sl = slice_size(B, nsl);
  const int64_t nslices = (B + sl - 1) / sl;
  const size_t ws_bytes = (size_t)rbg_step_workspace_bytes(sl, G, N);
  rbg_state ds;
  rbg_timestep dt;
  int32_t *da;
  uint8_t *ws;
  void *base;
  rc = scratch_carve(dev, &base, [&](Carver &c) {
    carve_state(c, B, G, N, &ds);
    carve_timestep(c, B, G, N, &dt);
    da = c.take<int32_t>((size_t)B * N);
    ws = c.take<uint8_t>((size_t)nslices * ws_bytes);
  });
  if (rc) return rc;
  scratch_claim(ScratchSig{3, B, G, N, params->autoreset_kind, base}, ws, ws_bytes, nslices);
  rc = [&]() -> int {
    int si = 0, r;
    for (int64_t off = 0; off < B; off += sl, ++si) {
      const int64_t n = (B - off) < sl ? (B - off) : sl;
      cudaStream_t st = g_hc->streams[si % 3];
      if ((r = copy_state(&ds, in, off, n, G, N, cudaMemcpyHostToDevice, off, st))) return r;
      RBG_CPY(da + off * N, action + off * N, n * N * 4, cudaMemcpyHostToDevice, st);
      rbg_state dss = state_at(ds, off, G, N);
      rbg_timestep dts = timestep_at(dt, off, G, N);
      if ((r = rbg_connector_step(&dss, &dss, da + off * N, n, G, N, params, &dts, ws + (size_t)si * ws_bytes, st))) return r;
      if ((r = copy_state(out, &ds, off, n, G, N, cudaMemcpyDeviceToHost, off, st))) return r;
      if ((r = copy_timestep(ts, &dt, off, n, G, N, cudaMemcpyDeviceToHost, off, st))) return r;
    }
    return RBG_OK;
  }();
  return rc ? fail_synced(rc) : sync_streams();
}

// Env-pool style step: the State stays on the device (updated in place), the actions come from and
// the TimeStep goes to HOST buffers, pipelined over env slices on three streams.
int rbg_connector_step_host_io(const rbg_state *state, const int32_t *action, int64_t B, int G, int N,
                               const rbg_env_params *params, const rbg_timestep *ts, int device) {
  int rc, dev;
  if ((rc = check_dims(B, G, N, 1))) return rc;
  if (B == 0) return RBG_OK;  // an empty batch has no buffers to check
  if (!action || !params || !ts) return set_error(RBG_EINVAL, "rbg_connector_step_host_io: NULL pointer");
  if ((rc = check_state(state, "state", G))) return rc;
  if ((rc = check_host_params(params))) return rc;
  if ((rc = use_device(device, &dev))) return rc;
  std::lock_guard<std::mutex> lock(g_scratch_mu);
  cudaError_t e;
  const auto t_call0 = std::chrono::steady_clock::now();
  int tune_slot = -1;  // which candidate this call measures (odd calls of the tuning phase)
  if (!host_pool_fixed() && host_pool_max_threads() >= 4) {
    const int64_t key = B * 4096 + (int64_t)G * 64 + N;
    if (g_hc->tune_B != key) {
      g_hc->tune_B = key;
      g_hc->tune_call = 0;
      g_hc->tune_best = 0;
      g_hc->tune_best_s = 0.0;
    }
    // candidates: a big pool (one rank per host) tries 1/4, 3/8 and 1/2 of the cores: beyond half of them the calling thread
    // (which polls the copy events), the driver's threads and whatever else the process runs collide with the workers and
    // the step becomes bimodal (16-core boxes: 8 threads 61-66 M env-steps/s; 12 threads 35-58 M; 16 threads 25-44 M).  A
    // small pool (several ranks share the host) tries 1/4, 1/2, 3/4 and all of its few workers.
    const bool big = host_pool_max_threads() >= 8;
    const int ncand = big ? 3 : 4;
    if (g_hc->tune_call < 4 * ncand) {
      const int cand = g_hc->tune_call / 4;  // four calls each, the last three timed
      int n = big ? host_pool_max_threads() * (cand + 2) / 8 : host_pool_max_threads() * (cand + 1) / 4;
      host_pool_set_threads(n < 1 ? 1 : n);
      if (g_hc->tune_call & 3) tune_slot = cand;
      g_hc->tune_call++;
    } else if (g_hc->tune_call == 4 * ncand) {
      host_pool_set_threads(g_hc->tune_best ? g_hc->tune_best : (host_pool_max_threads() + 1) / 2);
      g_hc->tune_call++;
    }
  }
  // 16 slices for big batches: the host starts widening after 1/16 of the copies and ends 1/16 after them (measured at
  // 65 536 envs 10x10/5: 8 slices 1.27-1.6 ms per step, 16 slices 1.17-1.24 ms)
  const int nsl = B >= 32768 ? 16 : B >= 4096 ? 8 : 1;
  const int64_t sl = slice_size(B, nsl);
  const int64_t nslices = (B + sl - 1) / sl;
  const size_t obs_n = (size_t)B * N * G * G;
  const size_t ws_bytes = (size_t)rbg_step_workspace_bytes(sl, G, N);
  rbg_timestep dt;
  int32_t *da;
  uint8_t *ws, *obs8;
  void *base;
  rc = scratch_carve(dev, &base, [&](Carver &c) {
    carve_timestep(c, B, G, N, &dt);
    da = c.take<int32_t>((size_t)B * N);
    ws = c.take<uint8_t>((size_t)nslices * ws_bytes);
    obs8 = c.take<uint8_t>(obs_n);
  });
  if (rc) return rc;
  scratch_claim(ScratchSig{4, B, G, N, params->autoreset_kind, base}, ws, ws_bytes, nslices);
  if (g_hc->stage8_bytes < obs_n) {
    if (g_hc->stage8) cudaFreeHost(g_hc->stage8);
    g_hc->stage8 = nullptr;
    g_hc->stage8_bytes = 0;
    if ((e = cudaHostAlloc(reinterpret_cast<void **>(&g_hc->stage8), obs_n, cudaHostAllocDefault)) != cudaSuccess) return set_cuda_error(e, "cudaHostAlloc(observation staging)");
    g_hc->stage8_bytes = obs_n;
  }
  // One compute stream runs the slices' kernels back to back (the whole batch is ~0.1 ms of kernels); the two
  // copy streams take the observation (96 % of the bytes) of each slice as soon as its kernel is done, so the
  // bus is busy from the first slice on.  The small leaves go once for the whole batch: 8 copies instead of 8 per
  // slice.  The observation's codes cross the bus as bytes into a pinned staging buffer and the host pool widens
  // slice s into the caller's int32 buffer while slices s+1.. are in flight; the caller's observation buffer need
  // not be pinned.
  cudaEvent_t *slice_ev = g_hc->slice_ev, *copy_ev = g_hc->copy_ev;
  cudaStream_t cs = g_hc->streams[0];
  // The State was produced by the caller on the device's default stream (or a stream that stream synchronises
  // with: every blocking stream does): our compute stream is ordered behind it by an event, the host does not wait.
  if (!g_hc->entry_ev && (e = cudaEventCreateWithFlags(&g_hc->entry_ev, cudaEventDisableTiming)) != cudaSuccess) return set_cuda_error(e, "cudaEventCreate");
  if ((e = cudaEventRecord(g_hc->entry_ev, cudaStreamLegacy)) != cudaSuccess) return set_cuda_error(e, "cudaEventRecord(entry)");
  if ((e = cudaStreamWaitEvent(cs, g_hc->entry_ev, 0)) != cudaSuccess) return set_cuda_error(e, "cudaStreamWaitEvent(entry)");
  RBG_CPY(da, action, (size_t)B * N * 4, cudaMemcpyHostToDevice, cs);
  g_h2d_bytes.fetch_add((long long)B * N * 4, std::memory_order_relaxed);
  const size_t per_env = (size_t)N * G * G;
  // Observation codes are <= 3 N: with at most 5 agents they fit a nibble, two cells per byte over the bus (a slice is a
  // multiple of 64 envs, so every slice starts on a whole, 16-byte aligned byte when an env has an even number of cells).
  const int obits = (3 * N <= 15 && (per_env & 1u) == 0) ? 4 : 8;
  const int oshift = obits == 4 ? 1 : 0;
  rc = [&]() -> int {
    int si = 0, r;
    for (int64_t off = 0; off < B; off += sl, ++si) {
      const int64_t n = (B - off) < sl ? (B - off) : sl;
      const size_t codes_off = ((size_t)off * per_env) >> oshift;
      rbg_state dss = state_at(*state, off, G, N);
      rbg_timestep dts = timestep_at(dt, off, G, N);
      if ((r = rbg_connector_step(&dss, &dss, da + off * N, n, G, N, params, &dts, ws + (size_t)si * ws_bytes, cs))) return r;
      if ((r = launch_narrow_codes(dts.obs_grid, obs8 + codes_off, (int64_t)((size_t)n * per_env), cs, obits))) return r;
      if (!slice_ev[si] && (e = cudaEventCreateWithFlags(&slice_ev[si], cudaEventDisableTiming)) != cudaSuccess) return set_cuda_error(e, "cudaEventCreate");
      if ((e = cudaEventRecord(slice_ev[si], cs)) != cudaSuccess) return set_cuda_error(e, "cudaEventRecord");
      cudaStream_t xs = g_hc->streams[1 + (si & 1)];
      if ((e = cudaStreamWaitEvent(xs, slice_ev[si], 0)) != cudaSuccess) return set_cuda_error(e, "cudaStreamWaitEvent");
      RBG_CPY(g_hc->stage8 + codes_off, obs8 + codes_off, ((size_t)n * per_env) >> oshift, cudaMemcpyDeviceToHost, xs);
      if (!copy_ev[si] && (e = cudaEventCreateWithFlags(&copy_ev[si], cudaEventDisableTiming)) != cudaSuccess) return set_cuda_error(e, "cudaEventCreate");
      if ((e = cudaEventRecord(copy_ev[si], xs)) != cudaSuccess) return set_cuda_error(e, "cudaEventRecord(copy)");
    }
    return copy_timestep(ts, &dt, 0, B, G, N, cudaMemcpyDeviceToHost, 0, cs, false);
  }();
  if (rc) return fail_synced(rc);
  g_d2h_bytes.fetch_add((long long)(obs_n >> oshift) + (long long)B * (N * 5 + 4 + N * 8 + 1 + 12), std::memory_order_relaxed);
  int si = 0;
  for (int64_t off = 0; off < B; off += sl, ++si) {
    const int64_t n = (B - off) < sl ? (B - off) : sl;
    if ((e = cudaEventSynchronize(copy_ev[si])) != cudaSuccess) {
      host_pool_wait();
      return set_cuda_error(e, "cudaEventSynchronize(copy)");
    }
    const size_t codes_off = ((size_t)off * per_env) >> oshift;
    if (obits == 4)
      host_pool_widen4(g_hc->stage8 + codes_off, ts->obs_grid + (size_t)off * per_env, (size_t)n * per_env);
    else
      host_pool_widen(g_hc->stage8 + codes_off, ts->obs_grid + (size_t)off * per_env, (size_t)n * per_env);
  }
  rc = sync_streams();
  host_pool_wait();
  if (tune_slot >= 0 && rc == RBG_OK) {
    const double dt = std::chrono::duration<double>(std::chrono::steady_clock::now() - t_call0).count();
    // the fastest call decides; a larger thread count must beat a smaller one by 1 % to replace it (the candidates of a
    // single-rank host stop at half of the cores, where more threads still help: 6 / 8 threads 65.4 / 68.1 M env-steps/s)
    const int nthr = host_pool_threads();
    if (g_hc->tune_best == 0 || (nthr == g_hc->tune_best ? dt < g_hc->tune_best_s : dt < 0.99 * g_hc->tune_best_s)) {
      g_hc->tune_best = nthr;
      g_hc->tune_best_s = dt;
    }
  }
  return rc;
}

int rbg_host_widen(const uint8_t *src, int32_t *dst, int64_t n) {
  if (n < 0 || (n > 0 && (!src || !dst))) return set_error(RBG_EINVAL, "rbg_host_widen: n=%lld, src=%p, dst=%p", (long long)n, (const void *)src, (void *)dst);
  if (n == 0) return RBG_OK;
  host_pool_widen(src, dst, (size_t)n);
  host_pool_wait();
  return RBG_OK;
}

int rbg_host_widen4(const uint8_t *src, int32_t *dst, int64_t n) {
  if (n < 0 || (n & 1) || (n > 0 && (!src || !dst))) return set_error(RBG_EINVAL, "rbg_host_widen4: n=%lld (even), src=%p, dst=%p", (long long)n, (const void *)src, (void *)dst);
  if (n == 0) return RBG_OK;
  host_pool_widen4(src, dst, (size_t)n);
  host_pool_wait();
  return RBG_OK;
}

int rbg_host_transfer_stats(int64_t *h2d_bytes, int64_t *d2h_bytes, int *host_threads, int reset) {
  if (h2d_bytes) *h2d_bytes = reset ? g_h2d_bytes.exchange(0) : g_h2d_bytes.load();
  if (d2h_bytes) *d2h_bytes = reset ? g_d2h_bytes.exchange(0) : g_d2h_bytes.load();
  if (host_threads) *host_threads = host_pool_threads();
  return RBG_OK;
}

}  // extern "C"
