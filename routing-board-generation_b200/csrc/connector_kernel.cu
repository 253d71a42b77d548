// connector_kernel.cu -- Jumanji Connector step / observe for sm_100a.
//
// Replaces jit(vmap(Connector.step)) and the observation half of
// jit(vmap(Connector.reset)) (jumanji==0.2.2 environments/routing/connector/
// env.py -- UPSTREAM; reference call sites rl_training/setup_train.py:158-166,400,
// demos/board_generator_demo.py:83-96; the agent-stepping / collision rule is
// mirrored in the reference at parallel_random_walk.py:101-145,376-429).
//
// One launch fuses: (optional) random-policy action sampling, _step_agents
// with the collision rule, step_count, DenseRewardFn, action mask, done /
// discount / step_type, extras, the per-agent observation and (with
// auto-reset) the compaction of finished envs into a reset list.
//
// The kernels are HBM-write bound by bytes (DESIGN.md "K2", "K2b"): the per-step
// kernel reads the State once (int32 -> uint8 into shared memory) and writes State +
// observation [N,G,G] int32 exactly once; the fused rollout kernel keeps the State on
// chip for a whole chunk of steps.  All bulk traffic is 128-bit coalesced.
#include <cuda/atomic>

#include "connector_device.cuh"
#include "gen_warp.cuh"
#include "obs_stage.cuh"
#include "rbg_host.h"

namespace rbg {

// row stride of the per-step kernel's observation table: codes 0..3N, rounded up to whole words
__host__ __device__ inline int obs_lut_stride(int N) { return (3 * N + 1 + 3) & ~3; }

// number of PATH codes (v % 3 == 1) among the four byte codes of a packed word,
// two 16-bit lanes at a time: x / 3 == (x * 171) >> 9 for x < 256
__device__ __forceinline__ int count_path_codes(uint32_t w) {
  const uint32_t e = w & 0x00FF00FFu, o = (w >> 8) & 0x00FF00FFu;
  const uint32_t re = e - 3u * (((e * 171u) >> 9) & 0x007F007Fu);
  const uint32_t ro = o - 3u * (((o * 171u) >> 9) & 0x007F007Fu);
  const uint32_t ie = re & ~(re >> 1) & 0x00010001u, io = ro & ~(ro >> 1) & 0x00010001u;
  return __popc(ie | (io << 1));
}

// uniform pick over the legal actions, NOOP included (include/rbg_b200.h
// rbg_random_actions): mk bit (a-1) <=> action a legal.
__device__ __forceinline__ int random_action(uint32_t k0, uint32_t k1,
                                             uint32_t step, uint32_t agent,
                                             uint32_t mk) {
  uint32_t o0, o1;
  tf_block(k0, k1, step, agent, o0, o1);
  const uint32_t n = 1u + __popc(mk);
  const int pick = (int)__umulhi(o0, n);  // 0 = NOOP, k = the k-th legal move in action order
  if (pick == 0) return NOOP;
  uint32_t b = mk;
  if (pick > 1) b &= b - 1u;
  if (pick > 2) b &= b - 1u;
  if (pick > 3) b &= b - 1u;
  return __ffs((int)b);
}

// ---------------------------------------------------------------------------
// The phases of one Connector step in the warp-per-K-envs layout that every kernel below uses: a warp owns
// K = 32 / Np envs (Np = lanes per env, the next power of two >= N), lane = (env j, agent a), and the env grids are
// uint8 codes in the warp's slice of shared memory, env j at wg + j * cells.

// observation table: row x maps a grid code v (0..3N) to agent x's view of it; rows are RS bytes apart
__device__ __forceinline__ void build_obs_lut(uint8_t *lut, int N, int RS, int warp, int nwarps, int lane) {
  for (int x = warp; x < N; x += nwarps)
    for (int v = lane; v < RS; v += 32) lut[x * RS + v] = v <= 3 * N ? (uint8_t)obs_value(v, 3 * x, 3 * N) : (uint8_t)0;
}

// State.grid int32 of envs e0 .. e0 + kc - 1 -> the warp's uint8 grids (VEC: one packed word per int4)
template <bool VEC>
__device__ __forceinline__ void load_grids(const int32_t *grid, long long e0, int kc, int cells, int lane, uint8_t *wg) {
  if (VEC) {
    // four loads in flight per lane before the first one is used (a load-use pair per iteration
    // made a warp pay one L2 round trip per 32 words: 19 % of the kernel's stall samples)
    uint32_t *wg32 = reinterpret_cast<uint32_t *>(wg);
    const int4 *src = reinterpret_cast<const int4 *>(grid) + e0 * (cells >> 2);
    const int nq = kc * (cells >> 2);
    for (int q0 = lane; q0 < nq; q0 += 128) {
      int4 v[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) v[u] = (q0 + 32 * u < nq) ? __ldg(src + q0 + 32 * u) : make_int4(0, 0, 0, 0);
#pragma unroll
      for (int u = 0; u < 4; ++u)
        if (q0 + 32 * u < nq)
          wg32[q0 + 32 * u] = (uint32_t)(v[u].x & 0xff) | ((uint32_t)(v[u].y & 0xff) << 8) | ((uint32_t)(v[u].z & 0xff) << 16) | ((uint32_t)(v[u].w & 0xff) << 24);
    }
  } else {
    const int32_t *src = grid + e0 * cells;
    for (int i = lane; i < kc * cells; i += 32) wg[i] = (uint8_t)__ldg(src + i);
  }
}

// PATH cells of env j (extras: total_path_length), summed over the env's Np lanes
template <bool VEC>
__device__ __forceinline__ int count_paths(const uint8_t *wg, int j, int a, int cells, int c4, int Np, bool env_ok) {
  int paths = 0;
  if (env_ok) {
    if (VEC) {
      const uint32_t *wg32 = reinterpret_cast<const uint32_t *>(wg);
      for (int q = a; q < c4; q += Np) paths += count_path_codes(wg32[j * c4 + q]);
    } else {
      const uint8_t *g = wg + (size_t)j * cells;
      for (int i = a; i < cells; i += Np) paths += (g[i] % 3u == 1u) ? 1 : 0;
    }
  }
  for (int off = Np >> 1; off; off >>= 1) paths += __shfl_xor_sync(FULL, paths, off);
  return paths;
}

// destination cell of a random-policy action (-1: none), the action written to out[row] if out is set.  mk is
// is_valid_position of the four moves on this very grid (empty for a connected agent), so a non-NOOP action needs no
// second validity test.
__device__ __forceinline__ int random_dest(uint32_t k0, uint32_t k1, int sc, int a, uint32_t mk, int r, int c, int G, int32_t *out,
                                           long long row) {
  const int action = random_action(k0, k1, (uint32_t)sc, (uint32_t)a, mk);
  if (out) out[row] = action;
  return action != NOOP ? r * G + c + (action == UP ? -G : (action == DOWN ? G : (action == RIGHT ? 1 : -1))) : -1;
}

// two cells of a G x G grid in one register (ObsStager::emit_delta); pin_cell: the cell of a packed (row << 8 | col)
__device__ __forceinline__ uint32_t cell_pair(int c0, int c1) { return (uint32_t)c0 | ((uint32_t)c1 << 16); }
__device__ __forceinline__ int pin_cell(int rc, int G) { return (rc >> 8) * G + (rc & 255); }

// the collision rule and move_agent: of the agents of one env with the same destination only the highest agent id
// moves; a mover's old head becomes PATH and its new cell POSITION on the env grid g.  Returns the lane's position
// after the move; win: it moved.
__device__ __forceinline__ int resolve_moves(int dest, int j, int lane, int a, int r, int c, int G, uint8_t *g, const FastDiv &divG, int pos,
                                             bool &win) {
  const uint32_t mval = dest >= 0 ? (((uint32_t)j << 16) | (uint32_t)dest) : (0x80000000u | (uint32_t)lane);
  const uint32_t mm = __match_any_sync(FULL, mval);
  win = dest >= 0 && lane == 31 - __clz(mm);
  __syncwarp();  // every read of the pre-move grid is done
  if (win) {
    g[r * G + c] = (uint8_t)(3 * a + PATH);
    g[dest] = (uint8_t)(3 * a + POSITION);
    uint32_t nr, nc;
    divG.divmod((uint32_t)dest, nr, nc);
    pos = (int)((nr << 8) | nc);
  }
  __syncwarp();
  return pos;
}

// what the step leaves on the new grid: per agent, per env (group-uniform counts)
struct StepResult {
  uint32_t mk3;  // action mask (bit m-1: move m legal)
  bool done;     // connected_or_blocked
  float rew;     // DenseRewardFn
  int ndone, nconn, nmoved;
};

// rw: anything with the env's connected_reward and timestep_reward (rbg_env_params, EpisodeParams, EvalStepParams)
template <class Rewards>
__device__ __forceinline__ StepResult after_move(const SmemGrid &sg, bool agent, int a, int pos, int tgt, bool was, bool win, uint32_t gmask,
                                                 const Rewards &rw) {
  const bool now = agent && pos == tgt;
  uint32_t mk3 = 0;
  if (agent) mk3 = move_mask(sg, pos >> 8, pos & 255, a, now);
  const bool done = now || mk3 == 0u;
  const float rew = __fadd_rn(__fmul_rn(rw.connected_reward, (!was && now) ? 1.0f : 0.0f), __fmul_rn(rw.timestep_reward, was ? 0.0f : 1.0f));
  const int ndone = __popc(__ballot_sync(FULL, agent && done) & gmask);
  const int nconn = __popc(__ballot_sync(FULL, now) & gmask);
  const int nmoved = __popc(__ballot_sync(FULL, win) & gmask);
  return StepResult{mk3, done, rew, ndone, nconn, nmoved};
}

// swap in a new episode (group-uniform): env grid g holds only the pins, heads then targets (PRWG:63-64); returns the
// fresh action mask of agent a at pos (lanes a >= N return mk3 as it is).  cleared() runs once the grid is cleared,
// before the pins go in.
template <class F>
__device__ __forceinline__ uint32_t place_episode(uint8_t *g, const SmemGrid &sg, int a, int N, int Np, int cells, int G, uint32_t gmask,
                                                  int pos, int tgt, uint32_t mk3, F cleared) {
  for (int i = a; i < cells; i += Np) g[i] = 0;
  cleared();
  __syncwarp(gmask);
  if (a < N) g[(pos >> 8) * G + (pos & 255)] = (uint8_t)(3 * a + POSITION);
  __syncwarp(gmask);
  if (a < N) g[(tgt >> 8) * G + (tgt & 255)] = (uint8_t)(3 * a + TARGET);
  __syncwarp(gmask);
  if (a < N) mk3 = move_mask(sg, pos >> 8, pos & 255, a, pos == tgt);
  return mk3;
}

// observation.grid of kc envs through the table, one store per cell (cells % 4 != 0); env m is skipped where bit
// m * Np of skipm is set.  Env m goes to row m of odst, or to row rows[m] when a row table is given.
__device__ __forceinline__ void write_obs_scalar(int32_t *odst, const uint8_t *wg, const uint8_t *lut, int RS, int kc, int cells, int N, int Np,
                                                 uint32_t skipm, const FastDiv &divCells, int lane, const int *rows = nullptr) {
  for (int i = lane; i < kc * cells; i += 32) {
    const int m = (int)divCells.div((uint32_t)i);
    if ((skipm >> (m * Np)) & 1u) continue;
    const uint32_t v = wg[i];
    int32_t *o = odst + (size_t)(rows ? rows[m] : m) * N * cells + (i - m * cells);
    for (int x = 0; x < N; ++x, o += cells) *o = lut[x * RS + v];
  }
}

// the State at the end of a rollout, written once: the warp's grids, and per env / agent what the steps moved
template <bool VEC>
__device__ __forceinline__ void write_state_once(const rbg_state &out, const uint8_t *wg, long long e0, int kc, int cells, int lane, long long e,
                                                 int N, int a, bool env_ok, bool agent, int pos, int tgt, int start, int sc, uint32_t k0, uint32_t k1) {
  if (VEC) {
    const uint32_t *wg32 = reinterpret_cast<const uint32_t *>(wg);
    int4 *gdst = reinterpret_cast<int4 *>(out.grid) + e0 * (cells >> 2);
    for (int q = lane; q < kc * (cells >> 2); q += 32) gdst[q] = bytes_to_int4(wg32[q]);
  } else {
    int32_t *gdst = out.grid + e0 * cells;
    for (int i = lane; i < kc * cells; i += 32) gdst[i] = wg[i];
  }
  if (env_ok && a == 0) {
    out.step_count[e] = sc;
    out.key[2 * e] = k0;
    out.key[2 * e + 1] = k1;
  }
  if (agent) {
    const long long ga = e * N + a;
    reinterpret_cast<int2 *>(out.position)[ga] = make_int2(pos >> 8, pos & 255);
    reinterpret_cast<int2 *>(out.target)[ga] = make_int2(tgt >> 8, tgt & 255);
    reinterpret_cast<int2 *>(out.start)[ga] = make_int2(start >> 8, start & 255);
    out.agent_id[ga] = a;
  }
}

// ---------------------------------------------------------------------------
// env_warp_kernel: one Connector step (or observe) per WARP.  A warp owns K = 32 / Np envs
// (Np = lanes per env, the next power of two >= N; lane = (env, agent)), keeps their
// grids in its own slice of shared memory and runs every phase with __syncwarp only,
// so warps in different phases overlap freely (the first, CTA-wide version of this
// kernel spent half of its warp-time at __syncthreads waiting for the agent phases;
// it is in the history, profiles/r01a_env_full.csv is its ncu capture).
constexpr int EW_WARPS = 4;
constexpr int kEnvMinCtas = 12;

template <bool VEC>
__global__ void __launch_bounds__(EW_WARPS * 32, kEnvMinCtas) env_warp_kernel(const EnvParams p) {
  extern __shared__ __align__(16) uint8_t smem_raw[];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int G = p.G, N = p.N, cells = p.cells;
  const int Np = p.Np, K = 32 / Np, c4 = cells >> 2;
  const int RS = obs_lut_stride(N);
  uint8_t *lut = smem_raw;
  build_obs_lut(lut, N, RS, warp, EW_WARPS, lane);
  __syncthreads();  // the only CTA-wide barrier

  const long long e0 = ((long long)blockIdx.x * EW_WARPS + warp) * K;
  if (e0 >= p.B) return;
  const int kc = (int)((p.B - e0) < (long long)K ? (p.B - e0) : (long long)K);
  const bool is_step = (p.mode == ENV_MODE_STEP);
  // BoardDatasetGeneratorJAX resets are a table lookup (a few threefry blocks + N pins): done right here
  const bool ds = is_step && p.env.autoreset_kind == RBG_GEN_DATASET;
  const bool autoreset = is_step && p.env.autoreset_kind >= 0 && (p.list != nullptr || ds);
  const bool inplace_grid = is_step && p.out.grid == p.in.grid;
  uint8_t *wg = smem_raw + p.so[0] + (size_t)warp * p.so[1];
  uint32_t *wg32 = reinterpret_cast<uint32_t *>(wg);

  const int j = lane / Np, a = lane & (Np - 1);
  const bool env_ok = j < kc, agent = env_ok && a < N;
  const long long e = e0 + (env_ok ? j : 0);
  const uint32_t gmask = Np == 32 ? FULL : (((1u << Np) - 1u) << (j * Np));

  // ---- load: State.grid int32 -> uint8, agent and env scalars
  load_grids<VEC>(p.in.grid, e0, kc, cells, lane, wg);
  int pos = 0, tgt = 0, action = 0, sc0 = 0;
  uint32_t k0 = 0, k1 = 0;
  if (agent) {
    const int2 ps = __ldg(reinterpret_cast<const int2 *>(p.in.position) + e * N + a);
    const int2 tg = __ldg(reinterpret_cast<const int2 *>(p.in.target) + e * N + a);
    pos = (ps.x << 8) | ps.y;
    tgt = (tg.x << 8) | tg.y;
    if (is_step && !p.random_policy) action = __ldg(p.action + e * N + a);
  }
  if (env_ok) {
    sc0 = p.in.step_count[e];
    if (is_step) {
      k0 = p.in.key[2 * e];
      k1 = p.in.key[2 * e + 1];
    }
  }
  __syncwarp();

  uint8_t *g = wg + (size_t)j * cells;
  const SmemGrid sg{g, G, 0, G};
  // PATH cells of the env before the move (extras: total_path_length)
  const int paths = count_paths<VEC>(wg, j, a, cells, c4, Np, env_ok);

  // ---- agents: (sample action,) move_position, is_valid_position, collisions
  const bool was = agent && pos == tgt;
  const int r = pos >> 8, c = pos & 255;
  int dest = -1;
  if (is_step && agent) {
    if (p.random_policy) {
      const uint32_t mk = move_mask(sg, r, c, a, was);
      action = random_action(k0, k1, (uint32_t)sc0, (uint32_t)a, mk);
      if (p.action_out) p.action_out[e * N + a] = action;
    }
    const int am = action < 0 ? 0 : (action > 4 ? 4 : action);  // lax.switch clamps
    const int nr = r + (am == UP ? -1 : (am == DOWN ? 1 : 0));
    const int nc = c + (am == RIGHT ? 1 : (am == LEFT ? -1 : 0));
    const bool inb = (unsigned)nr < (unsigned)G && (unsigned)nc < (unsigned)G;
    const uint32_t v = inb ? sg.at(nr, nc) : 0xFFu;
    if (inb && (v == 0u || v == 3u * a + TARGET) && !was && action != NOOP) dest = nr * G + nc;
  }
  // same destination in the same env -> only the highest agent id moves
  const uint32_t mval = dest >= 0 ? (((uint32_t)j << 16) | (uint32_t)dest) : (0x80000000u | (uint32_t)lane);
  const uint32_t mm = __match_any_sync(FULL, mval);
  const bool win = dest >= 0 && lane == 31 - __clz(mm);
  __syncwarp();  // every read of the pre-move grid is done
  if (win) {  // move_agent: old head -> PATH, new cell -> POSITION
    g[r * G + c] = (uint8_t)(3 * a + PATH);
    g[dest] = (uint8_t)(3 * a + POSITION);
    if (inplace_grid) {  // State.grid updated in place: only these two cells change
      int32_t *gg = p.out.grid + e * cells;
      gg[r * G + c] = 3 * a + PATH;
      gg[dest] = 3 * a + POSITION;
    }
    uint32_t nr, nc;
    p.divG.divmod((uint32_t)dest, nr, nc);
    pos = (int)((nr << 8) | nc);
  }
  __syncwarp();

  // ---- action mask, connected / done, reward on the new grid
  const StepResult s = after_move(sg, agent, a, pos, tgt, was, win, gmask, p.env);
  uint32_t mk3 = s.mk3;

  // ---- per env: termination, auto-reset bookkeeping (group-uniform values)
  const int sc = sc0 + (is_step ? 1 : 0);
  const bool terminal = is_step && env_ok && (s.ndone == N || sc >= p.env.time_limit);
  int tflag = terminal ? 1 : 0;
  // The cache entry may be REPLACED by the previous step's refill, which this kernel runs under, e.g. when a
  // State is stepped twice (functional use, inplace=False) or two batches share a workspace.  The entry is
  // a seqlock whose version is its tag: the writer (prw_kernel, to_cache) invalidates the tag, fences,
  // writes key and pins, fences, publishes the new tag; a reader takes the entry only if the tag reads as
  // expected BEFORE and AFTER its own loads of key / pin, and every lane of the env must agree (ballot),
  // otherwise the env goes down the synchronous reset path like any other miss.
  int hit_i = 0;
  uint32_t ck0 = 0, ck1 = 0, cpin = 0;
  if (terminal && autoreset && !ds && p.cache_tag) {
    const unsigned long long want = ((unsigned long long)k1 << 32) | k0;
    if (__ldcg(p.cache_tag + e) == want) {
      __threadfence();
      const uint2 nk = __ldcg(p.cache_key + e);
      ck0 = nk.x;
      ck1 = nk.y;
      if (a < N) cpin = __ldcg(p.cache_pins + e * N + a);
      __threadfence();
      hit_i = __ldcg(p.cache_tag + e) == want ? 1 : 0;
    }
  }
  {
    const uint32_t okm = __ballot_sync(FULL, hit_i != 0) & gmask;
    hit_i = (okm == gmask) ? 1 : 0;
  }
  if (terminal && ds) {
    // VmapAutoResetWrapper._auto_reset: key, _ = split(state.key); then BoardDatasetGeneratorJAX.__call__
    uint32_t a0, a1, b0, b1;
    split2(k0, k1, a0, a1, b0, b1);
    const uint32_t which = dataset_pick(a0, a1, (uint32_t)p.env.dataset_K, ck0, ck1);
    if (a < N) {
      const int32_t *h = p.env.dataset_heads + (size_t)which * 2 * N, *t = p.env.dataset_targets + (size_t)which * 2 * N;
      const int hi = G - 1;
      const int sr = min(max(__ldg(h + a), 0), hi), sc_ = min(max(__ldg(h + N + a), 0), hi);
      const int tr = min(max(__ldg(t + a), 0), hi), tc = min(max(__ldg(t + N + a), 0), hi);
      cpin = ((uint32_t)sr << 24) | ((uint32_t)sc_ << 16) | ((uint32_t)tr << 8) | (uint32_t)tc;
    }
    hit_i = 1;
  }
  if (terminal && autoreset) {
    const bool hit = hit_i != 0;
    uint32_t nk0 = ck0, nk1 = ck1;
    if (!hit) {  // State.key of the next episode: split(split(key)[0])[0]
      uint32_t a0, a1, b0, b1;
      split2(k0, k1, a0, a1, b0, b1);
      split2(a0, a1, nk0, nk1, b0, b1);
    }
    if (a == 0 && !ds) {
      if (!hit) p.list[atomicAdd(p.list_count, 1)] = (int32_t)e;
      if (p.refill_list) {
        const int slot = atomicAdd(p.refill_count, 1);
        p.refill_list[slot] = (int32_t)e;
        p.refill_keys[2 * slot] = nk0;
        p.refill_keys[2 * slot + 1] = nk1;
      }
    }
    if (hit) {
      k0 = nk0;
      k1 = nk1;
    }
    tflag |= hit ? 4 : 2;
  }
  if (tflag & 4) {
    // swap in the cached episode: pins-only grid (heads, then targets: PRWG:63-64),
    // position = start, fresh action mask; reward / discount / step_type / extras stay
    // those of the terminal step
    for (int i = a; i < cells; i += Np) g[i] = 0;
    if (a < N) {
      pos = (int)(cpin >> 16);
      tgt = (int)(cpin & 0xffffu);
    }
    __syncwarp(gmask);
    if (a < N) g[(pos >> 8) * G + (pos & 255)] = (uint8_t)(3 * a + POSITION);
    __syncwarp(gmask);
    if (a < N) g[(tgt >> 8) * G + (tgt & 255)] = (uint8_t)(3 * a + TARGET);
    __syncwarp(gmask);
    if (a < N) mk3 = move_mask(sg, pos >> 8, pos & 255, a, pos == tgt);
  }
  __syncwarp();

  // ---- small outputs
  if (env_ok && a == 0) {
    p.ts.step_type[e] = (int8_t)(is_step ? (terminal ? 2 : 1) : 0);
    p.ts.num_connections[e] = s.nconn;
    p.ts.ratio_connections[e] = __fdiv_rn((float)s.nconn, (float)N);
    p.ts.total_path_length[e] = paths + s.nmoved + N;
    if (!(tflag & 2)) p.ts.obs_step_count[e] = (tflag & 4) ? 0 : sc;
    if (is_step) {
      p.out.step_count[e] = (tflag & 4) ? 0 : sc;
      if (p.out.key != p.in.key || (tflag & 4)) {
        p.out.key[2 * e] = k0;
        p.out.key[2 * e + 1] = k1;
      }
    }
  }
  if (agent) {
    const long long ga = e * N + a;
    p.ts.reward[ga] = is_step ? s.rew : 0.0f;
    p.ts.discount[ga] = is_step ? ((terminal || s.done) ? 0.0f : 1.0f) : 1.0f;
    if (!(tflag & 2)) store_mask5(p.ts.action_mask + ga * 5, mk3);
    if (is_step) {
      const int2 pos2 = make_int2(pos >> 8, pos & 255);
      reinterpret_cast<int2 *>(p.out.position)[ga] = pos2;
      if (tflag & 4) {
        reinterpret_cast<int2 *>(p.out.target)[ga] = make_int2(tgt >> 8, tgt & 255);
        reinterpret_cast<int2 *>(p.out.start)[ga] = pos2;
        p.out.agent_id[ga] = a;
      } else if (p.out.target != p.in.target) {
        reinterpret_cast<int2 *>(p.out.target)[ga] = make_int2(tgt >> 8, tgt & 255);
        reinterpret_cast<int2 *>(p.out.start)[ga] = reinterpret_cast<const int2 *>(p.in.start)[ga];
        p.out.agent_id[ga] = p.in.agent_id[ga];
      }
    }
  }

  // ---- bulk outputs: State.grid and observation.grid
  const uint32_t skipm = __ballot_sync(FULL, a == 0 && (tflag & 2));  // bit j*Np: env j is rewritten by the reset kernel
  const uint32_t hitm = __ballot_sync(FULL, a == 0 && (tflag & 4));
  if (VEC) {
    // (Staging + bulk copies as in the rollout kernel measured SLOWER here, 77 vs 50 us per step: a
    // warp of this kernel lives for one step, so it would wait for its own copy to be read before
    // it may exit; the rollout kernel's hoisted store loop measured the same as this one.)
    int4 *gdst = reinterpret_cast<int4 *>(p.out.grid) + e0 * c4;
    int4 *odst = reinterpret_cast<int4 *>(p.ts.obs_grid) + e0 * N * c4;
    for (int q = lane; q < kc * c4; q += 32) {
      const int m = (int)p.divC4.div((uint32_t)q);
      if ((skipm >> (m * Np)) & 1u) continue;
      const uint32_t w = wg32[q];
      const uint32_t b0 = w & 0xffu, b1 = (w >> 8) & 0xffu, b2 = (w >> 16) & 0xffu, b3 = w >> 24;
      if (is_step && (!inplace_grid || ((hitm >> (m * Np)) & 1u))) gdst[q] = make_int4((int)b0, (int)b1, (int)b2, (int)b3);
      int4 *o = odst + (size_t)m * N * c4 + (q - m * c4);
      const uint8_t *row = lut;
#pragma unroll 2
      for (int x = 0; x < N; ++x, o += c4, row += RS) *o = make_int4(row[b0], row[b1], row[b2], row[b3]);
    }
  } else {
    int32_t *gdst = p.out.grid + e0 * cells;
    int32_t *odst = p.ts.obs_grid + e0 * N * cells;
    for (int i = lane; i < kc * cells; i += 32) {
      const int m = (int)p.divCells.div((uint32_t)i);
      if ((skipm >> (m * Np)) & 1u) continue;
      const uint32_t v = wg[i];
      if (is_step) gdst[i] = (int)v;
      int32_t *o = odst + (size_t)m * N * cells + (i - m * cells);
      for (int x = 0; x < N; ++x, o += cells) *o = lut[x * RS + v];
    }
  }
}

// ---------------------------------------------------------------------------
// rollout_warp_kernel: T random-policy steps with auto-reset from a board dataset
// (BoardDatasetGeneratorJAX) in ONE launch (the reference's `n_steps` scan: reset and
// stepping fused).  Same lane layout as env_warp_kernel, but the warp keeps its K envs on
// chip for the whole rollout: the State is read once and written once per launch, so a
// step only pays for what it must emit (observation, mask, reward, discount, step_type,
// extras, action); PATH counts are carried instead of recounted.  A finished env's next
// episode is a table lookup in the dataset.
struct RolloutParams {
  int T;
  int32_t *action_out;   // [T,B,N] or NULL
  int ratio_off;         // smem byte offset of the n / N table
  int stage_off;         // smem byte offset of the per-warp observation staging
  int stage_bytes;       // bytes per buffer
  int stage_nbuf;        // 1: one chunk per step (a whole step passes before it is refilled); 2: alternate
  int stage_warp;        // bytes per warp (>= stage_nbuf * stage_bytes)
  int ce, cv;            // a staged chunk = ce whole envs (cv == N) or cv views of one env (ce == 1)
  int delta;             // 1: the one buffer holds the warp's whole observation range (nbuf == 1, ce == K), so after the
                         // first step of a group only the cells that changed are restaged (ObsStager::emit_delta)
};

constexpr int kRolloutMinCtas = 6;
// OBS: 0 scalar stores (cells % 4 != 0), 1 direct 128-bit stores, 2 staged + bulk copies (obs_stage.cuh)
template <int OBS>
__global__ void __launch_bounds__(EW_WARPS * 32, kRolloutMinCtas) rollout_warp_kernel(const EnvParams p, const RolloutParams rp) {
  constexpr bool VEC = OBS != 0;
  extern __shared__ __align__(16) uint8_t smem_raw[];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int G = p.G, N = p.N, cells = p.cells;
  const int Np = p.Np, K = 32 / Np, c4 = cells >> 2;
  constexpr int RS = OBS_RS;
  uint8_t *lut = smem_raw;
  build_obs_lut(lut, N, RS, warp, EW_WARPS, lane);
  float *ratio_lut = reinterpret_cast<float *>(smem_raw + rp.ratio_off);  // n / N for n = 0..N (extras: ratio_connections)
  if (tid <= N) ratio_lut[tid] = __fdiv_rn((float)tid, (float)N);
  __syncthreads();  // the only CTA-wide barrier

  const long long e0 = ((long long)blockIdx.x * EW_WARPS + warp) * K;
  if (e0 >= p.B) return;
  const int kc = (int)((p.B - e0) < (long long)K ? (p.B - e0) : (long long)K);
  uint8_t *wg = smem_raw + p.so[0] + (size_t)warp * p.so[1];
  uint32_t *wg32 = reinterpret_cast<uint32_t *>(wg);

  const int j = lane / Np, a = lane & (Np - 1);
  const bool env_ok = j < kc, agent = env_ok && a < N;
  const long long e = e0 + (env_ok ? j : 0);
  const uint32_t gmask = Np == 32 ? FULL : (((1u << Np) - 1u) << (j * Np));

  // ---- load the State once
  load_grids<VEC>(p.in.grid, e0, kc, cells, lane, wg);
  int pos = 0, tgt = 0, start = 0, sc = 0;
  uint32_t k0 = 0, k1 = 0;
  if (agent) {
    const int2 ps = __ldg(reinterpret_cast<const int2 *>(p.in.position) + e * N + a);
    const int2 tg = __ldg(reinterpret_cast<const int2 *>(p.in.target) + e * N + a);
    const int2 st = __ldg(reinterpret_cast<const int2 *>(p.in.start) + e * N + a);
    pos = (ps.x << 8) | ps.y;
    tgt = (tg.x << 8) | tg.y;
    start = (st.x << 8) | st.y;
  }
  if (env_ok) {
    sc = p.in.step_count[e];
    k0 = p.in.key[2 * e];
    k1 = p.in.key[2 * e + 1];
  }
  __syncwarp();
  uint8_t *g = wg + (size_t)j * cells;
  const SmemGrid sg{g, G, 0, G};
  int paths = count_paths<VEC>(wg, j, a, cells, c4, Np, env_ok);  // carried across steps
  // the action mask of the state an env is in: what step t emits is what step t+1's policy samples from
  uint32_t mk3 = 0;
  if (agent) mk3 = move_mask(sg, pos >> 8, pos & 255, a, pos == tgt);

  // observation: staged in shared memory, written by bulk copies (obs_stage.cuh)
  ObsStager os;
  int4 *obs_t = nullptr;
  long long obs_step = 0;
  if (VEC) {
    os.init(smem_raw + rp.stage_off + (size_t)warp * rp.stage_warp, lut, wg32, N, c4, p.divC4, lane, rp.stage_bytes, rp.stage_nbuf, rp.ce, rp.cv);
    obs_t = reinterpret_cast<int4 *>(p.ts.obs_grid) + e0 * N * c4;
    obs_step = p.B * N * c4;
  }

  for (int t = 0; t < rp.T; ++t) {
    const long long tb = (long long)t * p.B;  // row offset of step t in the stacked outputs
    // ---- agents: sample action, move_position, is_valid_position, collisions
    const bool was = agent && pos == tgt;
    const int r = pos >> 8, c = pos & 255;
    const long long row_e = tb + e, row_a = row_e * N + a;  // this lane's rows in the stacked per-env / per-agent outputs
    const int dest = agent ? random_dest(k0, k1, sc, a, mk3, r, c, G, rp.action_out, row_a) : -1;
    bool win;
    pos = resolve_moves(dest, j, lane, a, r, c, G, g, p.divG, pos, win);
    uint32_t dirty = win ? cell_pair(r * G + c, dest) : OBS_CLEAN;  // the cells of g this step changed
    // ---- action mask, connected / done, reward on the new grid
    const StepResult s = after_move(sg, agent, a, pos, tgt, was, win, gmask, p.env);
    mk3 = s.mk3;
    paths += s.nmoved;
    sc += 1;
    const bool terminal = env_ok && (s.ndone == N || sc >= p.env.time_limit);
    const int tpl = paths + N;

    // ---- auto-reset: the dataset board that follows
    uint32_t nk0 = 0, nk1 = 0;
    int npos = pos, ntgt = tgt;
    if (terminal) {
      // VmapAutoResetWrapper._auto_reset: key, _ = split(state.key); then BoardDatasetGeneratorJAX.__call__
      uint32_t a0, a1, b0, b1;
      split2(k0, k1, a0, a1, b0, b1);
      const uint32_t which = dataset_pick(a0, a1, (uint32_t)p.env.dataset_K, nk0, nk1);
      if (a < N) {
        const int32_t *h = p.env.dataset_heads + (size_t)which * 2 * N, *tt = p.env.dataset_targets + (size_t)which * 2 * N;
        const int hi = G - 1;
        npos = (min(max(__ldg(h + a), 0), hi) << 8) | min(max(__ldg(h + N + a), 0), hi);
        ntgt = (min(max(__ldg(tt + a), 0), hi) << 8) | min(max(__ldg(tt + N + a), 0), hi);
      }
    }
    // ---- small outputs of step t (terminal step's reward / discount / step_type / extras)
    if (env_ok && a == 0) {
      p.ts.step_type[row_e] = (int8_t)(terminal ? 2 : 1);
      p.ts.num_connections[row_e] = s.nconn;
      p.ts.ratio_connections[row_e] = ratio_lut[s.nconn];
      p.ts.total_path_length[row_e] = tpl;
      p.ts.obs_step_count[row_e] = terminal ? 0 : sc;
    }
    if (agent) {
      p.ts.reward[row_a] = s.rew;
      p.ts.discount[row_a] = (terminal || s.done) ? 0.0f : 1.0f;
    }
    if (terminal) {  // group-uniform: swap in the new episode
      pos = npos;
      tgt = ntgt;
      start = npos;
      k0 = nk0;
      k1 = nk1;
      sc = 0;
      paths = 0;
      mk3 = place_episode(g, sg, a, N, Np, cells, G, gmask, pos, tgt, mk3, [] {});
      dirty = a < N ? cell_pair(pin_cell(pos, G), pin_cell(tgt, G)) : OBS_CLEAN;
    }
    __syncwarp();
    if (agent) store_mask5(p.ts.action_mask + row_a * 5, mk3);
    // ---- observation of step t
    if (VEC) {
      int4 *odst = obs_t;
      obs_t += obs_step;
      if (OBS == 2 && rp.delta && t > 0)
        os.emit_delta(kc, N, lane, j, __ffs(Np) - 1, (uint32_t)__cvta_generic_to_shared(g), dirty, terminal && a == 0, odst);
      else if (OBS == 2)
        os.emit(kc, N, c4, lane, odst);
      else
        os.emit_direct(lut, wg32, kc, N, c4, lane, odst);
    } else {
      write_obs_scalar(p.ts.obs_grid + (tb + e0) * N * cells, wg, lut, RS, kc, cells, N, Np, 0u, p.divCells, lane);
    }
    __syncwarp();  // the next step's writes must not overtake these reads
  }

  if (OBS == 2) os.drain(lane);
  write_state_once<VEC>(p.out, wg, e0, kc, cells, lane, e, N, a, env_ok, agent, pos, tgt, start, sc, k0, k1);
}

// ---------------------------------------------------------------------------
// rollout_persist_kernel: the fused rollout as a PERSISTENT kernel with generator warps.
//
// Same step logic and lane layout as rollout_warp_kernel.  What changes is who does what, when:
//  * the grid is sized to the machine (resident CTAs x SM count); an env warp pulls groups of K envs from a
//    global counter until none are left, so there are no CTA waves and the DRAM write rate does not dip at
//    wave boundaries;
//  * every CTA carries GEN_WARPS generator warps (gen_warp.cuh).  When an env finishes, its warp swaps in the
//    env's cached next episode and posts a request for the episode AFTER that one; a generator warp of the
//    same CTA produces it (ParallelRandomWalk walk / Uniform selection, W lanes per board) into the env's
//    cache entry while the env warps keep streaming observations.  Generation is integer-issue bound, the
//    rollout HBM-write bound with half of the issue slots idle: inside one CTA the two share an SM, which a
//    separate refill kernel could not (the rollout CTAs' shared memory fills the SM);
//  * an env that needs an episode which is not there yet (a second termination within a few steps of the
//    first) waits for its generator warp; nothing is generated by env warps, no refill kernel, no lists;
//  * launch overlap: a persistent grid ends raggedly (env warps finish within one group time of each other,
//    the generator warps drain their rings after that: together 12-16 % of a 20-step launch with nothing
//    to do).  Consecutive rollout launches on a stream are therefore chained by programmatic dependent
//    launch: the next launch's CTAs take the SM slots as this launch's CTAs leave.  What orders the two
//    launches is per GROUP, not per grid: group g of launch e+1 is loaded only when launch e has written
//    group g's State (group_done[g] >= e) AND every episode it requested for those envs has been published
//    (group_pending[g] == 0), both with release / acquire semantics at GPU scope.
//    The group counter of a launch is one of kPersistSets sets {next group, env warps done, owner}; a launch may
//    use set (epoch % kPersistSets) only once the launch that used it last has recycled it (owner == epoch), so
//    however many small launches are in flight at once they never share a counter.
constexpr int kPersistSets = 16;
constexpr int kPersistSetInts = 4;
constexpr int kPersistMinCtas = 4;

struct PersistParams {
  int *counter;   // [0] next env group, [1] env warps that have finished (the last one clears both), [2] epoch that may use the set next (0: any of the first kPersistSets)
  int *group_done;     // [ngroups] last launch epoch that has written the group's State
  int *group_pending;  // [ngroups] episode requests in flight
  int epoch;           // this launch (> 0, +1 per launch on the workspace)
  int ngroups;    // groups of K envs in the batch
  int env_warps;  // env warps per CTA (1..EW_WARPS)
  int gen_warps;  // generator warps per CTA (1..2)
  int tmpl_off;   // smem byte offsets: empty padded board, queues, done flag, generator scratch
  int q_off, done_off, gscr_off, gscr_stride;
  int gcand_bytes, gsel_bytes;
};

template <int OBS>
__global__ void __launch_bounds__((EW_WARPS + 2) * 32, kPersistMinCtas)
    rollout_persist_kernel(const EnvParams p, const RolloutParams rp, const PersistParams pp, const GenWarpCfg gc) {
  constexpr bool VEC = OBS != 0;
  extern __shared__ __align__(16) uint8_t smem_raw[];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int G = p.G, N = p.N, cells = p.cells;
  const int Np = p.Np, K = 32 / Np, c4 = cells >> 2;
  constexpr int RS = OBS_RS;
  uint8_t *lut = smem_raw;
  const int nthreads = blockDim.x, nwarps = nthreads >> 5;
  build_obs_lut(lut, N, RS, warp, nwarps, lane);
  float *ratio_lut = reinterpret_cast<float *>(smem_raw + rp.ratio_off);  // n / N for n = 0..N (extras: ratio_connections)
  if (tid <= N) ratio_lut[tid] = __fdiv_rn((float)tid, (float)N);
  uint8_t *tmpl = smem_raw + pp.tmpl_off;
  for (int i = tid; i < gc.SBp; i += nthreads) {
    const int r = i / gc.S, c = i - r * gc.S;
    tmpl[i] = (r >= 2 && r < G + 2 && c >= 2 && c < G + 2) ? 0 : 0xFF;
  }
  GenQueue *queues = reinterpret_cast<GenQueue *>(smem_raw + pp.q_off);
  volatile int *env_done = reinterpret_cast<volatile int *>(smem_raw + pp.done_off);
  if (warp < pp.gen_warps) genq_init(queues + warp, lane);
  if (tid == 0) *env_done = 0;
  // the next launch on the stream may start as soon as SM slots free up (it orders itself per group, see above)
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  __syncthreads();  // the only CTA-wide barrier

  if (warp >= pp.env_warps) {  // ---- generator warp
    const int gw = warp - pp.env_warps;
    if (gw >= pp.gen_warps) return;
    uint8_t *gb = smem_raw + pp.gscr_off + (size_t)gw * pp.gscr_stride;
    GenWarpScratch gs;
    gs.cand = reinterpret_cast<uint64_t *>(gb);
    gs.sel = reinterpret_cast<uint16_t *>(gb + pp.gcand_bytes);
    gs.board = gb + pp.gcand_bytes + pp.gsel_bytes;
    gs.tmpl = tmpl;
    gen_warp_loop(gc, gs, queues + gw, env_done, pp.env_warps, lane);
    return;
  }

  // ---- env warp
  uint8_t *wg = smem_raw + p.so[0] + (size_t)warp * p.so[1];
  uint32_t *wg32 = reinterpret_cast<uint32_t *>(wg);
  const int j = lane / Np, a = lane & (Np - 1);
  const uint32_t gmask = Np == 32 ? FULL : (((1u << Np) - 1u) << (j * Np));
  uint8_t *g = wg + (size_t)j * cells;
  const SmemGrid sg{g, G, 0, G};
  ObsStager os;
  if (VEC) os.init(smem_raw + rp.stage_off + (size_t)warp * rp.stage_warp, lut, wg32, N, c4, p.divC4, lane, rp.stage_bytes, rp.stage_nbuf, rp.ce, rp.cv);

  if (lane == 0) {  // the launch that used this counter set last (kPersistSets launches ago) must have recycled it
    for (;;) {
      const int owner = ld_acquire_s32(pp.counter + 2);
      if (owner == pp.epoch || (owner == 0 && pp.epoch <= kPersistSets)) break;
      __nanosleep(500);
    }
  }
  __syncwarp();
  for (;;) {
    int grp = 0;
    if (lane == 0) grp = atomicAdd(pp.counter, 1);
    grp = __shfl_sync(FULL, grp, 0);
    if (grp >= pp.ngroups) break;
    const long long e0 = (long long)grp * K;
    const int kc = (int)((p.B - e0) < (long long)K ? (p.B - e0) : (long long)K);
    const bool env_ok = j < kc, agent = env_ok && a < N;
    const long long e = e0 + (env_ok ? j : 0);
    GenQueue *myq = queues + (int)(e % pp.gen_warps);
    // the previous launch may still be running: its State of this group, and the episodes it asked for
    if (lane == 0) {
      while (ld_acquire_s32(pp.group_done + grp) < pp.epoch - 1 || ld_acquire_s32(pp.group_pending + grp) != 0) __nanosleep(200);
    }
    __syncwarp();

    // ---- load the State once
    load_grids<VEC>(p.in.grid, e0, kc, cells, lane, wg);
    int pos = 0, tgt = 0, start = 0, sc = 0;
    uint32_t k0 = 0, k1 = 0;
    if (agent) {
      const int2 ps = __ldg(reinterpret_cast<const int2 *>(p.in.position) + e * N + a);
      const int2 tg = __ldg(reinterpret_cast<const int2 *>(p.in.target) + e * N + a);
      const int2 st = __ldg(reinterpret_cast<const int2 *>(p.in.start) + e * N + a);
      pos = (ps.x << 8) | ps.y;
      tgt = (tg.x << 8) | tg.y;
      start = (st.x << 8) | st.y;
    }
    if (env_ok) {
      sc = p.in.step_count[e];
      k0 = p.in.key[2 * e];
      k1 = p.in.key[2 * e + 1];
      // an env whose next episode is not in the cache (first use of the workspace): ask for it right away
      if (a == 0 && ld_acquire_u64(p.cache_tag + e) != (((unsigned long long)k1 << 32) | k0)) {
        atomicAdd(pp.group_pending + grp, 1);
        genq_post(myq, (int)e, k0, k1);
      }
    }
    __syncwarp();
    int paths = count_paths<VEC>(wg, j, a, cells, c4, Np, env_ok);  // carried across steps
    uint32_t mk3 = 0;  // the action mask of the state an env is in: what step t emits is what step t+1's policy samples from
    if (agent) mk3 = move_mask(sg, pos >> 8, pos & 255, a, pos == tgt);
    int4 *obs_t = nullptr;
    long long obs_step = 0;
    if (VEC) {
      obs_t = reinterpret_cast<int4 *>(p.ts.obs_grid) + e0 * N * c4;
      obs_step = p.B * N * c4;
    }

    for (int t = 0; t < rp.T; ++t) {
      const long long tb = (long long)t * p.B;
      // ---- agents: sample action, move_position, is_valid_position, collisions
      const bool was = agent && pos == tgt;
      const int r = pos >> 8, c = pos & 255;
      const long long row_e = tb + e, row_a = row_e * N + a;
      const int dest = agent ? random_dest(k0, k1, sc, a, mk3, r, c, G, rp.action_out, row_a) : -1;
      bool win;
      pos = resolve_moves(dest, j, lane, a, r, c, G, g, p.divG, pos, win);
      uint32_t dirty = win ? cell_pair(r * G + c, dest) : OBS_CLEAN;  // the cells of g this step changed
      // ---- action mask, connected / done, reward on the new grid
      const StepResult s = after_move(sg, agent, a, pos, tgt, was, win, gmask, p.env);
      mk3 = s.mk3;
      paths += s.nmoved;
      sc += 1;
      const bool terminal = env_ok && (s.ndone == N || sc >= p.env.time_limit);
      const int tpl = paths + N;
      // ---- small outputs of step t (the terminal step keeps its reward / discount / step_type / extras)
      if (env_ok && a == 0) {
        p.ts.step_type[row_e] = (int8_t)(terminal ? 2 : 1);
        p.ts.num_connections[row_e] = s.nconn;
        p.ts.ratio_connections[row_e] = ratio_lut[s.nconn];
        p.ts.total_path_length[row_e] = tpl;
        p.ts.obs_step_count[row_e] = terminal ? 0 : sc;
      }
      if (agent) {
        p.ts.reward[row_a] = s.rew;
        p.ts.discount[row_a] = (terminal || s.done) ? 0.0f : 1.0f;
      }
      // ---- auto-reset: the env's cached next episode; its generator warp may still be working on it
      if (terminal) {  // group-uniform
        const unsigned long long want = ((unsigned long long)k1 << 32) | k0;
        if (a == 0)
          while (ld_acquire_u64(p.cache_tag + e) != want) {
            myq->urgent = 1;
            __nanosleep(100);
          }
        __syncwarp(gmask);
        if (a != 0) (void)ld_acquire_u64(p.cache_tag + e);  // every lane orders its own reads behind the published tag
        const uint2 nk = __ldcg(p.cache_key + e);
        const uint32_t pin = a < N ? __ldcg(p.cache_pins + e * N + a) : 0u;
        pos = (int)(pin >> 16);
        tgt = (int)(pin & 0xffffu);
        start = pos;
        k0 = nk.x;
        k1 = nk.y;
        sc = 0;
        paths = 0;
        mk3 = place_episode(g, sg, a, N, Np, cells, G, gmask, pos, tgt, mk3, [a, e, k0, k1, myq, pending = pp.group_pending + grp] {
          if (a == 0) {  // the episode after this one
            atomicAdd(pending, 1);
            genq_post(myq, (int)e, k0, k1);
          }
        });
        dirty = a < N ? cell_pair(pin_cell(pos, G), pin_cell(tgt, G)) : OBS_CLEAN;
      }
      __syncwarp();
      if (agent) store_mask5(p.ts.action_mask + row_a * 5, mk3);
      // ---- observation of step t
      if (VEC) {
        int4 *odst = obs_t;
        obs_t += obs_step;
        if (OBS == 2 && rp.delta && t > 0)
          os.emit_delta(kc, N, lane, j, __ffs(Np) - 1, (uint32_t)__cvta_generic_to_shared(g), dirty, terminal && a == 0, odst);
        else if (OBS == 2)
          os.emit(kc, N, c4, lane, odst);
        else
          os.emit_direct(lut, wg32, kc, N, c4, lane, odst);
      } else {
        write_obs_scalar(p.ts.obs_grid + (tb + e0) * N * cells, wg, lut, RS, kc, cells, N, Np, 0u, p.divCells, lane);
      }
      __syncwarp();  // the next step's writes must not overtake these reads
    }

    write_state_once<VEC>(p.out, wg, e0, kc, cells, lane, e, N, a, env_ok, agent, pos, tgt, start, sc, k0, k1);
    // the group's State is written (the observation copies of its last steps may still be in flight: nothing
    // of a later launch depends on them); requests posted above were counted before this store
    __threadfence();
    __syncwarp();  // the next group's load overwrites the warp's grid slice
    if (lane == 0) st_release_s32(pp.group_done + grp, pp.epoch);
  }
  if (OBS == 2) os.drain(lane);  // shared memory must outlive the bulk copies
  // this env warp is done: tell the CTA's generator warps, and the grid (the last warp recycles the counters)
  __syncwarp();
  if (lane == 0) {
    __threadfence_block();
    atomicAdd(const_cast<int *>(env_done), 1);
    __threadfence();
    if (atomicAdd(pp.counter + 1, 1) == (int)gridDim.x * pp.env_warps - 1) {
      pp.counter[0] = 0;
      pp.counter[1] = 0;
      __threadfence();
      st_release_s32(pp.counter + 2, pp.epoch + kPersistSets);
    }
  }
}

// standalone random policy: one thread per (env, agent), grid read from global
__global__ void __launch_bounds__(256) random_actions_kernel(rbg_state st, long long B, int G, int N,
                                                             FastDiv divN, int32_t *action) {
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= B * N) return;
  const long long e = t / N;
  const int a = (int)(t - e * N);
  const int2 ps = reinterpret_cast<const int2 *>(st.position)[t];
  const int2 tg = reinterpret_cast<const int2 *>(st.target)[t];
  const bool connected = ps.x == tg.x && ps.y == tg.y;
  const int32_t *g = st.grid + e * G * G;
  const uint32_t tgt = 3u * a + TARGET;
  auto ok = [&](int r, int c) {
    if ((unsigned)r >= (unsigned)G || (unsigned)c >= (unsigned)G) return 0u;
    const uint32_t v = (uint32_t)__ldg(g + r * G + c);
    return (v == 0u || v == tgt) ? 1u : 0u;
  };
  uint32_t mk = ok(ps.x - 1, ps.y) | (ok(ps.x, ps.y + 1) << 1) | (ok(ps.x + 1, ps.y) << 2) | (ok(ps.x, ps.y - 1) << 3);
  if (connected) mk = 0;
  action[t] = random_action(st.key[2 * e], st.key[2 * e + 1], (uint32_t)st.step_count[e], (uint32_t)a, mk);
}

static size_t up16(size_t x) { return (x + 15) & ~(size_t)15; }

// What every launcher of the warp-per-K-envs kernels derives from G and N: Np lanes per env (the next power of two
// >= N), K = 32 / Np envs per warp, the bytes of one warp's grid slice and the kernels' divisors.
struct WarpShape {
  int cells, Np, K;
  size_t wgrid;
  FastDiv divG, divC4, divCells;
  bool vec() const { return (cells & 3) == 0; }
};

static WarpShape warp_shape(int G, int N) {
  WarpShape s;
  s.cells = G * G;
  s.Np = 1;
  while (s.Np < N) s.Np <<= 1;
  s.K = 32 / s.Np;
  s.wgrid = up16((size_t)s.K * s.cells);
  s.divG = FastDiv::make((uint32_t)G);
  s.divC4 = FastDiv::make((uint32_t)(s.vec() ? s.cells >> 2 : 1));
  s.divCells = FastDiv::make((uint32_t)s.cells);
  return s;
}

// bytes of an observation table of N rows RS bytes apart, with 256 bytes to spare
static size_t lut_bytes(int N, int RS) { return up16((size_t)N * RS + 256); }

// EnvParams / EvalStepParams: the shape fields and the shared-memory offsets {table, grid slice}
template <class P>
static void set_warp_shape(P &p, const WarpShape &s, size_t lutB) {
  p.cells = s.cells;
  p.Np = s.Np;
  p.divG = s.divG;
  p.divC4 = s.divC4;
  p.divCells = s.divCells;
  p.so[0] = (int)lutB;
  p.so[1] = (int)s.wgrid;
}

int launch_env(EnvParams p, cudaStream_t stream, bool pdl) {
  if (p.B <= 0) return RBG_OK;
  const WarpShape s = warp_shape(p.G, p.N);
  const size_t lutB = lut_bytes(p.N, obs_lut_stride(p.N));
  set_warp_shape(p, s, lutB);
  const size_t smem = lutB + EW_WARPS * s.wgrid;
  const int64_t E = EW_WARPS * s.K;  // envs per CTA
  const int64_t ctas = (p.B + E - 1) / E;
  void (*fn)(const EnvParams) = s.vec() ? env_warp_kernel<true> : env_warp_kernel<false>;
  return launch_kernel(fn, (unsigned)ctas, EW_WARPS * 32, smem, stream, RBG_K_ENV, "env_warp_kernel", pdl, p);
}

// Wave balance: a launch of `ctas` CTAs runs in ceil(ctas / (148 * c)) rounds when c CTAs fit on an
// SM; pick the residency c in [cmin, cmax] with the smallest rounds * c and enforce it by padding
// the dynamic shared memory (4096 CTAs: 8 per SM = 3.46 -> 4 rounds of 8; 7 per SM = 3.95 -> 4
// rounds of 7, measured 3 % faster).
static size_t balance_waves(int64_t ctas, int cmax, int cmin, size_t smem_needed) {
  int best = cmax;
  int64_t best_cost = -1;
  for (int c = cmax; c >= cmin; --c) {
    const int64_t rounds = (ctas + (int64_t)device_sm_count() * c - 1) / ((int64_t)device_sm_count() * c);
    const int64_t cost = rounds * c;
    if (best_cost < 0 || cost < best_cost) {
      best_cost = cost;
      best = c;
    }
  }
  if (best == cmax) return smem_needed;
  // per-SM shared memory 228 KB, 1 KB reserved per CTA: c CTAs fit, c + 1 do not
  const size_t pad = device_smem_per_sm() / (size_t)(best + 1) + 1024;
  return pad > smem_needed ? pad : smem_needed;
}

// The shared-memory layout of the fused rollout kernels, a function of the shape and the auto-reset generator kind
// alone: rollout_warp_kernel for RBG_GEN_DATASET (resets are a table lookup), rollout_persist_kernel with its generator
// warps for RBG_GEN_PRW / RBG_GEN_UNIFORM.  `smem` is the CTA's need before launch_rollout's wave-balance padding.
struct RolloutLayout {
  WarpShape s;
  size_t lutB, smem;
  bool isolated;     // rollout_persist_kernel: 3 env warps and 1 generator warp per CTA
  int PW;            // env warps per CTA
  RolloutParams rp;  // offsets and the observation staging plan
  PersistParams pp;  // rollout_persist_kernel: offsets and warp counts
  GenWarpCfg gc;     // rollout_persist_kernel: the generator warps
};

static RolloutLayout rollout_layout(int kind, int G, int N) {
  RolloutLayout L;
  memset(&L, 0, sizeof(L));
  L.s = warp_shape(G, N);
  const WarpShape &s = L.s;
  const bool persist = kind != RBG_GEN_DATASET;
  L.lutB = lut_bytes(N, OBS_RS);
  RolloutParams &rp = L.rp;
  PersistParams &pp = L.pp;
  // CTA shape of the persistent kernel.  "Isolated": 3 env warps + 1 generator warp = 4 warps per CTA, one per SM
  // sub-partition, so the generator warps of all resident CTAs share ONE sub-partition and never compete with env warps
  // for issue slots, at most 4 CTAs per SM.  "Packed": 4 env + 2 generator warps, as many CTAs as fit.  Measured (65 536
  // envs, M env-steps/s, isolated / packed): 10x10/5 2501 / 2338, 12x12/6 1649 / 1508, 10x10/4 2884 / 2850, 10x10/8 1598 /
  // 1596; 8x8/4 2817 / 3432, 8x8/8 1477 / 1687, 6x6/3 2623 / 2989 (issue-bound: more env warps win); 14x14/7 1013 / 1034,
  // 16x16/8 761 / 774, 20x20/10 372 / 378, 32x32/16 94.9 / 96.8 (resets are rare per byte: packed is 2 % ahead).
  const bool isolated = persist && G >= 9 && G <= 13 && N <= 8;
  L.isolated = isolated;
  L.PW = isolated ? 3 : EW_WARPS;
  size_t off = L.lutB + L.PW * s.wgrid;
  rp.ratio_off = (int)off;
  off = up16(off + 4 * (RBG_MAX_N + 4));
  if (persist) {
    GenWarpCfg &gc = L.gc;
    gc = gen_warp_cfg(kind, G, N, &pp.gcand_bytes, &pp.gsel_bytes, &pp.gscr_stride);
    gc.patience = 20;
    gc.seqlock = 0;  // nobody reads an entry while it is rewritten here (see gen_warp_batch)
    gc.kshift = 0;
    while ((1 << gc.kshift) < s.K) ++gc.kshift;
    pp.gen_warps = isolated ? 1 : 2;
    pp.env_warps = L.PW;
    pp.tmpl_off = (int)off;
    off = up16(off + gc.SBp);
    pp.q_off = (int)off;
    off = up16(off + pp.gen_warps * sizeof(GenQueue));
    pp.done_off = (int)off;
    off += 16;
    pp.gscr_off = (int)off;
    off += (size_t)pp.gen_warps * pp.gscr_stride;
  }
  rp.stage_off = (int)off;
  rp.stage_nbuf = 1;
  rp.ce = 1;
  rp.cv = N;
  if (s.vec()) {
    const ObsStagePlan pl = obs_stage_plan(s.K, N, s.cells, 4096, 8192);
    rp.stage_bytes = pl.bytes;
    rp.stage_nbuf = pl.nbuf;
    rp.ce = pl.ce;
    rp.cv = pl.cv;
    rp.delta = pl.nbuf == 1 && pl.ce == s.K;
    rp.stage_warp = (int)up16((size_t)rp.stage_nbuf * rp.stage_bytes);
    off += (size_t)L.PW * rp.stage_warp;
  }
  L.smem = up16(off);
  return L;
}

size_t rollout_smem(int kind, int G, int N) { return rollout_layout(kind, G, N).smem; }

int launch_rollout(EnvParams p, int T, int32_t *action_out, cudaStream_t stream) {
  if (p.B <= 0 || T <= 0) return RBG_OK;
  const RolloutLayout L = rollout_layout(RBG_GEN_DATASET, p.G, p.N);
  const WarpShape &s = L.s;
  const int K = s.K;
  const bool vec = s.vec();
  set_warp_shape(p, s, L.lutB);
  RolloutParams rp = L.rp;
  rp.T = T;
  rp.action_out = action_out;
  size_t smem = L.smem;
  if (smem > kRolloutMaxSmem) return set_error(RBG_EINVAL, "rollout: shared memory %zu too large", smem);
  const int64_t E = EW_WARPS * K;  // envs per CTA
  const int64_t ctas = (p.B + E - 1) / E;
  {  // residency: registers allow kRolloutMinCtas per SM, shared memory (1 KB reserved per CTA) maybe fewer
    int cmax = (int)(device_smem_per_sm() / (smem + 1024));
    if (cmax > kRolloutMinCtas) cmax = kRolloutMinCtas;
    if (cmax >= 3) smem = balance_waves(ctas, cmax, cmax - 2, smem);
  }
  const bool staged = vec && rp.stage_nbuf != 0;
  void (*fn)(const EnvParams, const RolloutParams) = staged ? rollout_warp_kernel<2> : (vec ? rollout_warp_kernel<1> : rollout_warp_kernel<0>);
  return launch_kernel(fn, (unsigned)ctas, EW_WARPS * 32, smem, stream, RBG_K_ROLLOUT, "rollout_warp_kernel", false, p, rp);
}

// The persistent rollout with in-CTA generator warps (rollout_persist_kernel).  `cache_*` of `p` must be set;
// `counter` points at two zeroed ints that the kernel recycles by itself.
int launch_rollout_persist(EnvParams p, int kind, int T, int32_t *action_out, int32_t *counter, int32_t *group_done, int32_t *group_pending,
                           int epoch, bool overlap, uint64_t *cache_tag_w, uint2 *cache_key_w, uint32_t *cache_pins_w, cudaStream_t stream) {
  if (p.B <= 0 || T <= 0) return RBG_OK;
  const RolloutLayout L = rollout_layout(kind, p.G, p.N);
  const WarpShape &s = L.s;
  const int K = s.K, PW = L.PW;
  const bool vec = s.vec(), isolated = L.isolated;
  set_warp_shape(p, s, L.lutB);
  RolloutParams rp = L.rp;
  rp.T = T;
  rp.action_out = action_out;
  PersistParams pp = L.pp;
  pp.counter = counter + (epoch % kPersistSets) * kPersistSetInts;
  pp.group_done = group_done;
  pp.group_pending = group_pending;
  pp.epoch = epoch;
  pp.ngroups = (int)((p.B + K - 1) / K);
  GenWarpCfg gc = L.gc;
  gc.cache_tag = reinterpret_cast<unsigned long long *>(cache_tag_w);
  gc.cache_key = cache_key_w;
  gc.cache_pins = cache_pins_w;
  gc.group_pending = group_pending;
  const size_t smem = L.smem;
  if (smem > kRolloutMaxSmem) return set_error(RBG_EINVAL, "rollout: shared memory %zu too large", smem);
  const bool staged = vec && rp.stage_nbuf != 0;
  const int threads = (PW + pp.gen_warps) * 32;
  void (*fn)(const EnvParams, const RolloutParams, const PersistParams, const GenWarpCfg) =
      staged ? rollout_persist_kernel<2> : (vec ? rollout_persist_kernel<1> : rollout_persist_kernel<0>);
  if (int rc = opt_in_smem(fn, smem, "rollout_persist_kernel")) return rc;
  cudaError_t ce;
  int resident = 0;
  if ((ce = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&resident, fn, threads, smem)) != cudaSuccess) return set_cuda_error(ce, "cudaOccupancyMaxActiveBlocksPerMultiprocessor");
  if (resident < 1) return set_error(RBG_EINVAL, "rollout_persist_kernel does not fit an SM (%zu bytes of shared memory)", smem);
  if (isolated && resident > 4) resident = 4;  // more resident CTAs measure slower (10x10/5 on B200: 5 -0.4 %, 6 -0.8 %)
  int64_t ctas = (int64_t)resident * device_sm_count();
  const int64_t need = (pp.ngroups + PW - 1) / PW;
  if (ctas > need) ctas = need;
  // overlap: this grid may begin under the tail of the previous rollout_persist_kernel of the stream
  return launch_kernel(fn, (unsigned)ctas, threads, smem, stream, RBG_K_ROLLOUT, "rollout_persist_kernel", overlap, p, rp, pp, gc);
}

int launch_random_actions(const rbg_state &st, int64_t B, int G, int N, int32_t *action, cudaStream_t stream) {
  const int64_t n = B * N;
  if (n <= 0) return RBG_OK;
  return launch_kernel(random_actions_kernel, (unsigned)((n + 255) / 256), 256, 0, stream, RBG_K_RANDACT, "random_actions_kernel", false, st, B, G, N,
                       FastDiv::make((uint32_t)N), action);
}

// ---------------------------------------------------------------------------
// episode_warp_kernel: every env of a batch from its State to its FIRST LAST step under the random policy, one
// metrics record per env (the random-agent evaluation of a board generator).  Lane layout and step body are those
// of rollout_warp_kernel: a warp owns K = 32 / Np envs, a lane is one (env, agent), the grids are uint8 in the
// warp's slice of shared memory.  Nothing is written per step: returns accumulate in registers and an env writes
// ~40 bytes when its episode ends.  A group of Np lanes whose episode has ended takes the next env of the batch from
// a global counter (episodes of one warp differ in length: without the refill a warp would run for as long as its
// longest episode).  A group with no env left idles through the warp-wide match / ballots; the warp exits when every
// group is idle.  The grid is persistent (resident CTAs x SMs).  The input State is never written.
constexpr int EP_WARPS = 4;
constexpr int kEpisodeMinCtas = 8;

struct EpisodeParams {
  rbg_state in;               // read only
  rbg_state fin;              // State after each env's terminal step; fin.grid == NULL: not written
  rbg_episode_metrics out;
  long long B;
  int G, N, cells, Np;
  int time_limit;
  float timestep_reward, connected_reward;
  int ratio_off;  // smem byte offset of the n / N table
  int wgrid;      // smem bytes of one warp's grid slice
  int *counter;   // next env index, zeroed
  FastDiv divG;
};

__global__ void __launch_bounds__(EP_WARPS * 32, kEpisodeMinCtas) episode_warp_kernel(const EpisodeParams p) {
  extern __shared__ __align__(16) uint8_t smem_raw[];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int G = p.G, N = p.N, cells = p.cells, Np = p.Np;
  float *ratio_lut = reinterpret_cast<float *>(smem_raw + p.ratio_off);  // n / N for n = 0..N (extras: ratio_connections)
  if (tid <= N) ratio_lut[tid] = __fdiv_rn((float)tid, (float)N);
  __syncthreads();  // the only CTA-wide barrier

  const int j = lane / Np, a = lane & (Np - 1), lead = j * Np;
  const uint32_t gmask = Np == 32 ? FULL : (((1u << Np) - 1u) << lead);
  uint8_t *g = smem_raw + (size_t)warp * p.wgrid + (size_t)j * cells;
  const SmemGrid sg{g, G, 0, G};

  long long e = 0;
  bool env_ok = false, agent = false, refill = true;
  int pos = 0, tgt = 0, sc = 0, len = 0, paths = 0;
  uint32_t k0 = 0, k1 = 0, mk3 = 0;
  float ret = 0.0f;
  for (;;) {
    if (refill) {  // group-uniform: the next env of the batch, State int32 -> uint8 grid, PATH cells recounted
      long long nx = 0;
      if (a == 0) nx = atomicAdd(p.counter, 1);
      nx = __shfl_sync(gmask, nx, lead);
      env_ok = nx < p.B;
      agent = env_ok && a < N;
      refill = false;
      if (env_ok) {
        e = nx;
        const int32_t *src = p.in.grid + e * cells;
        int pc = 0;
        for (int i = a; i < cells; i += Np) {
          const uint32_t v = (uint8_t)__ldg(src + i);
          g[i] = (uint8_t)v;
          pc += (v % 3u == 1u) ? 1 : 0;
        }
        for (int off = Np >> 1; off; off >>= 1) pc += __shfl_xor_sync(gmask, pc, off);
        paths = pc;
        sc = __ldg(p.in.step_count + e);
        k0 = __ldg(p.in.key + 2 * e);
        k1 = __ldg(p.in.key + 2 * e + 1);
        len = 0;
        ret = 0.0f;
        if (agent) {
          const int2 ps = __ldg(reinterpret_cast<const int2 *>(p.in.position) + e * N + a);
          const int2 tg = __ldg(reinterpret_cast<const int2 *>(p.in.target) + e * N + a);
          pos = (ps.x << 8) | ps.y;
          tgt = (tg.x << 8) | tg.y;
        }
        __syncwarp(gmask);  // the whole grid is in before anybody reads a neighbour
        mk3 = agent ? move_mask(sg, pos >> 8, pos & 255, a, pos == tgt) : 0u;
      }
    }
    if (__ballot_sync(FULL, env_ok) == 0u) break;

    // ---- one step: sample action, move, collisions
    const bool was = agent && pos == tgt;
    const int r = pos >> 8, c = pos & 255;
    const int dest = agent ? random_dest(k0, k1, sc, a, mk3, r, c, G, nullptr, 0) : -1;
    bool win;
    pos = resolve_moves(dest, j, lane, a, r, c, G, g, p.divG, pos, win);
    // ---- action mask, connected / done, reward on the new grid
    const StepResult s = after_move(sg, agent, a, pos, tgt, was, win, gmask, p);
    mk3 = s.mk3;
    paths += s.nmoved;
    sc += 1;
    len += 1;
    ret = __fadd_rn(ret, s.rew);
    const bool terminal = env_ok && (s.ndone == N || sc >= p.time_limit);

    // ---- the episode's record (group-uniform)
    if (terminal) {
      if (agent) p.out.episode_return[e * N + a] = ret;
      if (a == 0) {
        p.out.episode_length[e] = len;
        p.out.num_connections[e] = s.nconn;
        p.out.ratio_connections[e] = ratio_lut[s.nconn];
        p.out.total_path_length[e] = paths + N;
      }
      if (p.fin.grid) {  // Connector.step's State: grid, position and step_count move, the rest is the input's
        int32_t *dst = p.fin.grid + e * cells;
        for (int i = a; i < cells; i += Np) dst[i] = g[i];
        if (a == 0) {
          p.fin.step_count[e] = sc;
          p.fin.key[2 * e] = k0;
          p.fin.key[2 * e + 1] = k1;
        }
        if (agent) {
          const long long ga = e * N + a;
          reinterpret_cast<int2 *>(p.fin.position)[ga] = make_int2(pos >> 8, pos & 255);
          reinterpret_cast<int2 *>(p.fin.target)[ga] = make_int2(tgt >> 8, tgt & 255);
          reinterpret_cast<int2 *>(p.fin.start)[ga] = __ldg(reinterpret_cast<const int2 *>(p.in.start) + ga);
          p.fin.agent_id[ga] = __ldg(p.in.agent_id + ga);
        }
      }
      refill = true;
    }
    __syncwarp();  // the next episode's grid load must not overtake this step's reads
  }
}

int launch_episodes(const rbg_state &in, const rbg_state *fin, const rbg_episode_metrics &out, int64_t B, int G, int N,
                    const rbg_env_params &env, cudaStream_t stream) {
  if (B <= 0) return RBG_OK;
  EpisodeParams p;
  memset(&p, 0, sizeof(p));
  p.in = in;
  if (fin) p.fin = *fin;
  p.out = out;
  p.B = B;
  p.G = G;
  p.N = N;
  const WarpShape s = warp_shape(G, N);
  const int K = s.K;
  p.cells = s.cells;
  p.Np = s.Np;
  p.time_limit = env.time_limit;
  p.timestep_reward = env.timestep_reward;
  p.connected_reward = env.connected_reward;
  p.divG = s.divG;
  p.wgrid = (int)s.wgrid;
  p.ratio_off = EP_WARPS * p.wgrid;
  const size_t smem = (size_t)p.ratio_off + 4 * (RBG_MAX_N + 4);
  // few agents on a big board: up to 4 warps x 32 envs x 1 600 cells = 200 KB (40x40/1), past the 48 KB default
  if (int rc = opt_in_smem(episode_warp_kernel, smem, "episode_warp_kernel")) return rc;
  cudaError_t ce;
  int per_sm = 0;
  if ((ce = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, episode_warp_kernel, EP_WARPS * 32, smem)) != cudaSuccess)
    return set_cuda_error(ce, "cudaOccupancyMaxActiveBlocksPerMultiprocessor(episode_warp_kernel)");
  if (per_sm < 1) return set_error(RBG_EINVAL, "episode_warp_kernel does not fit an SM (%zu bytes of shared memory)", smem);
  const int64_t resident = (int64_t)per_sm * device_sm_count();
  const int64_t need = (B + (int64_t)EP_WARPS * K - 1) / ((int64_t)EP_WARPS * K);
  const unsigned ctas = (unsigned)(need < resident ? need : resident);
  // the env counter: stream-ordered scratch, so that the caller needs no workspace and launches on different
  // streams never share it
  keep_pool_cached();
  void *scratch = nullptr;
  if ((ce = cudaMallocAsync(&scratch, 256, stream)) != cudaSuccess) return set_cuda_error(ce, "cudaMallocAsync(episode counter)");
  p.counter = static_cast<int *>(scratch);
  int rc = RBG_OK;
  if ((ce = cudaMemsetAsync(scratch, 0, 256, stream)) != cudaSuccess)
    rc = set_cuda_error(ce, "cudaMemsetAsync(episode counter)");
  else
    rc = launch_kernel(episode_warp_kernel, ctas, EP_WARPS * 32, smem, stream, RBG_K_EPISODES, "episode_warp_kernel", false, p);
  cudaFreeAsync(scratch, stream);
  return rc;
}

// ---------------------------------------------------------------------------
// eval_step_kernel: one plain Connector.step (actions given, no auto-reset) of the envs whose live byte is set, with
// each env's episode record accumulated in place: the step of a policy evaluation, one launch per policy call.  Lane
// layout, observation table and in-place grid scatter are env_warp_kernel's (a warp owns K = 32 / Np envs, a lane is
// one (env, agent)).  An env whose live byte is 0 costs the read of that byte: its State, TimeStep row, record and
// action are neither read nor written, so the step's traffic scales with the live envs, and a warp with no live env
// exits after that read.  On LAST the extras go to the record, the live byte is cleared and live_count drops by the
// warp's number of finished envs (one atomic per warp).
//
// LIST (rbg_connector_eval_step_live): the same step of the envs order_in[0, L), all of them live, with action row i
// belonging to env order_in[i].  The step also compacts the list: an env that did not reach LAST gets output row r =
// the number of such envs before it in order_in, order_out[r] = env, and its observation (grid, action mask, step
// count) goes to row r of ts; *count_out = the number of them.  Nothing else of the TimeStep is written.  A CTA is
// a tile of EW_WARPS * K consecutive list entries; r comes from a warp ballot, a scan of the CTA's warp counts and a
// single-pass decoupled look-back over the tiles before it (tile_status), with tiles numbered by a ticket counter
// so that a CTA waits only on CTAs that are already running.  The grids stay in shared memory until r is known.
struct EvalStepParams {
  rbg_state st;  // stepped in place
  rbg_timestep ts;
  rbg_episode_metrics acc;
  const int32_t *action;
  uint8_t *live;
  int32_t *live_count;
  long long B;
  int G, N, cells, Np;
  int time_limit;
  float timestep_reward, connected_reward;
  int so[2];  // shared memory: [0] bytes of the observation table, [1] bytes of one warp's grid slice
  FastDiv divG, divC4, divCells;
  // LIST only
  const int32_t *order_in;
  int32_t *order_out, *count_out;
  unsigned long long *tile_status;  // [tiles]: flag << 32 | count, zeroed; flag 1: the tile's own count, 2: inclusive prefix
  int *ticket;                      // zeroed
  long long L, tiles;
  int so_list;  // smem byte offset of the LIST scratch (LS_*)
};

// LIST scratch in shared memory, in ints: per warp 32 slots (env index of slot j, then its output row or -1), the
// warp counts of survivors, their exclusive prefixes over the list, the tile
enum : int { LS_SLOTS = 0, LS_WCOUNT = EW_WARPS * 32, LS_WBASE = LS_WCOUNT + EW_WARPS, LS_TILE = LS_WBASE + EW_WARPS, LS_INTS = LS_TILE + 1 };

// decoupled look-back, warp-wide: publish this tile's count, wait for the tiles before it in windows of 32 until one
// with an inclusive prefix is found, publish the inclusive prefix; returns the exclusive prefix (every lane)
__device__ __forceinline__ int tile_prefix(unsigned long long *status, long long tile, int agg, int lane) {
  using ref = cuda::atomic_ref<unsigned long long, cuda::thread_scope_device>;
  if (tile == 0) {
    if (lane == 0) ref(status[0]).store((2ull << 32) | (uint32_t)agg, cuda::memory_order_relaxed);
    return 0;
  }
  if (lane == 0) ref(status[tile]).store((1ull << 32) | (uint32_t)agg, cuda::memory_order_relaxed);
  int excl = 0;
  for (long long top = tile - 1;; top -= 32) {
    const long long t = top - lane;
    unsigned long long w = 2ull << 32;  // before tile 0: an inclusive prefix of 0
    if (t >= 0) {
      ref s(status[t]);
      do w = s.load(cuda::memory_order_relaxed);
      while ((w >> 32) == 0);
    }
    const uint32_t incl = __ballot_sync(FULL, (w >> 32) == 2);
    const int stop = incl ? __ffs((int)incl) - 1 : 31;  // the nearest tile with an inclusive prefix
    int v = lane <= stop ? (int)(uint32_t)w : 0;
    for (int off = 16; off; off >>= 1) v += __shfl_xor_sync(FULL, v, off);
    excl += v;
    if (incl) break;
  }
  if (lane == 0) ref(status[tile]).store((2ull << 32) | (uint32_t)(excl + agg), cuda::memory_order_relaxed);
  return excl;
}

template <bool VEC, bool LIST>
__global__ void __launch_bounds__(EW_WARPS * 32, kEnvMinCtas) eval_step_kernel(const EvalStepParams p) {
  extern __shared__ __align__(16) uint8_t smem_raw[];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int G = p.G, N = p.N, cells = p.cells;
  const int Np = p.Np, K = 32 / Np, c4 = cells >> 2;
  const int RS = obs_lut_stride(N);
  int *ls = reinterpret_cast<int *>(smem_raw + p.so_list);  // LIST scratch
  int *slots = ls + LS_SLOTS + warp * 32;

  long long tile = blockIdx.x;
  if (LIST) {
    if (tid == 0) ls[LS_TILE] = atomicAdd(p.ticket, 1);
    __syncthreads();
    tile = ls[LS_TILE];
  }
  // e0: the warp's first env (LIST: its first list entry)
  const long long e0 = (tile * EW_WARPS + warp) * K, n = LIST ? p.L : p.B;
  const int kc = e0 >= n ? 0 : (int)((n - e0) < (long long)K ? (n - e0) : (long long)K);
  const int j = lane / Np, a = lane & (Np - 1);
  const long long e = LIST ? (j < kc ? (long long)__ldg(p.order_in + e0 + j) : 0) : e0 + (j < kc ? j : 0);
  const bool env_ok = j < kc && (LIST || p.live[e] != 0), agent = env_ok && a < N;
  const uint32_t livem = __ballot_sync(FULL, env_ok);  // bit j * Np (and the env's other lanes): env j is live
  if (!LIST && !__syncthreads_or(livem != 0u)) return;  // a CTA without a live env builds no table
  uint8_t *lut = smem_raw;
  build_obs_lut(lut, N, RS, warp, EW_WARPS, lane);
  if (LIST && env_ok && a == 0) slots[j] = (int)e;
  __syncthreads();  // LIST: the last CTA-wide barrier but the two of the row scan
  if (!LIST && livem == 0u) return;
  uint8_t *wg = smem_raw + p.so[0] + (size_t)warp * p.so[1];
  uint32_t *wg32 = reinterpret_cast<uint32_t *>(wg);
  const uint32_t gmask = Np == 32 ? FULL : (((1u << Np) - 1u) << (j * Np));

  // ---- load the live envs: State.grid int32 -> uint8, agent and env scalars (LIST: env m of the warp is slots[m])
  if (VEC) {
    const int4 *src = reinterpret_cast<const int4 *>(p.st.grid) + e0 * c4;
    const int nq = kc * c4;
    for (int q0 = lane; q0 < nq; q0 += 128) {
      int4 v[4];
      bool ok[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int q = q0 + 32 * u;
        ok[u] = q < nq && ((livem >> ((int)p.divC4.div((uint32_t)q) * Np)) & 1u);
        if (!ok[u]) {
          v[u] = make_int4(0, 0, 0, 0);
        } else if (LIST) {
          const int m = (int)p.divC4.div((uint32_t)q);
          v[u] = __ldg(reinterpret_cast<const int4 *>(p.st.grid) + (size_t)slots[m] * c4 + (q - m * c4));
        } else {
          v[u] = __ldg(src + q);
        }
      }
#pragma unroll
      for (int u = 0; u < 4; ++u)
        if (ok[u])
          wg32[q0 + 32 * u] = (uint32_t)(v[u].x & 0xff) | ((uint32_t)(v[u].y & 0xff) << 8) | ((uint32_t)(v[u].z & 0xff) << 16) | ((uint32_t)(v[u].w & 0xff) << 24);
    }
  } else {
    const int32_t *src = p.st.grid + e0 * cells;
    for (int i = lane; i < kc * cells; i += 32) {
      const int m = (int)p.divCells.div((uint32_t)i);
      if ((livem >> (m * Np)) & 1u) wg[i] = (uint8_t)__ldg(LIST ? p.st.grid + (size_t)slots[m] * cells + (i - m * cells) : src + i);
    }
  }
  int pos = 0, tgt = 0, action = 0, sc0 = 0;
  if (agent) {
    const int2 ps = __ldg(reinterpret_cast<const int2 *>(p.st.position) + e * N + a);
    const int2 tg = __ldg(reinterpret_cast<const int2 *>(p.st.target) + e * N + a);
    pos = (ps.x << 8) | ps.y;
    tgt = (tg.x << 8) | tg.y;
    action = __ldg(p.action + (LIST ? e0 + j : e) * N + a);
  }
  if (env_ok) sc0 = p.st.step_count[e];
  __syncwarp();

  uint8_t *g = wg + (size_t)j * cells;
  const SmemGrid sg{g, G, 0, G};
  // PATH cells of the env before the move (extras: total_path_length)
  const int paths = count_paths<VEC>(wg, j, a, cells, c4, Np, env_ok);

  // ---- agents: move_position, is_valid_position, collisions; State.grid in place
  const bool was = agent && pos == tgt;
  const int r = pos >> 8, c = pos & 255;
  int dest = -1;
  if (agent) {
    const int am = action < 0 ? 0 : (action > 4 ? 4 : action);  // lax.switch clamps
    const int nr = r + (am == UP ? -1 : (am == DOWN ? 1 : 0));
    const int nc = c + (am == RIGHT ? 1 : (am == LEFT ? -1 : 0));
    const bool inb = (unsigned)nr < (unsigned)G && (unsigned)nc < (unsigned)G;
    const uint32_t v = inb ? sg.at(nr, nc) : 0xFFu;
    if (inb && (v == 0u || v == 3u * a + TARGET) && !was && action != NOOP) dest = nr * G + nc;
  }
  // same destination in the same env -> only the highest agent id moves
  const uint32_t mval = dest >= 0 ? (((uint32_t)j << 16) | (uint32_t)dest) : (0x80000000u | (uint32_t)lane);
  const uint32_t mm = __match_any_sync(FULL, mval);
  const bool win = dest >= 0 && lane == 31 - __clz(mm);
  __syncwarp();  // every read of the pre-move grid is done
  if (win) {  // move_agent: old head -> PATH, new cell -> POSITION; State.grid in place: only these two cells change
    g[r * G + c] = (uint8_t)(3 * a + PATH);
    g[dest] = (uint8_t)(3 * a + POSITION);
    int32_t *gg = p.st.grid + e * cells;
    gg[r * G + c] = 3 * a + PATH;
    gg[dest] = 3 * a + POSITION;
    uint32_t nr, nc;
    p.divG.divmod((uint32_t)dest, nr, nc);
    pos = (int)((nr << 8) | nc);
  }
  __syncwarp();

  // ---- action mask, connected / done, reward on the new grid
  const StepResult s = after_move(sg, agent, a, pos, tgt, was, win, gmask, p);
  const int sc = sc0 + 1;
  const bool terminal = env_ok && (s.ndone == N || sc >= p.time_limit);

  // ---- TimeStep row, State scalars and the episode record of the live envs
  if (env_ok && a == 0) {
    const float ratio = __fdiv_rn((float)s.nconn, (float)N);
    const int tpl = paths + s.nmoved + N;
    if (!LIST) {
      p.ts.step_type[e] = (int8_t)(terminal ? 2 : 1);
      p.ts.num_connections[e] = s.nconn;
      p.ts.ratio_connections[e] = ratio;
      p.ts.total_path_length[e] = tpl;
      p.ts.obs_step_count[e] = sc;
    }
    p.st.step_count[e] = sc;
    p.acc.episode_length[e] += 1;
    if (terminal) {
      p.acc.num_connections[e] = s.nconn;
      p.acc.ratio_connections[e] = ratio;
      p.acc.total_path_length[e] = tpl;
      if (!LIST) p.live[e] = 0;
    }
  }
  if (agent) {
    const long long ga = e * N + a;
    if (!LIST) {
      p.ts.reward[ga] = s.rew;
      p.ts.discount[ga] = (terminal || s.done) ? 0.0f : 1.0f;
      store_mask5(p.ts.action_mask + ga * 5, s.mk3);
    }
    reinterpret_cast<int2 *>(p.st.position)[ga] = make_int2(pos >> 8, pos & 255);
    p.acc.episode_return[ga] = __fadd_rn(p.acc.episode_return[ga], s.rew);
  }
  uint32_t obsm = livem;  // bit m * Np: env m of the warp writes an observation row
  if (!LIST) {
    const int nfinished = __popc(__ballot_sync(FULL, a == 0 && terminal));
    if (lane == 0 && nfinished) atomicSub(p.live_count, nfinished);
  } else {
    // ---- the output rows of the survivors: rank in the warp (ballot), in the CTA (scan of the warp counts), in the
    // list (look-back over the tiles before this one)
    obsm = __ballot_sync(FULL, a == 0 && env_ok && !terminal);
    if (lane == 0) ls[LS_WCOUNT + warp] = __popc(obsm);
    __syncthreads();
    if (warp == 0) {
      const int own = lane < EW_WARPS ? ls[LS_WCOUNT + lane] : 0;
      int incl = own;
      for (int off = 1; off < EW_WARPS; off <<= 1) {
        const int t = __shfl_up_sync(FULL, incl, off);
        if (lane >= off) incl += t;
      }
      const int agg = __shfl_sync(FULL, incl, EW_WARPS - 1);
      const int before = tile_prefix(p.tile_status, tile, agg, lane);
      if (lane < EW_WARPS) ls[LS_WBASE + lane] = before + incl - own;
      if (lane == 0 && tile == p.tiles - 1) *p.count_out = before + agg;
    }
    __syncthreads();
    const bool keep = (obsm >> (j * Np)) & 1u;
    const int row = ls[LS_WBASE + warp] + __popc(obsm & ((1u << (j * Np)) - 1u));
    if (keep) {
      if (a == 0) {
        p.order_out[row] = (int32_t)e;
        p.ts.obs_step_count[row] = sc;
      }
      if (a < N) store_mask5(p.ts.action_mask + ((long long)row * N + a) * 5, s.mk3);
    }
    if (j < kc && a == 0) slots[j] = keep ? row : -1;
    __syncwarp();
  }

  // ---- observation.grid of the live envs (LIST: of the survivors, env m of the warp to row slots[m])
  if (VEC) {
    int4 *odst = reinterpret_cast<int4 *>(p.ts.obs_grid) + e0 * N * c4;
    for (int q = lane; q < kc * c4; q += 32) {
      const int m = (int)p.divC4.div((uint32_t)q);
      if (!((obsm >> (m * Np)) & 1u)) continue;
      const uint32_t w = wg32[q];
      const uint32_t b0 = w & 0xffu, b1 = (w >> 8) & 0xffu, b2 = (w >> 16) & 0xffu, b3 = w >> 24;
      int4 *o = (LIST ? reinterpret_cast<int4 *>(p.ts.obs_grid) + (size_t)slots[m] * N * c4 : odst + (size_t)m * N * c4) + (q - m * c4);
      const uint8_t *row = lut;
#pragma unroll 2
      for (int x = 0; x < N; ++x, o += c4, row += RS) *o = make_int4(row[b0], row[b1], row[b2], row[b3]);
    }
  } else if (LIST) {
    write_obs_scalar(p.ts.obs_grid, wg, lut, RS, kc, cells, N, Np, ~obsm, p.divCells, lane, slots);
  } else {
    write_obs_scalar(p.ts.obs_grid + e0 * N * cells, wg, lut, RS, kc, cells, N, Np, ~livem, p.divCells, lane);
  }
}

static EvalStepParams eval_step_params(const rbg_state &st, const int32_t *action, int64_t B, int G, int N, const rbg_env_params &env,
                                       const rbg_timestep &ts, const rbg_episode_metrics &acc, size_t &smem, int64_t &envs_per_cta, bool &vec) {
  EvalStepParams p;
  memset(&p, 0, sizeof(p));
  p.st = st;
  p.ts = ts;
  p.acc = acc;
  p.action = action;
  p.B = B;
  p.G = G;
  p.N = N;
  p.time_limit = env.time_limit;
  p.timestep_reward = env.timestep_reward;
  p.connected_reward = env.connected_reward;
  const WarpShape s = warp_shape(G, N);
  const size_t lutB = lut_bytes(N, obs_lut_stride(N));
  set_warp_shape(p, s, lutB);
  smem = lutB + EW_WARPS * s.wgrid;
  envs_per_cta = EW_WARPS * s.K;
  vec = s.vec();
  return p;
}

int launch_eval_step(const rbg_state &st, const int32_t *action, uint8_t *live, int32_t *live_count, int64_t B, int G, int N,
                     const rbg_env_params &env, const rbg_timestep &ts, const rbg_episode_metrics &acc, cudaStream_t stream) {
  if (B <= 0) return RBG_OK;
  size_t smem;
  int64_t E;
  bool vec;
  EvalStepParams p = eval_step_params(st, action, B, G, N, env, ts, acc, smem, E, vec);
  p.live = live;
  p.live_count = live_count;
  const int64_t ctas = (B + E - 1) / E;
  void (*fn)(const EvalStepParams) = vec ? eval_step_kernel<true, false> : eval_step_kernel<false, false>;
  return launch_kernel(fn, (unsigned)ctas, EW_WARPS * 32, smem, stream, RBG_K_EVAL_STEP, "eval_step_kernel", false, p);
}

int launch_eval_step_live(const rbg_state &st, const int32_t *action, const int32_t *order_in, int64_t L, int32_t *order_out, int32_t *count_out,
                          int64_t B, int G, int N, const rbg_env_params &env, const rbg_timestep &ts, const rbg_episode_metrics &acc,
                          cudaStream_t stream) {
  if (L <= 0) return RBG_OK;
  size_t smem;
  int64_t E;
  bool vec;
  EvalStepParams p = eval_step_params(st, action, B, G, N, env, ts, acc, smem, E, vec);
  p.so_list = (int)smem;
  smem += up16(sizeof(int) * LS_INTS);
  p.order_in = order_in;
  p.order_out = order_out;
  p.count_out = count_out;
  p.L = L;
  p.tiles = (L + E - 1) / E;
  // the tile status words and the ticket: stream-ordered scratch, cleared before the launch, so that the caller needs
  // no workspace and launches on different streams never share it
  const size_t bytes = 8 * (size_t)p.tiles + 16;
  keep_pool_cached();
  void *scratch = nullptr;
  cudaError_t ce;
  if ((ce = cudaMallocAsync(&scratch, bytes, stream)) != cudaSuccess) return set_cuda_error(ce, "cudaMallocAsync(eval step tile status)");
  p.tile_status = static_cast<unsigned long long *>(scratch);
  p.ticket = reinterpret_cast<int *>(static_cast<char *>(scratch) + 8 * (size_t)p.tiles);
  int rc = RBG_OK;
  if ((ce = cudaMemsetAsync(scratch, 0, bytes, stream)) != cudaSuccess) {
    rc = set_cuda_error(ce, "cudaMemsetAsync(eval step tile status)");
  } else {
    void (*fn)(const EvalStepParams) = vec ? eval_step_kernel<true, true> : eval_step_kernel<false, true>;
    rc = launch_kernel(fn, (unsigned)p.tiles, EW_WARPS * 32, smem, stream, RBG_K_EVAL_STEP, "eval_step_kernel<LIST>", false, p);
  }
  cudaFreeAsync(scratch, stream);
  return rc;
}

}  // namespace rbg
