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
  for (int a = warp; a < N; a += EW_WARPS)
    for (int v = lane; v < RS; v += 32) lut[a * RS + v] = v <= 3 * N ? (uint8_t)obs_value(v, 3 * a, 3 * N) : (uint8_t)0;
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

  // ---- load: State.grid int32 -> uint8 (one packed word per int4), agent and env scalars
  if (VEC) {
    // four loads in flight per lane before the first one is used (a load-use pair per iteration
    // made a warp pay one L2 round trip per 32 words: 19 % of the kernel's stall samples)
    const int4 *src = reinterpret_cast<const int4 *>(p.in.grid) + e0 * c4;
    const int nq = kc * c4;
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
    const int32_t *src = p.in.grid + e0 * cells;
    for (int i = lane; i < kc * cells; i += 32) wg[i] = (uint8_t)__ldg(src + i);
  }
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
  int paths = 0;
  if (env_ok) {
    if (VEC) {
      for (int q = a; q < c4; q += Np) paths += count_path_codes(wg32[j * c4 + q]);
    } else {
      for (int i = a; i < cells; i += Np) paths += (g[i] % 3u == 1u) ? 1 : 0;
    }
  }
  for (int off = Np >> 1; off; off >>= 1) paths += __shfl_xor_sync(FULL, paths, off);

  // ---- agents: (sample action,) move_position, is_valid_position, collisions
  const bool was = agent && pos == tgt;
  int r = pos >> 8, c = pos & 255, dest = -1;
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
  const bool now = agent && pos == tgt;
  uint32_t mk3 = 0;
  if (agent) mk3 = move_mask(sg, pos >> 8, pos & 255, a, now);
  const bool done = now || mk3 == 0u;  // connected_or_blocked
  const float rew = __fadd_rn(__fmul_rn(p.env.connected_reward, (!was && now) ? 1.0f : 0.0f), __fmul_rn(p.env.timestep_reward, was ? 0.0f : 1.0f));
  const int ndone = __popc(__ballot_sync(FULL, agent && done) & gmask);
  const int nconn = __popc(__ballot_sync(FULL, now) & gmask);
  const int nmoved = __popc(__ballot_sync(FULL, win) & gmask);

  // ---- per env: termination, auto-reset bookkeeping (group-uniform values)
  const int sc = sc0 + (is_step ? 1 : 0);
  const bool terminal = is_step && env_ok && (ndone == N || sc >= p.env.time_limit);
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
    p.ts.num_connections[e] = nconn;
    p.ts.ratio_connections[e] = __fdiv_rn((float)nconn, (float)N);
    p.ts.total_path_length[e] = paths + nmoved + N;
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
    p.ts.reward[ga] = is_step ? rew : 0.0f;
    p.ts.discount[ga] = is_step ? ((terminal || done) ? 0.0f : 1.0f) : 1.0f;
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

  // ---- bulk outputs: State.grid and observation.grid (see env_kernel phase 4)
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
  for (int a = warp; a < N; a += EW_WARPS)
    for (int v = lane; v < RS; v += 32) lut[a * RS + v] = v <= 3 * N ? (uint8_t)obs_value(v, 3 * a, 3 * N) : (uint8_t)0;
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
  if (VEC) {
    // four loads in flight per lane before the first one is used (a load-use pair per iteration
    // made a warp pay one L2 round trip per 32 words: 19 % of the kernel's stall samples)
    const int4 *src = reinterpret_cast<const int4 *>(p.in.grid) + e0 * c4;
    const int nq = kc * c4;
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
    const int32_t *src = p.in.grid + e0 * cells;
    for (int i = lane; i < kc * cells; i += 32) wg[i] = (uint8_t)__ldg(src + i);
  }
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
  int paths = 0;  // PATH cells of the env (extras: total_path_length), carried across steps
  if (env_ok) {
    if (VEC) {
      for (int q = a; q < c4; q += Np) paths += count_path_codes(wg32[j * c4 + q]);
    } else {
      for (int i = a; i < cells; i += Np) paths += (g[i] % 3u == 1u) ? 1 : 0;
    }
  }
  for (int off = Np >> 1; off; off >>= 1) paths += __shfl_xor_sync(FULL, paths, off);
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
    int dest = -1;
    if (agent) {
      // the action comes from mk3 = is_valid_position of the four moves on this very grid (empty mask
      // for a connected agent), so a non-NOOP action needs no second validity test
      const int action = random_action(k0, k1, (uint32_t)sc, (uint32_t)a, mk3);
      if (rp.action_out) rp.action_out[row_a] = action;
      if (action != NOOP) dest = r * G + c + (action == UP ? -G : (action == DOWN ? G : (action == RIGHT ? 1 : -1)));
    }
    const uint32_t mval = dest >= 0 ? (((uint32_t)j << 16) | (uint32_t)dest) : (0x80000000u | (uint32_t)lane);
    const uint32_t mm = __match_any_sync(FULL, mval);
    const bool win = dest >= 0 && lane == 31 - __clz(mm);
    __syncwarp();
    if (win) {
      g[r * G + c] = (uint8_t)(3 * a + PATH);
      g[dest] = (uint8_t)(3 * a + POSITION);
      uint32_t nr, nc;
      p.divG.divmod((uint32_t)dest, nr, nc);
      pos = (int)((nr << 8) | nc);
    }
    __syncwarp();
    // ---- action mask, connected / done, reward on the new grid
    const bool now = agent && pos == tgt;
    mk3 = 0;
    if (agent) mk3 = move_mask(sg, pos >> 8, pos & 255, a, now);
    const bool done = now || mk3 == 0u;
    const float rew = __fadd_rn(__fmul_rn(p.env.connected_reward, (!was && now) ? 1.0f : 0.0f), __fmul_rn(p.env.timestep_reward, was ? 0.0f : 1.0f));
    const int ndone = __popc(__ballot_sync(FULL, agent && done) & gmask);
    const int nconn = __popc(__ballot_sync(FULL, now) & gmask);
    paths += __popc(__ballot_sync(FULL, win) & gmask);
    sc += 1;
    const bool terminal = env_ok && (ndone == N || sc >= p.env.time_limit);
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
      p.ts.num_connections[row_e] = nconn;
      p.ts.ratio_connections[row_e] = ratio_lut[nconn];
      p.ts.total_path_length[row_e] = tpl;
      p.ts.obs_step_count[row_e] = terminal ? 0 : sc;
    }
    if (agent) {
      p.ts.reward[row_a] = rew;
      p.ts.discount[row_a] = (terminal || done) ? 0.0f : 1.0f;
    }
    if (terminal) {  // group-uniform: swap in the new episode (pins-only grid, heads then targets)
      for (int i = a; i < cells; i += Np) g[i] = 0;
      pos = npos;
      tgt = ntgt;
      start = npos;
      k0 = nk0;
      k1 = nk1;
      sc = 0;
      paths = 0;
      __syncwarp(gmask);
      if (a < N) g[(pos >> 8) * G + (pos & 255)] = (uint8_t)(3 * a + POSITION);
      __syncwarp(gmask);
      if (a < N) g[(tgt >> 8) * G + (tgt & 255)] = (uint8_t)(3 * a + TARGET);
      __syncwarp(gmask);
      if (a < N) mk3 = move_mask(sg, pos >> 8, pos & 255, a, pos == tgt);
    }
    __syncwarp();
    if (agent) store_mask5(p.ts.action_mask + row_a * 5, mk3);
    // ---- observation of step t
    if (VEC) {
      int4 *odst = obs_t;
      obs_t += obs_step;
      if (OBS == 2)
        os.emit(kc, N, c4, lane, odst);
      else
        os.emit_direct(lut, wg32, kc, N, c4, lane, odst);
    } else {
      int32_t *odst = p.ts.obs_grid + (tb + e0) * N * cells;
      for (int i = lane; i < kc * cells; i += 32) {
        const int m = (int)p.divCells.div((uint32_t)i);
        const uint32_t v = wg[i];
        int32_t *o = odst + (size_t)m * N * cells + (i - m * cells);
        for (int x = 0; x < N; ++x, o += cells) *o = lut[x * RS + v];
      }
    }
    __syncwarp();  // the next step's writes must not overtake these reads
  }

  // ---- write the State once
  if (VEC) {
    if (OBS == 2) os.drain(lane);
    int4 *gdst = reinterpret_cast<int4 *>(p.out.grid) + e0 * c4;
    for (int q = lane; q < kc * c4; q += 32) gdst[q] = bytes_to_int4(wg32[q]);
  } else {
    int32_t *gdst = p.out.grid + e0 * cells;
    for (int i = lane; i < kc * cells; i += 32) gdst[i] = wg[i];
  }
  if (env_ok && a == 0) {
    p.out.step_count[e] = sc;
    p.out.key[2 * e] = k0;
    p.out.key[2 * e + 1] = k1;
  }
  if (agent) {
    const long long ga = e * N + a;
    reinterpret_cast<int2 *>(p.out.position)[ga] = make_int2(pos >> 8, pos & 255);
    reinterpret_cast<int2 *>(p.out.target)[ga] = make_int2(tgt >> 8, tgt & 255);
    reinterpret_cast<int2 *>(p.out.start)[ga] = make_int2(start >> 8, start & 255);
    p.out.agent_id[ga] = a;
  }
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
  for (int a = warp; a < N; a += nwarps)
    for (int v = lane; v < RS; v += 32) lut[a * RS + v] = v <= 3 * N ? (uint8_t)obs_value(v, 3 * a, 3 * N) : (uint8_t)0;
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
    if (VEC) {
      const int4 *src = reinterpret_cast<const int4 *>(p.in.grid) + e0 * c4;
      const int nq = kc * c4;
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
      const int32_t *src = p.in.grid + e0 * cells;
      for (int i = lane; i < kc * cells; i += 32) wg[i] = (uint8_t)__ldg(src + i);
    }
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
    int paths = 0;  // PATH cells of the env (extras: total_path_length), carried across steps
    if (env_ok) {
      if (VEC) {
        for (int q = a; q < c4; q += Np) paths += count_path_codes(wg32[j * c4 + q]);
      } else {
        for (int i = a; i < cells; i += Np) paths += (g[i] % 3u == 1u) ? 1 : 0;
      }
    }
    for (int off = Np >> 1; off; off >>= 1) paths += __shfl_xor_sync(FULL, paths, off);
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
      int dest = -1;
      if (agent) {
        const int action = random_action(k0, k1, (uint32_t)sc, (uint32_t)a, mk3);
        if (rp.action_out) rp.action_out[row_a] = action;
        if (action != NOOP) dest = r * G + c + (action == UP ? -G : (action == DOWN ? G : (action == RIGHT ? 1 : -1)));
      }
      const uint32_t mval = dest >= 0 ? (((uint32_t)j << 16) | (uint32_t)dest) : (0x80000000u | (uint32_t)lane);
      const uint32_t mm = __match_any_sync(FULL, mval);
      const bool win = dest >= 0 && lane == 31 - __clz(mm);
      __syncwarp();
      if (win) {
        g[r * G + c] = (uint8_t)(3 * a + PATH);
        g[dest] = (uint8_t)(3 * a + POSITION);
        uint32_t nr, nc;
        p.divG.divmod((uint32_t)dest, nr, nc);
        pos = (int)((nr << 8) | nc);
      }
      __syncwarp();
      // ---- action mask, connected / done, reward on the new grid
      const bool now = agent && pos == tgt;
      mk3 = 0;
      if (agent) mk3 = move_mask(sg, pos >> 8, pos & 255, a, now);
      const bool done = now || mk3 == 0u;
      const float rew = __fadd_rn(__fmul_rn(p.env.connected_reward, (!was && now) ? 1.0f : 0.0f), __fmul_rn(p.env.timestep_reward, was ? 0.0f : 1.0f));
      const int ndone = __popc(__ballot_sync(FULL, agent && done) & gmask);
      const int nconn = __popc(__ballot_sync(FULL, now) & gmask);
      paths += __popc(__ballot_sync(FULL, win) & gmask);
      sc += 1;
      const bool terminal = env_ok && (ndone == N || sc >= p.env.time_limit);
      const int tpl = paths + N;
      // ---- small outputs of step t (the terminal step keeps its reward / discount / step_type / extras)
      if (env_ok && a == 0) {
        p.ts.step_type[row_e] = (int8_t)(terminal ? 2 : 1);
        p.ts.num_connections[row_e] = nconn;
        p.ts.ratio_connections[row_e] = ratio_lut[nconn];
        p.ts.total_path_length[row_e] = tpl;
        p.ts.obs_step_count[row_e] = terminal ? 0 : sc;
      }
      if (agent) {
        p.ts.reward[row_a] = rew;
        p.ts.discount[row_a] = (terminal || done) ? 0.0f : 1.0f;
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
        for (int i = a; i < cells; i += Np) g[i] = 0;
        pos = (int)(pin >> 16);
        tgt = (int)(pin & 0xffffu);
        start = pos;
        k0 = nk.x;
        k1 = nk.y;
        sc = 0;
        paths = 0;
        if (a == 0) {  // the episode after this one
          atomicAdd(pp.group_pending + grp, 1);
          genq_post(myq, (int)e, k0, k1);
        }
        __syncwarp(gmask);
        if (a < N) g[(pos >> 8) * G + (pos & 255)] = (uint8_t)(3 * a + POSITION);
        __syncwarp(gmask);
        if (a < N) g[(tgt >> 8) * G + (tgt & 255)] = (uint8_t)(3 * a + TARGET);
        __syncwarp(gmask);
        if (a < N) mk3 = move_mask(sg, pos >> 8, pos & 255, a, pos == tgt);
      }
      __syncwarp();
      if (agent) store_mask5(p.ts.action_mask + row_a * 5, mk3);
      // ---- observation of step t
      if (VEC) {
        int4 *odst = obs_t;
        obs_t += obs_step;
        if (OBS == 2)
          os.emit(kc, N, c4, lane, odst);
        else
          os.emit_direct(lut, wg32, kc, N, c4, lane, odst);
      } else {
        int32_t *odst = p.ts.obs_grid + (tb + e0) * N * cells;
        for (int i = lane; i < kc * cells; i += 32) {
          const int m = (int)p.divCells.div((uint32_t)i);
          const uint32_t v = wg[i];
          int32_t *o = odst + (size_t)m * N * cells + (i - m * cells);
          for (int x = 0; x < N; ++x, o += cells) *o = lut[x * RS + v];
        }
      }
      __syncwarp();  // the next step's writes must not overtake these reads
    }

    // ---- write the State once
    if (VEC) {
      int4 *gdst = reinterpret_cast<int4 *>(p.out.grid) + e0 * c4;
      for (int q = lane; q < kc * c4; q += 32) gdst[q] = bytes_to_int4(wg32[q]);
    } else {
      int32_t *gdst = p.out.grid + e0 * cells;
      for (int i = lane; i < kc * cells; i += 32) gdst[i] = wg[i];
    }
    if (env_ok && a == 0) {
      p.out.step_count[e] = sc;
      p.out.key[2 * e] = k0;
      p.out.key[2 * e + 1] = k1;
    }
    if (agent) {
      const long long ga = e * N + a;
      reinterpret_cast<int2 *>(p.out.position)[ga] = make_int2(pos >> 8, pos & 255);
      reinterpret_cast<int2 *>(p.out.target)[ga] = make_int2(tgt >> 8, tgt & 255);
      reinterpret_cast<int2 *>(p.out.start)[ga] = make_int2(start >> 8, start & 255);
      p.out.agent_id[ga] = a;
    }
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

int launch_env(EnvParams p, cudaStream_t stream, bool pdl) {
  const int G = p.G, N = p.N;
  p.cells = G * G;
  const bool vec = (p.cells & 3) == 0;
  p.divN = FastDiv::make((uint32_t)N);
  p.divG = FastDiv::make((uint32_t)G);
  p.divC4 = FastDiv::make((uint32_t)(vec ? p.cells >> 2 : 1));
  p.divCells = FastDiv::make((uint32_t)p.cells);
  if (p.B <= 0) return RBG_OK;
  int Np = 1;
  while (Np < N) Np <<= 1;
  p.Np = Np;
  const int K = 32 / Np;
  p.E = EW_WARPS * K;
  const size_t lutB = ((size_t)N * obs_lut_stride(N) + 256 + 15) & ~(size_t)15;
  const size_t wgrid = ((size_t)K * p.cells + 15) & ~(size_t)15;
  p.so[0] = (int)lutB;
  p.so[1] = (int)wgrid;
  const size_t smem = lutB + EW_WARPS * wgrid;
  const int64_t ctas = (p.B + p.E - 1) / p.E;
  LaunchScope scope(RBG_K_ENV, stream);
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = dim3((unsigned)ctas);
  cfg.blockDim = dim3(EW_WARPS * 32);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = pdl ? 1 : 0;
  cudaError_t ce = vec ? cudaLaunchKernelEx(&cfg, env_warp_kernel<true>, p) : cudaLaunchKernelEx(&cfg, env_warp_kernel<false>, p);
  if (ce != cudaSuccess) return set_cuda_error(ce, "cudaLaunchKernelEx(env_warp_kernel)");
  return check_launch("env_warp_kernel");
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

int launch_rollout(EnvParams p, int T, int32_t *action_out, cudaStream_t stream) {
  const int G = p.G, N = p.N;
  p.cells = G * G;
  const bool vec = (p.cells & 3) == 0;
  p.divN = FastDiv::make((uint32_t)N);
  p.divG = FastDiv::make((uint32_t)G);
  p.divC4 = FastDiv::make((uint32_t)(vec ? p.cells >> 2 : 1));
  p.divCells = FastDiv::make((uint32_t)p.cells);
  if (p.B <= 0 || T <= 0) return RBG_OK;
  int Np = 1;
  while (Np < N) Np <<= 1;
  p.Np = Np;
  const int K = 32 / Np;
  p.E = EW_WARPS * K;
  const size_t lutB = ((size_t)N * OBS_RS + 256 + 15) & ~(size_t)15;
  const size_t wgrid = ((size_t)K * p.cells + 15) & ~(size_t)15;
  p.so[0] = (int)lutB;
  p.so[1] = (int)wgrid;
  RolloutParams rp;
  rp.T = T;
  rp.action_out = action_out;
  rp.ratio_off = (int)(lutB + EW_WARPS * wgrid);
  size_t smem = (((size_t)rp.ratio_off + 4 * (RBG_MAX_N + 4)) + 15) & ~(size_t)15;
  rp.stage_off = (int)smem;
  rp.stage_bytes = 0;
  rp.stage_nbuf = 1;
  rp.stage_warp = 0;
  rp.ce = 1;
  rp.cv = N;
  if (vec) {
    const ObsStagePlan pl = obs_stage_plan(K, N, p.cells, 4096, 8192);
    rp.stage_bytes = pl.bytes;
    rp.stage_nbuf = pl.nbuf;
    rp.ce = pl.ce;
    rp.cv = pl.cv;
    rp.stage_warp = (rp.stage_nbuf * rp.stage_bytes + 15) & ~15;
    smem += (size_t)EW_WARPS * rp.stage_warp;
  }
  if (smem > 200 * 1024) return set_error(RBG_EINVAL, "rollout: shared memory %zu too large", smem);
  const int64_t ctas = (p.B + p.E - 1) / p.E;
  {  // residency: registers allow kRolloutMinCtas per SM, shared memory (1 KB reserved per CTA) maybe fewer
    int cmax = (int)(device_smem_per_sm() / (smem + 1024));
    if (cmax > kRolloutMinCtas) cmax = kRolloutMinCtas;
    if (cmax >= 3) smem = balance_waves(ctas, cmax, cmax - 2, smem);
  }
  LaunchScope scope(RBG_K_ROLLOUT, stream);
  const bool staged = vec && rp.stage_nbuf != 0;
  if (staged) {
    if (smem > 48 * 1024) cudaFuncSetAttribute(rollout_warp_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    rollout_warp_kernel<2><<<(unsigned)ctas, EW_WARPS * 32, smem, stream>>>(p, rp);
  } else if (vec) {
    if (smem > 48 * 1024) cudaFuncSetAttribute(rollout_warp_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    rollout_warp_kernel<1><<<(unsigned)ctas, EW_WARPS * 32, smem, stream>>>(p, rp);
  } else {
    if (smem > 48 * 1024) cudaFuncSetAttribute(rollout_warp_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    rollout_warp_kernel<0><<<(unsigned)ctas, EW_WARPS * 32, smem, stream>>>(p, rp);
  }
  return check_launch("rollout_warp_kernel");
}

// The persistent rollout with in-CTA generator warps (rollout_persist_kernel).  `cache_*` of `p` must be set;
// `counter` points at two zeroed ints that the kernel recycles by itself.
int launch_rollout_persist(EnvParams p, int kind, int T, int32_t *action_out, int32_t *counter, int32_t *group_done, int32_t *group_pending,
                           int epoch, bool overlap, uint64_t *cache_tag_w, uint2 *cache_key_w, uint32_t *cache_pins_w, cudaStream_t stream) {
  const int G = p.G, N = p.N;
  p.cells = G * G;
  const bool vec = (p.cells & 3) == 0;
  p.divN = FastDiv::make((uint32_t)N);
  p.divG = FastDiv::make((uint32_t)G);
  p.divC4 = FastDiv::make((uint32_t)(vec ? p.cells >> 2 : 1));
  p.divCells = FastDiv::make((uint32_t)p.cells);
  if (p.B <= 0 || T <= 0) return RBG_OK;
  int Np = 1;
  while (Np < N) Np <<= 1;
  p.Np = Np;
  const int K = 32 / Np;
  p.E = EW_WARPS * K;
  auto up16 = [](size_t x) { return (x + 15) & ~(size_t)15; };
  const size_t lutB = up16((size_t)N * OBS_RS + 256);
  const size_t wgrid = up16((size_t)K * p.cells);
  p.so[0] = (int)lutB;
  p.so[1] = (int)wgrid;
  RolloutParams rp;
  memset(&rp, 0, sizeof(rp));
  rp.T = T;
  rp.action_out = action_out;
  // CTA shape.  "Isolated": 3 env warps + 1 generator warp = 4 warps per CTA, one per SM sub-partition, so the generator
  // warps of all resident CTAs share ONE sub-partition and never compete with env warps for issue slots, at most 4 CTAs
  // per SM.  "Packed": 4 env + 2 generator warps, as many CTAs as fit.  Measured (65 536 envs, M env-steps/s, isolated /
  // packed): 10x10/5 2501 / 2338, 12x12/6 1649 / 1508, 10x10/4 2884 / 2850, 10x10/8 1598 / 1596; 8x8/4 2817 / 3432,
  // 8x8/8 1477 / 1687, 6x6/3 2623 / 2989 (issue-bound: more env warps win); 14x14/7 1013 / 1034, 16x16/8 761 / 774,
  // 20x20/10 372 / 378, 32x32/16 94.9 / 96.8 (resets are rare per byte: packed is 2 % ahead).
  const bool isolated = G >= 9 && G <= 13 && N <= 8;
  const int PW = isolated ? 3 : EW_WARPS;
  size_t off = lutB + PW * wgrid;
  rp.ratio_off = (int)off;
  off = up16(off + 4 * (RBG_MAX_N + 4));
  PersistParams pp;
  memset(&pp, 0, sizeof(pp));
  pp.counter = counter + (epoch % kPersistSets) * kPersistSetInts;
  pp.group_done = group_done;
  pp.group_pending = group_pending;
  pp.epoch = epoch;
  pp.ngroups = (int)((p.B + K - 1) / K);
  GenWarpCfg gc = gen_warp_cfg(kind, G, N, &pp.gcand_bytes, &pp.gsel_bytes, &pp.gscr_stride);
  gc.patience = 20;
  gc.cache_tag = reinterpret_cast<unsigned long long *>(cache_tag_w);
  gc.cache_key = cache_key_w;
  gc.cache_pins = cache_pins_w;
  gc.group_pending = group_pending;
  gc.seqlock = 0;  // nobody reads an entry while it is rewritten here (see gen_warp_batch)
  gc.kshift = 0;
  while ((1 << gc.kshift) < K) ++gc.kshift;
  pp.gen_warps = isolated ? 1 : 2;
  pp.env_warps = PW;
  pp.tmpl_off = (int)off;
  off = up16(off + gc.SBp);
  pp.q_off = (int)off;
  off = up16(off + pp.gen_warps * sizeof(GenQueue));
  pp.done_off = (int)off;
  off += 16;
  pp.gscr_off = (int)off;
  off += (size_t)pp.gen_warps * pp.gscr_stride;
  rp.stage_off = (int)off;
  rp.stage_nbuf = 1;
  rp.ce = 1;
  rp.cv = N;
  if (vec) {
    const ObsStagePlan pl = obs_stage_plan(K, N, p.cells, 4096, 8192);
    rp.stage_bytes = pl.bytes;
    rp.stage_nbuf = pl.nbuf;
    rp.ce = pl.ce;
    rp.cv = pl.cv;
    rp.stage_warp = (int)up16((size_t)rp.stage_nbuf * rp.stage_bytes);
    off += (size_t)PW * rp.stage_warp;
  }
  const size_t smem = up16(off);
  if (smem > 200 * 1024) return set_error(RBG_EINVAL, "rollout: shared memory %zu too large", smem);
  const bool staged = vec && rp.stage_nbuf != 0;
  const int threads = (PW + pp.gen_warps) * 32;
  const void *fn = staged ? (const void *)rollout_persist_kernel<2> : (vec ? (const void *)rollout_persist_kernel<1> : (const void *)rollout_persist_kernel<0>);
  cudaError_t ce;
  if (smem > 48 * 1024 && (ce = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)) != cudaSuccess)
    return set_cuda_error(ce, "cudaFuncSetAttribute(rollout_persist_kernel)");
  int resident = 0;
  if ((ce = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&resident, fn, threads, smem)) != cudaSuccess) return set_cuda_error(ce, "cudaOccupancyMaxActiveBlocksPerMultiprocessor");
  if (resident < 1) return set_error(RBG_EINVAL, "rollout_persist_kernel does not fit an SM (%zu bytes of shared memory)", smem);
  if (isolated && resident > 4) resident = 4;  // more resident CTAs measure slower (5: +0.6 %, 6-8: +1.1 %)
  int64_t ctas = (int64_t)resident * device_sm_count();
  const int64_t need = (pp.ngroups + PW - 1) / PW;
  if (ctas > need) ctas = need;
  LaunchScope scope(RBG_K_ROLLOUT, stream);
  // programmatic dependent launch: this grid may begin while the previous kernel of the stream is still
  // running, if that kernel said so (rollout_persist_kernel does; anything else completes first)
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = dim3((unsigned)ctas);
  cfg.blockDim = dim3((unsigned)threads);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = overlap ? 1 : 0;
  if (staged)
    ce = cudaLaunchKernelEx(&cfg, rollout_persist_kernel<2>, p, rp, pp, gc);
  else if (vec)
    ce = cudaLaunchKernelEx(&cfg, rollout_persist_kernel<1>, p, rp, pp, gc);
  else
    ce = cudaLaunchKernelEx(&cfg, rollout_persist_kernel<0>, p, rp, pp, gc);
  if (ce != cudaSuccess) return set_cuda_error(ce, "cudaLaunchKernelEx(rollout_persist_kernel)");
  return check_launch("rollout_persist_kernel");
}

int launch_random_actions(const rbg_state &st, int64_t B, int G, int N, int32_t *action, cudaStream_t stream) {
  const int64_t n = B * N;
  if (n <= 0) return RBG_OK;
  {
    LaunchScope scope(RBG_K_RANDACT, stream);
    random_actions_kernel<<<(unsigned)((n + 255) / 256), 256, 0, stream>>>(st, B, G, N, FastDiv::make((uint32_t)N), action);
  }
  return check_launch("random_actions_kernel");
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

    // ---- one step (rollout_warp_kernel's step body): sample action, move, collisions
    const bool was = agent && pos == tgt;
    const int r = pos >> 8, c = pos & 255;
    int dest = -1;
    if (agent) {
      const int action = random_action(k0, k1, (uint32_t)sc, (uint32_t)a, mk3);
      if (action != NOOP) dest = r * G + c + (action == UP ? -G : (action == DOWN ? G : (action == RIGHT ? 1 : -1)));
    }
    const uint32_t mval = dest >= 0 ? (((uint32_t)j << 16) | (uint32_t)dest) : (0x80000000u | (uint32_t)lane);
    const uint32_t mm = __match_any_sync(FULL, mval);
    const bool win = dest >= 0 && lane == 31 - __clz(mm);
    __syncwarp();
    if (win) {
      g[r * G + c] = (uint8_t)(3 * a + PATH);
      g[dest] = (uint8_t)(3 * a + POSITION);
      uint32_t nr, nc;
      p.divG.divmod((uint32_t)dest, nr, nc);
      pos = (int)((nr << 8) | nc);
    }
    __syncwarp();
    // ---- action mask, connected / done, reward on the new grid
    const bool now = agent && pos == tgt;
    mk3 = 0;
    if (agent) mk3 = move_mask(sg, pos >> 8, pos & 255, a, now);
    const bool done = now || mk3 == 0u;
    const float rew = __fadd_rn(__fmul_rn(p.connected_reward, (!was && now) ? 1.0f : 0.0f), __fmul_rn(p.timestep_reward, was ? 0.0f : 1.0f));
    const int ndone = __popc(__ballot_sync(FULL, agent && done) & gmask);
    const int nconn = __popc(__ballot_sync(FULL, now) & gmask);
    paths += __popc(__ballot_sync(FULL, win) & gmask);
    sc += 1;
    len += 1;
    ret = __fadd_rn(ret, rew);
    const bool terminal = env_ok && (ndone == N || sc >= p.time_limit);

    // ---- the episode's record (group-uniform)
    if (terminal) {
      if (agent) p.out.episode_return[e * N + a] = ret;
      if (a == 0) {
        p.out.episode_length[e] = len;
        p.out.num_connections[e] = nconn;
        p.out.ratio_connections[e] = ratio_lut[nconn];
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
  p.cells = G * G;
  int Np = 1;
  while (Np < N) Np <<= 1;
  p.Np = Np;
  p.time_limit = env.time_limit;
  p.timestep_reward = env.timestep_reward;
  p.connected_reward = env.connected_reward;
  p.divG = FastDiv::make((uint32_t)G);
  const int K = 32 / Np;
  p.wgrid = (int)(((size_t)K * p.cells + 15) & ~(size_t)15);
  p.ratio_off = EP_WARPS * p.wgrid;
  const size_t smem = (size_t)p.ratio_off + 4 * (RBG_MAX_N + 4);
  cudaError_t ce;
  // few agents on a big board: up to 4 warps x 32 envs x 1 600 cells = 200 KB (40x40/1), past the 48 KB default
  if (smem > 48 * 1024 && (ce = cudaFuncSetAttribute(episode_warp_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)) != cudaSuccess)
    return set_cuda_error(ce, "cudaFuncSetAttribute(episode_warp_kernel)");
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
  if ((ce = cudaMemsetAsync(scratch, 0, 256, stream)) != cudaSuccess) {
    rc = set_cuda_error(ce, "cudaMemsetAsync(episode counter)");
  } else {
    {
      LaunchScope scope(RBG_K_EPISODES, stream);
      episode_warp_kernel<<<ctas, EP_WARPS * 32, smem, stream>>>(p);
    }
    rc = check_launch("episode_warp_kernel");
  }
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
};

template <bool VEC>
__global__ void __launch_bounds__(EW_WARPS * 32, kEnvMinCtas) eval_step_kernel(const EvalStepParams p) {
  extern __shared__ __align__(16) uint8_t smem_raw[];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int G = p.G, N = p.N, cells = p.cells;
  const int Np = p.Np, K = 32 / Np, c4 = cells >> 2;
  const int RS = obs_lut_stride(N);

  const long long e0 = ((long long)blockIdx.x * EW_WARPS + warp) * K;
  const int kc = e0 >= p.B ? 0 : (int)((p.B - e0) < (long long)K ? (p.B - e0) : (long long)K);
  const int j = lane / Np, a = lane & (Np - 1);
  const long long e = e0 + (j < kc ? j : 0);
  const bool env_ok = j < kc && p.live[e] != 0, agent = env_ok && a < N;
  const uint32_t livem = __ballot_sync(FULL, env_ok);  // bit j * Np (and the env's other lanes): env j is live
  if (!__syncthreads_or(livem != 0u)) return;  // a CTA without a live env builds no table
  uint8_t *lut = smem_raw;
  for (int x = warp; x < N; x += EW_WARPS)
    for (int v = lane; v < RS; v += 32) lut[x * RS + v] = v <= 3 * N ? (uint8_t)obs_value(v, 3 * x, 3 * N) : (uint8_t)0;
  __syncthreads();  // the last CTA-wide barrier
  if (livem == 0u) return;
  uint8_t *wg = smem_raw + p.so[0] + (size_t)warp * p.so[1];
  uint32_t *wg32 = reinterpret_cast<uint32_t *>(wg);
  const uint32_t gmask = Np == 32 ? FULL : (((1u << Np) - 1u) << (j * Np));

  // ---- load the live envs: State.grid int32 -> uint8, agent and env scalars
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
        v[u] = ok[u] ? __ldg(src + q) : make_int4(0, 0, 0, 0);
      }
#pragma unroll
      for (int u = 0; u < 4; ++u)
        if (ok[u])
          wg32[q0 + 32 * u] = (uint32_t)(v[u].x & 0xff) | ((uint32_t)(v[u].y & 0xff) << 8) | ((uint32_t)(v[u].z & 0xff) << 16) | ((uint32_t)(v[u].w & 0xff) << 24);
    }
  } else {
    const int32_t *src = p.st.grid + e0 * cells;
    for (int i = lane; i < kc * cells; i += 32)
      if ((livem >> ((int)p.divCells.div((uint32_t)i) * Np)) & 1u) wg[i] = (uint8_t)__ldg(src + i);
  }
  int pos = 0, tgt = 0, action = 0, sc0 = 0;
  if (agent) {
    const int2 ps = __ldg(reinterpret_cast<const int2 *>(p.st.position) + e * N + a);
    const int2 tg = __ldg(reinterpret_cast<const int2 *>(p.st.target) + e * N + a);
    pos = (ps.x << 8) | ps.y;
    tgt = (tg.x << 8) | tg.y;
    action = __ldg(p.action + e * N + a);
  }
  if (env_ok) sc0 = p.st.step_count[e];
  __syncwarp();

  uint8_t *g = wg + (size_t)j * cells;
  const SmemGrid sg{g, G, 0, G};
  // PATH cells of the env before the move (extras: total_path_length)
  int paths = 0;
  if (env_ok) {
    if (VEC) {
      for (int q = a; q < c4; q += Np) paths += count_path_codes(wg32[j * c4 + q]);
    } else {
      for (int i = a; i < cells; i += Np) paths += (g[i] % 3u == 1u) ? 1 : 0;
    }
  }
  for (int off = Np >> 1; off; off >>= 1) paths += __shfl_xor_sync(FULL, paths, off);

  // ---- agents: move_position, is_valid_position, collisions
  const bool was = agent && pos == tgt;
  int r = pos >> 8, c = pos & 255, dest = -1;
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
  const bool now = agent && pos == tgt;
  uint32_t mk3 = 0;
  if (agent) mk3 = move_mask(sg, pos >> 8, pos & 255, a, now);
  const bool done = now || mk3 == 0u;  // connected_or_blocked
  const float rew = __fadd_rn(__fmul_rn(p.connected_reward, (!was && now) ? 1.0f : 0.0f), __fmul_rn(p.timestep_reward, was ? 0.0f : 1.0f));
  const int ndone = __popc(__ballot_sync(FULL, agent && done) & gmask);
  const int nconn = __popc(__ballot_sync(FULL, now) & gmask);
  const int nmoved = __popc(__ballot_sync(FULL, win) & gmask);
  const int sc = sc0 + 1;
  const bool terminal = env_ok && (ndone == N || sc >= p.time_limit);

  // ---- TimeStep row, State scalars and the episode record of the live envs
  if (env_ok && a == 0) {
    const float ratio = __fdiv_rn((float)nconn, (float)N);
    const int tpl = paths + nmoved + N;
    p.ts.step_type[e] = (int8_t)(terminal ? 2 : 1);
    p.ts.num_connections[e] = nconn;
    p.ts.ratio_connections[e] = ratio;
    p.ts.total_path_length[e] = tpl;
    p.ts.obs_step_count[e] = sc;
    p.st.step_count[e] = sc;
    p.acc.episode_length[e] += 1;
    if (terminal) {
      p.acc.num_connections[e] = nconn;
      p.acc.ratio_connections[e] = ratio;
      p.acc.total_path_length[e] = tpl;
      p.live[e] = 0;
    }
  }
  if (agent) {
    const long long ga = e * N + a;
    p.ts.reward[ga] = rew;
    p.ts.discount[ga] = (terminal || done) ? 0.0f : 1.0f;
    store_mask5(p.ts.action_mask + ga * 5, mk3);
    reinterpret_cast<int2 *>(p.st.position)[ga] = make_int2(pos >> 8, pos & 255);
    p.acc.episode_return[ga] = __fadd_rn(p.acc.episode_return[ga], rew);
  }
  const int nfinished = __popc(__ballot_sync(FULL, a == 0 && terminal));
  if (lane == 0 && nfinished) atomicSub(p.live_count, nfinished);

  // ---- observation.grid of the live envs
  if (VEC) {
    int4 *odst = reinterpret_cast<int4 *>(p.ts.obs_grid) + e0 * N * c4;
    for (int q = lane; q < kc * c4; q += 32) {
      const int m = (int)p.divC4.div((uint32_t)q);
      if (!((livem >> (m * Np)) & 1u)) continue;
      const uint32_t w = wg32[q];
      const uint32_t b0 = w & 0xffu, b1 = (w >> 8) & 0xffu, b2 = (w >> 16) & 0xffu, b3 = w >> 24;
      int4 *o = odst + (size_t)m * N * c4 + (q - m * c4);
      const uint8_t *row = lut;
#pragma unroll 2
      for (int x = 0; x < N; ++x, o += c4, row += RS) *o = make_int4(row[b0], row[b1], row[b2], row[b3]);
    }
  } else {
    int32_t *odst = p.ts.obs_grid + e0 * N * cells;
    for (int i = lane; i < kc * cells; i += 32) {
      const int m = (int)p.divCells.div((uint32_t)i);
      if (!((livem >> (m * Np)) & 1u)) continue;
      const uint32_t v = wg[i];
      int32_t *o = odst + (size_t)m * N * cells + (i - m * cells);
      for (int x = 0; x < N; ++x, o += cells) *o = lut[x * RS + v];
    }
  }
}

int launch_eval_step(const rbg_state &st, const int32_t *action, uint8_t *live, int32_t *live_count, int64_t B, int G, int N,
                     const rbg_env_params &env, const rbg_timestep &ts, const rbg_episode_metrics &acc, cudaStream_t stream) {
  if (B <= 0) return RBG_OK;
  EvalStepParams p;
  memset(&p, 0, sizeof(p));
  p.st = st;
  p.ts = ts;
  p.acc = acc;
  p.action = action;
  p.live = live;
  p.live_count = live_count;
  p.B = B;
  p.G = G;
  p.N = N;
  p.cells = G * G;
  const bool vec = (p.cells & 3) == 0;
  int Np = 1;
  while (Np < N) Np <<= 1;
  p.Np = Np;
  p.time_limit = env.time_limit;
  p.timestep_reward = env.timestep_reward;
  p.connected_reward = env.connected_reward;
  p.divG = FastDiv::make((uint32_t)G);
  p.divC4 = FastDiv::make((uint32_t)(vec ? p.cells >> 2 : 1));
  p.divCells = FastDiv::make((uint32_t)p.cells);
  const int K = 32 / Np;
  const size_t lutB = ((size_t)N * obs_lut_stride(N) + 256 + 15) & ~(size_t)15;
  const size_t wgrid = ((size_t)K * p.cells + 15) & ~(size_t)15;
  p.so[0] = (int)lutB;
  p.so[1] = (int)wgrid;
  const size_t smem = lutB + EW_WARPS * wgrid;
  const int64_t ctas = (B + (int64_t)EW_WARPS * K - 1) / ((int64_t)EW_WARPS * K);
  void (*fn)(const EvalStepParams) = vec ? eval_step_kernel<true> : eval_step_kernel<false>;
  cudaError_t ce;
  // few agents on a big board: up to 4 warps x 32 envs x 1 600 cells = 200 KB (40x40/1), past the 48 KB default
  if (smem > 48 * 1024 && (ce = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)) != cudaSuccess)
    return set_cuda_error(ce, "cudaFuncSetAttribute(eval_step_kernel)");
  {
    LaunchScope scope(RBG_K_EVAL_STEP, stream);
    fn<<<(unsigned)ctas, EW_WARPS * 32, smem, stream>>>(p);
  }
  return check_launch("eval_step_kernel");
}

}  // namespace rbg
