// gen_warp.cuh -- generator warps inside the fused rollout kernel.
//
// The fused rollout (connector_kernel.cu, rollout_persist_kernel) is HBM-write bound and leaves about
// half of the SM's issue slots idle; regenerating the boards of finished envs (VmapAutoResetWrapper
// with ParallelRandomWalkGenerator / UniformRandomGenerator) is integer-issue bound and needs no
// memory bandwidth.  A separate refill kernel cannot share an SM with the rollout CTAs (their shared
// memory fills it), so the two used to alternate.  Here every rollout CTA carries its own generator
// warps: the env warps post "generate the episode that follows key K for env e" requests into a
// shared-memory ring, a generator warp takes up to 32 / W of them at a time (W lanes per board, lane =
// agent, exactly the lane layout of prw_kernel's walk), and publishes each result into the env's
// next-episode cache entry in global memory (the same seqlock-tagged entry the per-step path uses).
//
// Algorithm and key derivation as prw_kernel.cu (reference parallel_random_walk.py:60-447,
// parallel_random_walk_generator.py:46-77, uniform_generator.py:70-109; VmapAutoResetWrapper's
// `key, _ = split(state.key)` first).
#pragma once

#include <string.h>

#include "rbg_device.cuh"
#include "select.cuh"

namespace rbg {

constexpr int GENQ_CAP = 64;  // requests in flight per queue (power of two)

// multi-producer (one lane per finished env), single-consumer (one generator warp) ring
struct GenQueue {
  unsigned tail;            // next ticket (producers, atomicAdd)
  volatile unsigned head;   // first ticket not yet taken (consumer)
  volatile int urgent;      // an env is waiting for its episode: do not hold a partial batch back
  volatile unsigned seq[GENQ_CAP];  // slot holds ticket t once seq == t + 1
  int env[GENQ_CAP];
  uint32_t k0[GENQ_CAP], k1[GENQ_CAP];
};

__device__ __forceinline__ void genq_init(GenQueue *q, int lane) {
  for (int i = lane; i < GENQ_CAP; i += 32) q->seq[i] = 0u;
  if (lane == 0) {
    q->tail = 0u;
    q->head = 0u;
    q->urgent = 0;
  }
}

// one lane: "generate the episode that follows State.key (k0, k1) of env e"
__device__ __forceinline__ void genq_post(GenQueue *q, int e, uint32_t k0, uint32_t k1) {
  const unsigned t = atomicAdd(&q->tail, 1u);
  while ((int)(t - q->head) >= GENQ_CAP) __nanosleep(64);  // ring full: the consumer never waits for us, so this ends
  const unsigned s = t & (GENQ_CAP - 1);
  q->env[s] = e;
  q->k0[s] = k0;
  q->k1[s] = k1;
  __threadfence_block();
  q->seq[s] = t + 1u;
}

struct GenWarpCfg {
  int kind;            // RBG_GEN_PRW / RBG_GEN_UNIFORM
  int G, N, W;         // W lanes per board (power of two >= N, >= N + 2 when that fits a warp)
  int S, SBp, cells;   // padded board: row stride, bytes
  int nsel, nselp, cap;
  int patience;        // polls (0.5 us each) a partial batch may wait for more requests
  uint32_t thresh;
  FastDiv divG;
  unsigned long long *cache_tag;
  uint2 *cache_key;
  uint32_t *cache_pins;
  // requests in flight per env group (see rollout_persist_kernel "launch overlap"): +1 when posted, -1 once published
  // (NULL: not counted)
  int *group_pending;
  int seqlock;         // readers may be running (per-step path): invalidate the entry's tag before rewriting it
  int kshift;          // log2(envs per group)
};

// The fields of a GenWarpCfg that follow from the board shape, and the bytes of one generator warp's GenWarpScratch
// arrays in shared memory (cand, sel; the whole stride includes the boards).  The caller sets the cache pointers,
// group_pending, kshift, seqlock and patience.
inline GenWarpCfg gen_warp_cfg(int kind, int G, int N, int *gcand_bytes, int *gsel_bytes, int *gscr_stride) {
  auto up16 = [](size_t x) { return (x + 15) & ~(size_t)15; };
  GenWarpCfg gc;
  memset(&gc, 0, sizeof(gc));
  gc.kind = kind;
  gc.G = G;
  gc.N = N;
  int W = 1;  // W lanes per board, N + 2 of them busy when that fits (agents + the two key-advance lanes)
  while (W < N + 2 && W < 32) W <<= 1;
  gc.W = W;
  gc.S = G + 4;
  gc.SBp = (int)up16((size_t)gc.S * gc.S);
  gc.cells = G * G;
  gc.nsel = kind == RBG_GEN_PRW ? N : 2 * N;
  gc.nselp = (gc.nsel + 1) & ~1;
  gc.cap = 4 * gc.nsel + 32;
  {
    const double frac = (2.0 * gc.nsel + 16.0) / (double)gc.cells;
    gc.thresh = frac >= 1.0 ? 0xffffffffu : (uint32_t)(frac * 4294967296.0);
  }
  gc.divG = FastDiv::make((uint32_t)G);
  const int gpw = 32 / W;
  *gcand_bytes = (int)up16((size_t)gc.cap * 8);
  *gsel_bytes = (int)up16((size_t)gpw * gc.nselp * 2);
  *gscr_stride = (int)up16((size_t)*gcand_bytes + *gsel_bytes + (size_t)gpw * gc.SBp);
  return gc;
}

struct GenWarpScratch {
  uint64_t *cand;        // [cap]
  uint16_t *sel;         // [gpw * nselp]
  uint8_t *board;        // [gpw * SBp]
  const uint8_t *tmpl;   // [SBp] empty padded board (0xFF border), shared by the CTA
};

// Generate the n <= 32 / W requested episodes (request r: env er, predecessor key (rk0, rk1) held by lane r)
// and publish them.  All 32 lanes must call.
__device__ inline void gen_warp_batch(const GenWarpCfg &c, const GenWarpScratch &s, int n, int req_env, uint32_t req_k0,
                                      uint32_t req_k1, int lane) {
  const int N = c.N, W = c.W, S = c.S, SBp = c.SBp;
  const bool uniform_mode = c.kind != RBG_GEN_PRW;
  // ---- keys: two lanes per request walk the split() chain (as prw_kernel phase A0)
  uint32_t sub0, sub1, ks0, ks1, nk0, nk1;
  {
    const int r = lane >> 1;
    const uint32_t cc = lane & 1u;
    uint32_t k0 = __shfl_sync(FULL, req_k0, r < n ? r : 0), k1 = __shfl_sync(FULL, req_k1, r < n ? r : 0);
    uint32_t o0, o1;
    const int extra = (uniform_mode ? 0 : 1) + 1;  // VmapAutoResetWrapper: key, _ = split(state.key); PRWG:52 key, pos_key = split(key)
    for (int sp = 0; sp < extra; ++sp) {
      tf_block(k0, k1, cc, cc + 2u, o0, o1);
      const uint32_t oth = __shfl_xor_sync(FULL, o0, 1);
      k0 = cc ? oth : o0;
      k1 = cc ? o0 : oth;
    }
    tf_block(k0, k1, cc, cc + 2u, o0, o1);
    const uint32_t oth0 = __shfl_xor_sync(FULL, o0, 1), oth1 = __shfl_xor_sync(FULL, o1, 1);
    const uint32_t f0 = cc ? oth0 : o0, f1 = cc ? o0 : oth0;  // split(key)[0]
    const uint32_t g0 = cc ? oth1 : o1, g1 = cc ? o1 : oth1;  // split(key)[1]
    // PRW: State.key = key, k_init = split[0] feeds _shuffle, k_step = split[1] (PRW:73-74)
    // UNIFORM: State.key = split[0], pos_key = split[1] feeds _shuffle (UG:76-82)
    const uint32_t sh0 = uniform_mode ? g0 : f0, sh1 = uniform_mode ? g1 : f1;
    uint32_t q0, q1;
    tf_block(sh0, sh1, cc, cc + 2u, q0, q1);  // _shuffle: key, sub = split(key)
    const uint32_t othq = __shfl_xor_sync(FULL, q1, 1);
    sub0 = cc ? othq : q1;
    sub1 = cc ? q1 : othq;
    ks0 = g0;
    ks1 = g1;
    nk0 = uniform_mode ? f0 : k0;
    nk1 = uniform_mode ? f1 : k1;
  }
  // ---- start cells: one board at a time, the whole warp (G*G/2 threefry blocks each)
  for (int r = 0; r < n; ++r) {
    const uint32_t a0 = __shfl_sync(FULL, sub0, 2 * r), a1 = __shfl_sync(FULL, sub1, 2 * r);
    uint16_t *sel = s.sel + r * c.nselp;
    select_smallest(a0, a1, c.cells, c.nsel, c.thresh, c.cap, s.cand, sel, lane, false);
    if (!uniform_mode) {
      uint32_t *g32 = reinterpret_cast<uint32_t *>(s.board + (size_t)r * SBp);
      const uint32_t *t32 = reinterpret_cast<const uint32_t *>(s.tmpl);
      for (int q = lane; q < (SBp >> 2); q += 32) g32[q] = t32[q];
    }
  }
  __syncwarp();
  // ---- the walk (PRW:78-80 while_loop of _step): W lanes per board, lane = agent
  const int a = lane & (W - 1), grp = lane / W, grp_base = lane & ~(W - 1);
  const uint32_t gm = (W == 32) ? FULL : (((1u << W) - 1u) << grp_base);
  const bool have = grp < n;
  const bool isagent = have && a < N;
  int r = 0, cc = 0;
  if (isagent) {
    uint32_t rr, c2;
    c.divG.divmod((uint32_t)s.sel[grp * c.nselp + a], rr, c2);
    r = (int)rr;
    cc = (int)c2;
  }
  const int start = (r << 8) | cc;
  int fin = start;
  if (uniform_mode) {
    if (isagent) {  // targets are the next N cells of the permutation (UG:82-92)
      uint32_t rr, c2;
      c.divG.divmod((uint32_t)s.sel[grp * c.nselp + N + a], rr, c2);
      fin = (int)((rr << 8) | c2);
    }
  } else {
    uint8_t *g = s.board + (size_t)(have ? grp : 0) * SBp;
    const uint32_t base3 = 3u * a + 1u;
    if (isagent) g[(r + 2) * S + (cc + 2)] = (uint8_t)(base3 + 1u);
    uint32_t k0 = __shfl_sync(FULL, ks0, have ? 2 * grp : 0), k1 = __shfl_sync(FULL, ks1, have ? 2 * grp : 0);
    __syncwarp();
    const bool adv_inline = (N + 2 <= W);
    const uint32_t cx0 = (a < N) ? (uint32_t)a : (uint32_t)(a - N);
    const uint32_t cx1 = (a < N) ? (uint32_t)(a + N) : (uint32_t)(a - N + 2);
    const int f0 = (a < N) ? 2 * a : 0, f1 = (a < N) ? 2 * a + 1 : 0;
    const int s0 = f0 < N ? f0 : f0 - N, s1 = f1 < N ? f1 : f1 - N;
    // The random numbers of a trip do not depend on the board: keys = split(key, N) and key' = split(key)[1]
    // are functions of the loop key alone.  So the first threefry level of trip t+1 (agent keys + key advance)
    // is computed in the same pass as the second level of trip t (the agents' uniform draws): two independent
    // blocks per iteration instead of two dependent ones, which halves the dependent-issue latency of a trip
    // (the generator warp is latency-bound).  The speculative pass after the last trip is simply dropped.
    auto level1 = [&](uint32_t key0, uint32_t key1, uint32_t &ak0, uint32_t &ak1, uint32_t &nx0, uint32_t &nx1) {
      uint32_t o0, o1;
      tf_block(key0, key1, cx0, cx1, o0, o1);  // keys = split(key, N); lanes N, N+1: split(key)[1]
      const uint32_t t00 = __shfl_sync(FULL, o0, s0, W), t01 = __shfl_sync(FULL, o1, s0, W);
      const uint32_t t10 = __shfl_sync(FULL, o0, s1, W), t11 = __shfl_sync(FULL, o1, s1, W);
      ak0 = f0 < N ? t00 : t01;
      ak1 = f1 < N ? t10 : t11;
      if (adv_inline) {
        nx0 = __shfl_sync(FULL, o1, N, W);
        nx1 = __shfl_sync(FULL, o1, N + 1, W);
      } else {
        uint32_t p0, p1;
        tf_block(key0, key1, (uint32_t)(a & 1), (uint32_t)((a & 1) + 2), p0, p1);
        nx0 = __shfl_sync(FULL, p1, 0, W);
        nx1 = __shfl_sync(FULL, p1, 1, W);
      }
    };
    uint32_t ak0, ak1, nx0, nx1;
    level1(k0, k1, ak0, ak1, nx0, nx1);  // trip 0
    bool walking = have;
    while (true) {
      uint8_t *pc = g + (r + 2) * S + (cc + 2);
      uint32_t m4 = 0;
      if (walking && isagent) {  // _available_cells (PRW:293-374): up, down, left, right
        const uint32_t u1 = pc[-S], d1 = pc[S], l1 = pc[-1], r1 = pc[1];
        const bool oul = own_wire(pc[-S - 1], base3), our = own_wire(pc[-S + 1], base3);
        const bool odl = own_wire(pc[S - 1], base3), odr = own_wire(pc[S + 1], base3);
        m4 |= (u1 == 0u && !own_wire(pc[-2 * S], base3) && !oul && !our) ? 1u : 0u;
        m4 |= (d1 == 0u && !own_wire(pc[2 * S], base3) && !odl && !odr) ? 2u : 0u;
        m4 |= (l1 == 0u && !own_wire(pc[-2], base3) && !oul && !odl) ? 4u : 0u;
        m4 |= (r1 == 0u && !own_wire(pc[2], base3) && !our && !odr) ? 8u : 0u;
      }
      const uint32_t any = __ballot_sync(FULL, m4 != 0u);
      if (any == 0u) break;                   // every board of the batch has finished
      walking = walking && (any & gm) != 0u;  // _continue_stepping (PRW:192-203) false: this board is done
      // second level of this trip and first level of the next one: independent instruction streams
      const uint32_t bits = bits_scalar(ak0, ak1);
      uint32_t bk0, bk1, by0, by1;
      level1(nx0, nx1, bk0, bk1, by0, by1);
      // _select_action (PRW:205-230): choice(key, cells, p=mask) in float32
      const float u = bits_to_uniform(bits);
      const int c1 = (int)(m4 & 1u), c2 = c1 + (int)((m4 >> 1) & 1u);
      const int c3 = c2 + (int)((m4 >> 2) & 1u), c4 = c3 + (int)((m4 >> 3) & 1u);
      const float rr_ = __fmul_rn((float)c4, __fsub_rn(1.0f, u));
      const int idx = ((float)c1 < rr_) + ((float)c2 < rr_) + ((float)c3 < rr_);
      const bool move = walking && isagent && c4 > 0;
      const int nr = r + (idx == 0 ? -1 : (idx == 1 ? 1 : 0));
      const int nc = cc + (idx == 2 ? -1 : (idx == 3 ? 1 : 0));
      // _step_agents (PRW:101-145): same destination on the same board -> the highest id moves
      const uint32_t val = move ? (((uint32_t)grp_base << 16) | ((uint32_t)nr << 8) | (uint32_t)nc) : (0x80000000u | (uint32_t)lane);
      const bool win = wins_collision(val, move, a, grp_base, N);
      __syncwarp();  // every lane's neighbour reads are done before any write
      if (win) {
        pc[0] = (uint8_t)base3;
        g[(nr + 2) * S + (nc + 2)] = (uint8_t)(base3 + 1u);
        r = nr;
        cc = nc;
      }
      ak0 = bk0;
      ak1 = bk1;
      nx0 = by0;
      nx1 = by1;
      __syncwarp();
    }
    fin = (r << 8) | cc;
  }
  // ---- publish: the env's next-episode cache entry, seqlock with the tag as version (prw_kernel phase C)
  const long long e = (long long)__shfl_sync(FULL, req_env, have ? grp : 0);
  const uint32_t tk0 = __shfl_sync(FULL, req_k0, have ? grp : 0), tk1 = __shfl_sync(FULL, req_k1, have ? grp : 0);
  const uint32_t pk0 = __shfl_sync(FULL, nk0, have ? 2 * grp : 0), pk1 = __shfl_sync(FULL, nk1, have ? 2 * grp : 0);
  // (nobody reads this entry while it is rewritten: its env consumed it before asking for the next one, and a
  // per-step refill that may still be running under a rollout launch writes the same episode, a board being a pure
  // function of its key; so no invalidation round, and one release store instead of fences.  bar.warp.sync orders the other lanes' pin stores before lane 0's release.)
  if (c.seqlock) {  // (warp-uniform) the tag is the version: invalidate, fence, write, publish
    if (have && a == 0) *reinterpret_cast<volatile unsigned long long *>(c.cache_tag + e) = 0ull;
    __threadfence();
    __syncwarp();
  }
  if (isagent) c.cache_pins[e * N + a] = ((uint32_t)start << 16) | (uint32_t)fin;
  if (have && a == 0) c.cache_key[e] = make_uint2(pk0, pk1);
  if (c.seqlock) __threadfence();
  __syncwarp();
  if (have && a == 0) {
    st_release_u64(c.cache_tag + e, ((unsigned long long)tk1 << 32) | tk0);
    if (c.group_pending) {
      __threadfence();  // the entry is visible before the group's count drops
      atomicSub(c.group_pending + (e >> c.kshift), 1);
    }
  }
}

// The generator warp's life: take requests while the CTA's env warps are running, leave when they are all
// done and the ring is empty.
__device__ inline void gen_warp_loop(const GenWarpCfg &c, const GenWarpScratch &s, GenQueue *q, volatile int *env_warps_done,
                                     int n_env_warps, int lane) {
  const int gpw = 32 / c.W;
  unsigned h = 0;
  int waited = 0;
  for (;;) {
    const bool done = __shfl_sync(FULL, *env_warps_done, 0) >= n_env_warps;  // read BEFORE scanning: a request posted before `done` is then visible
    int n = 0;
    while (n < gpw && q->seq[(h + n) & (GENQ_CAP - 1)] == h + n + 1u) ++n;
    if (n == 0) {
      if (done) break;
      __nanosleep(200);
      continue;
    }
    // A batch costs the same whether it holds one board or 32 / W (the walk is a dependent threefry chain,
    // W lanes per board), and an episode is only needed when the one that has just started ends, tens of
    // steps from now: a partial batch waits a little for company unless an env is actually blocked on it.
    if (n < gpw && !done && !q->urgent && waited < c.patience) {
      __nanosleep(500);
      ++waited;
      continue;
    }
    waited = 0;
    q->urgent = 0;
    int re = 0;
    uint32_t rk0 = 0, rk1 = 0;
    if (lane < n) {
      const unsigned sl = (h + lane) & (GENQ_CAP - 1);
      re = q->env[sl];
      rk0 = q->k0[sl];
      rk1 = q->k1[sl];
    }
    __syncwarp();
    h += n;
    if (lane == 0) q->head = h;  // the slots may be reused
    gen_warp_batch(c, s, n, re, rk0, rk1, lane);
  }
}

}  // namespace rbg
