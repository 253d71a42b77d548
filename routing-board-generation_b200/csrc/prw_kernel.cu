// prw_kernel.cu -- ParallelRandomWalk board generation (and the Uniform
// generator, which shares its start-cell selection) for sm_100a.
//
// Replaces jit(vmap(ParallelRandomWalkBoard.generate_board)) and
// jit(vmap(ParallelRandomWalkGenerator.__call__)):
//   reference parallel_random_walk.py:60-447, parallel_random_walk_generator.py:46-77,
//   uniform_generator.py:70-109 (all under /root/reference/routing_board_generation/).
//
// Design (see DESIGN.md "K1"): the walk is integer-issue bound (threefry2x32),
// not HBM bound, so the kernel is organised to keep lanes busy:
//   phase A0  two threads per board derive the split() keys
//   phase A   one warp per board draws the G*G sort keys of jax.random._shuffle
//             and keeps only the N smallest (threshold filter + rank by
//             counting; exact N-round fallback when the filter misses)
//   phase B   W lanes (W = 8/16/32 >= N) own one board: lane = agent; lanes
//             N and N+1 compute the loop's key advance in the same threefry
//             pass as the per-agent split; boards live in shared memory as
//             uint8 with a 2-cell 0xFF border, so the 12 neighbour reads need
//             no bounds tests; collisions are resolved with __match_any_sync
//             (highest agent id wins, parallel_random_walk.py:104-145); a
//             finished group pulls the next board of the CTA's pool, so
//             divergent walk lengths do not idle lanes
//   phase C   boards are widened uint8 -> int32 and written with 128-bit
//             coalesced stores; in auto-reset mode the Connector observation
//             and action mask of the fresh state are written here too.
#include "connector_device.cuh"
#include "gen_warp.cuh"
#include "rbg_host.h"
#include "select.cuh"

namespace rbg {

struct PrwSmem {
  uint64_t *cand;    // [nwarps * cap]
  uint32_t *kstep;   // [M*2]
  uint32_t *k0;      // [M*2]  State.key
  uint32_t *sub;     // [M*2]  sort-key subkey of _shuffle
  int32_t *stats;    // [M*2]
  int *pool_next;    // [1] (+pad)
  uint16_t *start;   // [M*Np] (r<<8 | c)
  uint16_t *fin;     // [M*Np]
  uint16_t *sel;     // [M*nselp] flat cells of the selection
  uint8_t *tmpl;     // [SBp]
  uint8_t *grid;     // [M*SBp]
};

__host__ __device__ inline size_t align_up(size_t x, size_t a) {
  return (x + a - 1) / a * a;
}

__host__ __device__ inline size_t prw_carve(const PrwParams &p, int nwarps,
                                            uint8_t *base, PrwSmem *s) {
  size_t off = 0;
  auto take = [&](size_t bytes, size_t al) {
    off = align_up(off, al);
    size_t o = off;
    off += bytes;
    return o;
  };
  const int nselp = (p.nsel + 1) & ~1;
  size_t o_cand = take(sizeof(uint64_t) * (size_t)nwarps * p.cap, 16);
  size_t o_kstep = take(sizeof(uint32_t) * 2 * p.M, 8);
  size_t o_k0 = take(sizeof(uint32_t) * 2 * p.M, 8);
  size_t o_sub = take(sizeof(uint32_t) * 2 * p.M, 8);
  size_t o_stats = take(sizeof(int32_t) * 2 * p.M, 8);
  size_t o_pool = take(sizeof(int) * 4, 16);
  size_t o_start = take(sizeof(uint16_t) * (size_t)p.M * p.Np, 4);
  size_t o_fin = take(sizeof(uint16_t) * (size_t)p.M * p.Np, 4);
  size_t o_sel = take(sizeof(uint16_t) * (size_t)p.M * nselp, 4);
  size_t o_tmpl = take((size_t)p.SBp, 16);
  size_t o_grid = take((size_t)p.M * p.SBp, 16);
  if (s) {
    s->cand = reinterpret_cast<uint64_t *>(base + o_cand);
    s->kstep = reinterpret_cast<uint32_t *>(base + o_kstep);
    s->k0 = reinterpret_cast<uint32_t *>(base + o_k0);
    s->sub = reinterpret_cast<uint32_t *>(base + o_sub);
    s->stats = reinterpret_cast<int32_t *>(base + o_stats);
    s->pool_next = reinterpret_cast<int *>(base + o_pool);
    s->start = reinterpret_cast<uint16_t *>(base + o_start);
    s->fin = reinterpret_cast<uint16_t *>(base + o_fin);
    s->sel = reinterpret_cast<uint16_t *>(base + o_sel);
    s->tmpl = base + o_tmpl;
    s->grid = base + o_grid;
  }
  return align_up(off, 16);
}

__device__ __forceinline__ void prw_body(const PrwParams &p, uint8_t *smem_raw) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int nthreads = blockDim.x, nwarps = nthreads >> 5;
  const long long total = p.list ? (long long)(*p.list_count) : p.B;
  // CTAs stride over pools of M boards (list launches are sized for the worst case
  // but usually hold a few percent of the batch)
  for (long long base = (long long)blockIdx.x * p.M; base < total; base += (long long)gridDim.x * p.M) {
  const int Mc = (int)((total - base) < (long long)p.M ? (total - base) : (long long)p.M);

  PrwSmem s;
  prw_carve(p, nwarps, smem_raw, &s);
  const int G = p.G, N = p.N, S = p.S, SBp = p.SBp, cells = p.cells, Np = p.Np;
  const int nsel = p.nsel, nselp = (nsel + 1) & ~1;
  const bool uniform_mode = (p.mode == PRW_MODE_UNIFORM);

  // ---- phase 0: empty-board template (0xFF border, 0 interior), pool counter
  for (int i = tid; i < SBp; i += nthreads) {
    const int r = i / S, c = i - r * S;
    const bool interior = r >= 2 && r < G + 2 && c >= 2 && c < G + 2;
    s.tmpl[i] = interior ? 0 : 0xFF;
  }
  const int W = p.W, gpw = 32 / W;
  if (tid == 0) *s.pool_next = nwarps * gpw;

  // ---- phase A0: key derivation, two threads per board
  for (int m0 = 0; m0 < Mc; m0 += nthreads >> 1) {
    const int m = m0 + (tid >> 1);
    const uint32_t c = tid & 1u;
    const int mm = m < Mc ? m : Mc - 1;
    const long long e = p.list ? (long long)p.list[base + mm] : base + mm;
    const long long ki = p.keys_compact ? base + mm : e;
    uint32_t k0 = p.keys[2 * ki], k1 = p.keys[2 * ki + 1];
    uint32_t o0, o1;
    for (int sp = 0; sp < p.extra_split; ++sp) {  // key = split(key)[0]
      tf_block(k0, k1, c, c + 2u, o0, o1);
      const uint32_t oth = __shfl_xor_sync(FULL, o0, 1);
      k0 = c ? oth : o0;
      k1 = c ? o0 : oth;
    }
    tf_block(k0, k1, c, c + 2u, o0, o1);
    const uint32_t oth0 = __shfl_xor_sync(FULL, o0, 1);
    const uint32_t oth1 = __shfl_xor_sync(FULL, o1, 1);
    const uint32_t f0 = c ? oth0 : o0, f1 = c ? o0 : oth0;  // split(key)[0]
    const uint32_t g0 = c ? oth1 : o1, g1 = c ? o1 : oth1;  // split(key)[1]
    // PRW:   k_init = split[0] feeds _shuffle, k_step = split[1] (PRW:73-74)
    // UNIF:  State.key = split[0], pos_key = split[1] feeds _shuffle (UG:76-82)
    const uint32_t sh0 = uniform_mode ? g0 : f0, sh1 = uniform_mode ? g1 : f1;
    uint32_t q0, q1;
    tf_block(sh0, sh1, c, c + 2u, q0, q1);  // _shuffle: key, sub = split(key)
    const uint32_t othq = __shfl_xor_sync(FULL, q1, 1);
    if (m < Mc && c == 0) {
      s.sub[2 * m] = q1;
      s.sub[2 * m + 1] = othq;
      s.kstep[2 * m] = g0;
      s.kstep[2 * m + 1] = g1;
      s.k0[2 * m] = uniform_mode ? f0 : k0;
      s.k0[2 * m + 1] = uniform_mode ? f1 : k1;
    }
  }
  __syncthreads();

  // ---- phase A: selection + board set-up, one warp per board
  for (int m = warp; m < Mc; m += nwarps) {
    uint16_t *sel = s.sel + m * nselp;
    select_smallest(s.sub[2 * m], s.sub[2 * m + 1], cells, nsel, p.thresh, p.cap,
                    s.cand + (size_t)warp * p.cap, sel, lane, (p.debug & 1) != 0);
    uint32_t *g32 = reinterpret_cast<uint32_t *>(s.grid + (size_t)m * SBp);
    const uint32_t *t32 = reinterpret_cast<const uint32_t *>(s.tmpl);
    for (int q = lane; q < (SBp >> 2); q += 32) g32[q] = t32[q];
    __syncwarp();
    uint8_t *g = s.grid + (size_t)m * SBp;
    if (lane < N) {
      uint32_t r, c;
      p.divG.divmod((uint32_t)sel[lane], r, c);
      s.start[m * Np + lane] = (uint16_t)((r << 8) | c);
      g[(r + 2) * S + (c + 2)] = (uint8_t)(3 * lane + POSITION);
    }
    if (uniform_mode) {
      __syncwarp();
      if (lane < N) {  // targets after heads (UG:93-94); cells are distinct anyway
        uint32_t r, c;
        p.divG.divmod((uint32_t)sel[N + lane], r, c);
        s.fin[m * Np + lane] = (uint16_t)((r << 8) | c);
        g[(r + 2) * S + (c + 2)] = (uint8_t)(3 * lane + TARGET);
      }
      if (lane == 0) {
        s.stats[2 * m] = 0;
        s.stats[2 * m + 1] = 0;
      }
    }
  }
  __syncthreads();

  // ---- phase B: the walk (PRW:78-80 while_loop of _step), W lanes per board
  if (!uniform_mode) {
    const int a = lane & (W - 1);
    const int grp_base = lane & ~(W - 1);
    const uint32_t gm = (W == 32) ? FULL : (((1u << W) - 1u) << grp_base);
    const int gid = warp * gpw + (lane / W);
    int cur = gid < Mc ? gid : -1;
    uint32_t k0 = 0, k1 = 0;
    int r = 0, c = 0, trips = 0, colls = 0;
    auto load_board = [&]() {
      if (cur >= 0) {
        k0 = s.kstep[2 * cur];
        k1 = s.kstep[2 * cur + 1];
        if (a < N) {
          const uint32_t rc = s.start[cur * Np + a];
          r = (int)(rc >> 8);
          c = (int)(rc & 255u);
        }
        trips = 0;
        colls = 0;
      }
    };
    load_board();
    const uint32_t base3 = 3u * a + 1u;
    const bool adv_inline = (N + 2 <= W);
    // counters of this lane's threefry block in the per-trip pass:
    // agents: block a of split(key, N) = (a, a+N); lanes N, N+1: the two
    // blocks of split(key) whose o1 words are the next loop key (PRW:98-99)
    const uint32_t cx0 = (a < N) ? (uint32_t)a : (uint32_t)(a - N);
    const uint32_t cx1 = (a < N) ? (uint32_t)(a + N) : (uint32_t)(a - N + 2);
    const int f0 = (a < N) ? 2 * a : 0, f1 = (a < N) ? 2 * a + 1 : 0;
    const int s0 = f0 < N ? f0 : f0 - N, s1 = f1 < N ? f1 : f1 - N;

    while (true) {
      const bool active = cur >= 0;
      if (!__any_sync(FULL, active)) break;
      const bool isagent = active && a < N;
      uint8_t *g = s.grid + (size_t)(active ? cur : 0) * SBp;
      uint8_t *pc = g + (r + 2) * S + (c + 2);
      // _available_cells (PRW:293-374): candidate order up, down, left, right;
      // free and touching the own wire only through the head itself.
      uint32_t m4 = 0;
      if (isagent) {
        const uint32_t u1 = pc[-S], d1 = pc[S], l1 = pc[-1], r1 = pc[1];
        const uint32_t uu = pc[-2 * S], dd = pc[2 * S], ll = pc[-2], rr = pc[2];
        const uint32_t ul = pc[-S - 1], ur = pc[-S + 1], dl = pc[S - 1], dr = pc[S + 1];
        const bool oul = own_wire(ul, base3), our = own_wire(ur, base3);
        const bool odl = own_wire(dl, base3), odr = own_wire(dr, base3);
        m4 |= (u1 == 0u && !own_wire(uu, base3) && !oul && !our) ? 1u : 0u;
        m4 |= (d1 == 0u && !own_wire(dd, base3) && !odl && !odr) ? 2u : 0u;
        m4 |= (l1 == 0u && !own_wire(ll, base3) && !oul && !odl) ? 4u : 0u;
        m4 |= (r1 == 0u && !own_wire(rr, base3) && !our && !odr) ? 8u : 0u;
      }
      const uint32_t grp_any = __ballot_sync(FULL, m4 != 0u) & gm;
      const bool dotrip = active && grp_any != 0u;    // _continue_stepping true
      const bool dofinish = active && grp_any == 0u;  // loop ends for this board

      if (__any_sync(FULL, dotrip)) {
        // pass 1: keys = split(key, N) (+ key advance on lanes N, N+1)
        uint32_t o0, o1;
        tf_block(k0, k1, cx0, cx1, o0, o1);
        const uint32_t t00 = __shfl_sync(FULL, o0, s0, W), t01 = __shfl_sync(FULL, o1, s0, W);
        const uint32_t t10 = __shfl_sync(FULL, o0, s1, W), t11 = __shfl_sync(FULL, o1, s1, W);
        const uint32_t ak0 = f0 < N ? t00 : t01, ak1 = f1 < N ? t10 : t11;
        uint32_t nk0, nk1;
        if (adv_inline) {
          nk0 = __shfl_sync(FULL, o1, N, W);
          nk1 = __shfl_sync(FULL, o1, N + 1, W);
        } else {
          uint32_t q0, q1;
          tf_block(k0, k1, (uint32_t)(a & 1), (uint32_t)((a & 1) + 2), q0, q1);
          nk0 = __shfl_sync(FULL, q1, 0, W);
          nk1 = __shfl_sync(FULL, q1, 1, W);
        }
        // pass 2: _select_action (PRW:205-230): choice(key, cells, p=mask)
        const uint32_t bits = bits_scalar(ak0, ak1);
        const float u = bits_to_uniform(bits);
        const int c1 = (int)(m4 & 1u), c2 = c1 + (int)((m4 >> 1) & 1u);
        const int c3 = c2 + (int)((m4 >> 2) & 1u), c4 = c3 + (int)((m4 >> 3) & 1u);
        const float rr_ = __fmul_rn((float)c4, __fsub_rn(1.0f, u));
        const int idx = ((float)c1 < rr_) + ((float)c2 < rr_) + ((float)c3 < rr_);
        const bool move = dotrip && isagent && c4 > 0;
        const int nr = r + (idx == 0 ? -1 : (idx == 1 ? 1 : 0));
        const int nc = c + (idx == 2 ? -1 : (idx == 3 ? 1 : 0));
        // _step_agents (PRW:101-145): same destination -> highest id moves
        const uint32_t val = move ? (((uint32_t)grp_base << 16) | ((uint32_t)nr << 8) | (uint32_t)nc)
                                  : (0x80000000u | (uint32_t)lane);
        const uint32_t mm = __match_any_sync(FULL, val);
        const bool win = move && (lane == 31 - __clz(mm));
        colls += __popc(__ballot_sync(FULL, move && !win) & gm);
        __syncwarp();  // every lane's neighbour reads are done before any write
        if (win) {
          pc[0] = (uint8_t)(base3);                              // old head -> PATH
          g[(nr + 2) * S + (nc + 2)] = (uint8_t)(base3 + 1u);    // POSITION
          r = nr;
          c = nc;
        }
        if (dotrip) {
          k0 = nk0;
          k1 = nk1;
          ++trips;
        }
      }
      __syncwarp();
      const uint32_t finmask = __ballot_sync(FULL, dofinish);
      if (dofinish) {
        if (isagent) s.fin[cur * Np + a] = (uint16_t)((r << 8) | c);
        if (p.mode == PRW_MODE_STATE) {  // training grid = pins only (PRWG:54-64)
          uint32_t *g32 = reinterpret_cast<uint32_t *>(g);
          const uint32_t *t32 = reinterpret_cast<const uint32_t *>(s.tmpl);
          for (int q = a; q < (SBp >> 2); q += W) g32[q] = t32[q];
        }
        __syncwarp(finmask);
        // heads first, then targets (PRW:435-447): targets win on zero-length wires
        if (isagent) {
          const uint32_t rc0 = s.start[cur * Np + a];
          g[((rc0 >> 8) + 2) * S + ((rc0 & 255u) + 2)] = (uint8_t)(base3 + 1u);
        }
        __syncwarp(finmask);
        if (isagent) g[(r + 2) * S + (c + 2)] = (uint8_t)(base3 + 2u);
        if (a == 0) {
          s.stats[2 * cur] = trips;
          s.stats[2 * cur + 1] = colls;
        }
        int nxt = 0;
        if (a == 0) nxt = atomicAdd(s.pool_next, 1);
        nxt = __shfl_sync(finmask, nxt, 0, W);
        cur = nxt < Mc ? nxt : -1;
        load_board();
      }
      __syncwarp();
    }
  }
  __syncthreads();

  // ---- phase C: outputs, one warp per board
  const bool vec = (cells & 3) == 0;
  for (int m = warp; m < Mc; m += nwarps) {
    const long long e = p.list ? (long long)p.list[base + m] : base + m;
    const uint8_t *g = s.grid + (size_t)m * SBp;
    if (p.to_cache) {
      // auto-reset cache entry: (start, target) pins + State.key of this episode, published under the key
      // of the episode it succeeds.  Seqlock with the tag as version: invalidate, fence, write, fence,
      // publish (readers re-check the tag after their loads: connector_kernel.cu env_warp_kernel)
      if (lane == 0) *reinterpret_cast<volatile unsigned long long *>(p.cache_tag + e) = 0ull;
      __threadfence();
      __syncwarp();
      if (lane < N) {
        const uint32_t st_ = s.start[m * Np + lane], fi = s.fin[m * Np + lane];
        p.cache_pins[e * N + lane] = (st_ << 16) | fi;
      }
      if (lane == 0) p.cache_key[e] = make_uint2(s.k0[2 * m], s.k0[2 * m + 1]);
      __threadfence();
      __syncwarp();
      if (lane == 0) {
        const long long ki = p.keys_compact ? base + m : e;
        const unsigned long long tag = ((unsigned long long)p.keys[2 * ki + 1] << 32) | p.keys[2 * ki];
        *reinterpret_cast<volatile unsigned long long *>(p.cache_tag + e) = tag;
      }
      continue;
    }
    int32_t *gout = (p.mode == PRW_MODE_BOARD ? p.solved : p.st.grid) + e * cells;
    if (vec) {
      int4 *o = reinterpret_cast<int4 *>(gout);
      for (int q = lane; q < (cells >> 2); q += 32) {
        uint32_t r, c;
        p.divG.divmod((uint32_t)(4 * q), r, c);
        int v[4];
#pragma unroll
        for (int t = 0; t < 4; ++t) {
          v[t] = g[(r + 2) * S + (c + 2)];
          if (++c == (uint32_t)G) {
            c = 0;
            ++r;
          }
        }
        o[q] = make_int4(v[0], v[1], v[2], v[3]);
      }
    } else {
      for (int i = lane; i < cells; i += 32) {
        uint32_t r, c;
        p.divG.divmod((uint32_t)i, r, c);
        gout[i] = g[(r + 2) * S + (c + 2)];
      }
    }
    if (lane < N) {
      const uint32_t st_ = s.start[m * Np + lane], fi = s.fin[m * Np + lane];
      const int sr = (int)(st_ >> 8), sc = (int)(st_ & 255u);
      const int fr = (int)(fi >> 8), fc = (int)(fi & 255u);
      if (p.mode == PRW_MODE_BOARD) {  // heads = start.T, targets = position.T (PRW:83-84)
        p.heads[e * 2 * N + lane] = sr;
        p.heads[e * 2 * N + N + lane] = sc;
        p.targets[e * 2 * N + lane] = fr;
        p.targets[e * 2 * N + N + lane] = fc;
      } else {  // Agent pytree (PRWG:68-73): position = start
        p.st.agent_id[e * N + lane] = lane;
        reinterpret_cast<int2 *>(p.st.start)[e * N + lane] = make_int2(sr, sc);
        reinterpret_cast<int2 *>(p.st.target)[e * N + lane] = make_int2(fr, fc);
        reinterpret_cast<int2 *>(p.st.position)[e * N + lane] = make_int2(sr, sc);
      }
      if (p.observe) {
        SmemGrid sg{g, S, 2, G};
        const uint32_t mk = move_mask(sg, sr, sc, lane, sr == fr && sc == fc);
        store_mask5(p.ts.action_mask + (e * N + lane) * 5, mk);
      }
    }
    if (lane == 0) {
      if (p.mode != PRW_MODE_BOARD) {
        p.st.step_count[e] = 0;
        p.st.key[2 * e] = s.k0[2 * m];
        p.st.key[2 * e + 1] = s.k0[2 * m + 1];
      }
      if (p.stats) {
        p.stats[2 * e] = s.stats[2 * m];
        p.stats[2 * e + 1] = s.stats[2 * m + 1];
      }
      if (p.observe) p.ts.obs_step_count[e] = 0;
    }
    if (p.observe) {
      SmemGrid sg{g, S, 2, G};
      warp_write_obs(sg, N, p.divG, p.ts.obs_grid + (size_t)e * N * cells, lane);
    }
  }
  __syncthreads();  // shared memory is reused by the next pool
  }
  // list launches recycle their counter: the last CTA to finish clears it (every CTA
  // has read it by then), so the host needs no memset between steps
  if (p.list_ticket) {
    __syncthreads();
    if (tid == 0) {
      __threadfence();
      if (atomicAdd(p.list_ticket, 1) == (int)gridDim.x - 1) {
        *const_cast<int32_t *>(p.list_count) = 0;
        *p.list_ticket = 0;
        __threadfence();
      }
    }
  }
}

__global__ void __launch_bounds__(256) prw_kernel(const PrwParams p) {
  extern __shared__ __align__(16) uint8_t smem_raw[];
  if (p.trigger_dependents) asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  prw_body(p, smem_raw);
}

// The two list launches of a per-step auto-reset in one: `a` regenerates the envs whose next episode was not in
// the cache (State + observation, needed by the next step: prw_body), then the cache entries consumed in this step
// are refilled (needed many steps from now).  Between the two every CTA says launch_dependents, so that the next env
// kernel (launched with programmatic stream serialization) starts once all of `a` is done, under the refill.
// The refill is latency-bound (a few thousand boards, one walk each), so it runs on the generator-warp code of the
// fused rollout (gen_warp.cuh: both threefry levels of a trip in one pass, shuffles instead of MATCH), a warp taking
// 32 / W list entries at a time.
struct RefillParams {
  const int32_t *list;     // env ids
  const uint32_t *keys;    // [slot, 2] State.key of the episode that has just started (the entry's tag)
  int32_t *list_count;     // device count; cleared by the last CTA together with the ticket
  int32_t *list_ticket;
  int gcand_bytes, gsel_bytes, gscr_stride, tmpl_off, gscr_off;
};

__global__ void __launch_bounds__(64) prw_pair_kernel(const PrwParams a, const RefillParams rf, const GenWarpCfg gc) {
  extern __shared__ __align__(16) uint8_t smem_raw[];
  prw_body(a, smem_raw);
  __threadfence();
  __syncthreads();
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarps = blockDim.x >> 5;
  uint8_t *tmpl = smem_raw + rf.tmpl_off;
  for (int i = tid; i < gc.SBp; i += blockDim.x) {
    const int r = i / gc.S, c = i - r * gc.S;
    tmpl[i] = (r >= 2 && r < gc.G + 2 && c >= 2 && c < gc.G + 2) ? 0 : 0xFF;
  }
  __syncthreads();
  uint8_t *gb = smem_raw + rf.gscr_off + (size_t)warp * rf.gscr_stride;
  GenWarpScratch gs;
  gs.cand = reinterpret_cast<uint64_t *>(gb);
  gs.sel = reinterpret_cast<uint16_t *>(gb + rf.gcand_bytes);
  gs.board = gb + rf.gcand_bytes + rf.gsel_bytes;
  gs.tmpl = tmpl;
  const int total = *rf.list_count, gpw = 32 / gc.W;
  for (int base = (blockIdx.x * nwarps + warp) * gpw; base < total; base += gridDim.x * nwarps * gpw) {
    const int n = total - base < gpw ? total - base : gpw;
    int re = 0;
    uint32_t rk0 = 0, rk1 = 0;
    if (lane < n) {
      re = rf.list[base + lane];
      rk0 = rf.keys[2 * (base + lane)];
      rk1 = rf.keys[2 * (base + lane) + 1];
    }
    gen_warp_batch(gc, gs, n, re, rk0, rk1, lane);
  }
  // the last CTA to finish recycles the list counter (every CTA has read it by then)
  __syncthreads();
  if (tid == 0) {
    __threadfence();
    if (atomicAdd(rf.list_ticket, 1) == (int)gridDim.x - 1) {
      *rf.list_count = 0;
      *rf.list_ticket = 0;
      __threadfence();
    }
  }
}

// ---------------------------------------------------------------- host side
// derived fields of PrwParams + launch shape
static int prw_prepare(PrwParams &p, int64_t max_boards, int *threads_out, size_t *smem_out, int64_t *ctas_out) {
  const int G = p.G, N = p.N;
  p.cells = G * G;
  p.S = G + 4;
  p.SBp = (int)align_up((size_t)p.S * p.S, 16);
  p.Np = (N + 1) & ~1;
  p.nsel = (p.mode == PRW_MODE_UNIFORM) ? 2 * N : N;
  p.W = N <= 8 ? 8 : (N <= 16 ? 16 : 32);
  p.divG = FastDiv::make((uint32_t)G);
  p.cap = 4 * p.nsel + 32;
  {
    const double lam = 2.0 * p.nsel + 16.0;
    const double frac = lam / (double)p.cells;
    p.thresh = frac >= 1.0 ? 0xffffffffu : (uint32_t)(frac * 4294967296.0);
  }
  // boards per CTA / threads per CTA: big pools for bulk generation (lane
  // refill balances the divergent walk lengths), small CTAs for short lists
  int threads = 256, M = 64;
  const int gpw = 32 / p.W;
  const int64_t sms = device_sm_count();
  if (max_boards <= sms * 64) {
    threads = 64;
    M = 2 * gpw * 2;  // one board per group + one refill
  }
  if (p.list) {  // per-step lists: a few percent of the batch, latency matters
    threads = 64;
    M = 2 * gpw;
  }
  // keep shared memory per CTA moderate so several CTAs share an SM
  for (;;) {
    p.M = M;
    size_t bytes = prw_carve(p, threads / 32, nullptr, nullptr);
    if (bytes <= 48 * 1024 || M <= (threads / 32) * gpw) break;
    M >>= 1;
  }
  p.M = M;
  const size_t smem = prw_carve(p, threads / 32, nullptr, nullptr);
  if (smem > 200 * 1024) return set_error(RBG_EINVAL, "prw_kernel: %zu bytes of shared memory per CTA", smem);
  int64_t ctas = (max_boards + M - 1) / M;
  if (p.list && ctas > sms * (p.to_cache ? 4 : 2)) ctas = sms * (p.to_cache ? 4 : 2);  // per-step lists hold a few percent of the batch and the kernel strides over them
  *threads_out = threads;
  *smem_out = smem;
  *ctas_out = ctas;
  return RBG_OK;
}

int launch_prw(PrwParams p, int64_t max_boards, cudaStream_t stream) {
  int threads = 0, rc;
  size_t smem = 0;
  int64_t ctas = 0;
  if ((rc = prw_prepare(p, max_boards, &threads, &smem, &ctas))) return rc;
  if (ctas <= 0) return RBG_OK;
  if (smem > 48 * 1024) {
    cudaError_t e = cudaFuncSetAttribute(prw_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return set_cuda_error(e, "cudaFuncSetAttribute(prw_kernel)");
  }
  {
    LaunchScope scope(RBG_K_PRW, stream);
    prw_kernel<<<(unsigned)ctas, threads, smem, stream>>>(p);
  }
  return check_launch("prw_kernel");
}

// per-step auto-reset: synchronous list `a` and the cache refill `b` (both short lists of the same batch) in one launch
int launch_prw_pair(PrwParams a, PrwParams b, int64_t max_boards, cudaStream_t stream) {
  int ta = 0, rc;
  size_t sa = 0;
  int64_t ca = 0;
  if ((rc = prw_prepare(a, max_boards, &ta, &sa, &ca))) return rc;
  if (ta != 64 || !a.list || !b.list || !b.to_cache || !b.keys_compact) return set_error(RBG_EINVAL, "prw_pair_kernel: a 64-thread list launch and a compact-key cache refill");
  auto up16 = [](size_t x) { return (x + 15) & ~(size_t)15; };
  RefillParams rf;
  memset(&rf, 0, sizeof(rf));
  rf.list = b.list;
  rf.keys = b.keys;
  rf.list_count = const_cast<int32_t *>(b.list_count);
  rf.list_ticket = b.list_ticket;
  GenWarpCfg gc = gen_warp_cfg(b.mode == PRW_MODE_UNIFORM ? RBG_GEN_UNIFORM : RBG_GEN_PRW, b.G, b.N, &rf.gcand_bytes, &rf.gsel_bytes, &rf.gscr_stride);
  gc.cache_tag = b.cache_tag;
  gc.cache_key = b.cache_key;
  gc.cache_pins = b.cache_pins;
  gc.seqlock = 1;  // the next env kernel runs under this refill
  const int gpw = 32 / gc.W;
  rf.tmpl_off = 0;
  rf.gscr_off = (int)up16((size_t)gc.SBp);
  const size_t sb = (size_t)rf.gscr_off + 2 * (size_t)rf.gscr_stride;  // the refill reuses the shared memory of `a`
  const size_t smem = sa > sb ? sa : sb;
  if (smem > 200 * 1024) return set_error(RBG_EINVAL, "prw_pair_kernel: %zu bytes of shared memory per CTA", smem);
  const int sms = device_sm_count();
  int64_t ctas = (max_boards + 2 * gpw - 1) / (2 * gpw);
  if (ctas > (int64_t)sms * 4) ctas = (int64_t)sms * 4;  // per-step lists hold a few percent of the batch; both halves stride
  if (ca > ctas) ctas = ca;
  if (ctas <= 0) return RBG_OK;
  if (smem > 48 * 1024) {
    cudaError_t e = cudaFuncSetAttribute(prw_pair_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return set_cuda_error(e, "cudaFuncSetAttribute(prw_pair_kernel)");
  }
  {
    LaunchScope scope(RBG_K_PRW, stream);
    prw_pair_kernel<<<(unsigned)ctas, 64, smem, stream>>>(a, rf, gc);
  }
  return check_launch("prw_pair_kernel");
}

}  // namespace rbg
