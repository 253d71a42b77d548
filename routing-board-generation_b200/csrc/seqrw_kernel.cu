// seqrw_kernel.cu -- SequentialRandomWalkBoard / SequentialRandomWalkGenerator for sm_100a (SURVEY §8 f4).
//
// Replaces jit(vmap(SequentialRandomWalkBoard.generate)) / generate_starts_ends and
// jit(vmap(SequentialRandomWalkGenerator.__call__)):
//   reference board_generation_methods/jax_implementation/board_generation/sequential_random_walk.py:23-431 (SRW),
//   rl_training/online_generators/sequential_random_walk_generator.py:19-62 (both under
//   /root/reference/routing_board_generation/).
//
// What the reference computes, per board: up to rows + cols attempts, ALL from the same key, with a maximum
// walk length of rows + cols - i in attempt i (SRW:324-392); an attempt places the wires one after the other
// (SRW:290-322): a start cell drawn among the empty cells (pick_start, :34-83), then up to max_length steps,
// each to one of the <= 4 adjacent cells that are free and touch the wire only through the cell it stands on
// (:115-191), until none is left; the attempt succeeds when every wire could start and moved at least once.
// Every draw is jax.random.choice(p in {0,1}, replace=False) = a float32 Gumbel top-k, which for such p is
// "the candidate whose uniform has the largest 23-bit mantissa, lowest index on ties" for any strictly monotone
// float32 log (DESIGN.md §8 f4; checked on every draw of the fixtures by tests/tools/make_seqrw_fixtures.py): integer work.
//
// Bound: integer issue (threefry2x32), like prw_kernel.  The work per wire is G*G/2 blocks for the start cell
// and, per step, one split (2 blocks) + the 4 words of the step's draw that can matter (the reference draws
// G + 1 words, one per entry of its padded candidate list; only entries 0..3 can have p = 1).
//
// Organisation: 8 lanes own a board (4 boards per warp), the board in shared memory as uint8 with a 2-cell 0xFF
// border (no bounds tests).  The lanes of a warp run ONE loop whose body is one threefry block per lane plus the
// bookkeeping of whatever phase each board is in, so boards in different phases (different wires, different
// attempts) share every hash pass:
//   SPLIT_WIRE   lanes 0,1: split(key)           -> subkey b             (SRW:307)
//   SPLIT_START  lanes 0,1: split(b)             -> chain key c, draw key d   (:51)
//   PICK         8 blocks of random_bits(d, (G*G,)) per pass, every lane keeps its best empty cell; reduce   (:57-71)
//   SPLIT_WALK   lanes 0,1: split(c)             -> c', step key s        (:204, first step)
//   WALK         lanes 2..5: the step's 4 words under s and the availability of their direction;
//                lanes 0,1: split(c') for the NEXT step in the same pass (the chain does not depend on the
//                board); ballot, pick, move                              (:193-228, :230-288)
// The body is written so that all 32 lanes execute the same instructions whatever phase their board is in (operands
// are selected, board reads are unconditional on a safe cell); only the once-per-wire events (start cell found, walk
// over) and the once-per-board events (new board, failed attempt, output) branch, behind warp votes.  The first
// version branched on the phase and spent 70 % of its instructions in bookkeeping executed one group at a time
// (profiles/r02g_seqrw_full.csv: 13.6 k warp-instructions per 10x10/5 board).
// A failed attempt is abandoned at once (its board can only be discarded, :355-366), the attempts that would repeat it
// exactly are skipped, and the next one resumes where it first differs: all attempts start from the same key, so an
// attempt differs from the previous one only from the first wire whose walk the smaller max_length truncates; the wires
// before it stay on the board and that wire restarts its walk from the same start cell.  Groups take boards from a
// global queue.  The finished board goes to a byte scratch and through se_finish_kernel's outputs (board /
// first POSITION and TARGET cell per wire / State + observation), which SeedExtension shares.
#include "connector_device.cuh"
#include "rbg_host.h"

namespace rbg {

constexpr int SQ_THREADS = 128;
// lanes per board: 8 (4 boards per warp) or 6 (5 boards per warp, lanes 30 and 31 idle: the walk pass uses exactly 2 split
// lanes + 4 draw lanes, the start-cell scan takes ceil(G*G/2 / 6) passes instead of ceil(G*G/2 / 8))
template <int SQ_W>
struct SqShape {
  static constexpr int GPW = 32 / SQ_W;                      // groups per warp
  static constexpr int GROUPS = (SQ_THREADS / 32) * GPW;     // boards in flight per CTA
};

enum : int { SQ_SPLIT_WIRE = 0, SQ_SPLIT_START = 1, SQ_PICK = 2, SQ_SPLIT_WALK = 3, SQ_WALK = 4, SQ_IDLE = 5, SQ_DONE = 6 };

template <int SQ_W>
__global__ void __launch_bounds__(SQ_THREADS) seqrw_walk_kernel(const SeqRwParams p, uint8_t *__restrict__ out_board, uint32_t *__restrict__ out_gkey,
                                                                const int CB, int *__restrict__ queue, const FastDiv divG) {
  extern __shared__ __align__(16) uint8_t smem_raw[];
  constexpr int GPW = SqShape<SQ_W>::GPW, SQ_GROUPS = SqShape<SQ_W>::GROUPS;
  const int tid = threadIdx.x, lane = tid & 31, l = lane % SQ_W, gbase = lane - l;
  const bool spare = lane >= GPW * SQ_W;  // SQ_W = 6: lanes 30, 31 own no board (they run along, DONE from the start)
  constexpr unsigned spare_mask = GPW * SQ_W < 32 ? (FULL << ((GPW * SQ_W) & 31)) : 0u;
  const unsigned gmask = spare ? spare_mask : (((1u << SQ_W) - 1u) << gbase);
  const int G = p.G, N = p.N, S = G + 4, cells = G * G;
  const int SB = (S * S + 15) & ~15;
  uint8_t *tmpl = smem_raw + (size_t)SQ_GROUPS * SB;  // the empty board: 0xFF border, 0 interior
  const int grp = spare ? 0 : (tid >> 5) * GPW + lane / SQ_W;
  uint8_t *board = spare ? tmpl : smem_raw + (size_t)grp * SB;
  // per placed wire of the current attempt: chain key at the start of its walk (2 words), start cell, steps walked
  uint32_t *winfo = reinterpret_cast<uint32_t *>(smem_raw + (size_t)(SQ_GROUPS + 1) * SB) + (size_t)grp * 4 * RBG_MAX_N;
  for (int i = tid; i < SB; i += SQ_THREADS) {
    const int r = i / S, c = i - r * S;
    tmpl[i] = (r >= 2 && r < G + 2 && c >= 2 && c < G + 2) ? 0 : 0xFF;
  }
  __syncthreads();
  const long long total = p.list ? (long long)(*p.list_count) : p.B;
  const int n1 = cells, h1 = (cells + 1) >> 1;  // pick_start: random_bits(d, (G*G,)), odd sizes padded with a zero counter
  const int n2 = G + 1, h2 = (n2 + 1) >> 1;     // one_step:   random_bits(s, (G+1,))
  const int P = (h1 + SQ_W - 1) / SQ_W;
  const int safe = 2 * S + 2;  // an interior cell: what the unconditional board reads fall back to

  // per-lane constants of the walk pass: lanes 2..5 draw word k = l - 2 of random_bits(s, (G+1,)) (o0 of block k, or o1 of
  // block k - h2) and test direction k of [up, down, left, right]
  const bool draw_lane = (unsigned)(l - 2) < 4u;
  const int kdir = (l - 2) & 3;
  const bool k_low = kdir < h2;
  const uint32_t wx0 = (uint32_t)(k_low ? kdir : kdir - h2);
  const uint32_t wx1 = ((int)wx0 + h2 < n2) ? wx0 + (uint32_t)h2 : 0u;
  const int dirk = kdir == 0 ? -S : kdir == 1 ? S : kdir == 2 ? -1 : 1;
  const uint32_t sx0 = (uint32_t)(l & 1), sx1 = sx0 + 2u;  // split(): blocks (0,2), (1,3)

  int phase = spare ? SQ_DONE : SQ_IDLE;
  long long m = -1, e = -1;
  uint32_t K0 = 0, K1 = 0;    // the board's key (every attempt starts from it)
  uint32_t h0 = 0, h1k = 0;   // the key the next pass hashes: the wire's key, its subkey, the draw key of the start, the chain key
  uint32_t c0 = 0, c1 = 0;    // chain key of the walk (committed) = the tuple's key between wires
  uint32_t s0 = 0, s1 = 0;    // the step's draw key
  int w = 0, L = 0, t = 0, filled = 0, cur = safe, startc = safe, j = 0, steps = 0, attempt = 0;
  int max_t = 0;  // longest walk among the wires placed so far in this attempt
  unsigned long long best = 0;  // PICK: (mantissa << 32) | (0xffff - cell) of the lane's best empty cell, 0 = none

  for (;;) {
    __syncwarp();
    if (__all_sync(FULL, phase == SQ_DONE)) break;
    if (__any_sync(FULL, phase == SQ_IDLE)) {
      bool fresh = false;
      if (phase == SQ_IDLE) {
        int nm = 0;
        if (l == 0) nm = atomicAdd(queue, 1);
        nm = __shfl_sync(gmask, nm, gbase);
        if ((long long)nm >= total) {
          phase = SQ_DONE;
        } else {
          m = nm;
          e = p.list ? (long long)p.list[m] : m;
          uint32_t k0 = p.keys[2 * e], k1 = p.keys[2 * e + 1], a0, a1, b0, b1;
          for (int sp = 0; sp < p.extra_split; ++sp) {  // generator / auto-reset: key = split(key)[0]
            split2(k0, k1, a0, a1, b0, b1);
            k0 = a0;
            k1 = a1;
          }
          K0 = k0;
          K1 = k1;
          if (l == 0) {
            out_gkey[2 * m] = k0;
            out_gkey[2 * m + 1] = k1;
          }
          L = 2 * G - 1;  // SRW:352 max_length_int - i, i = 1
          attempt = 1;
          fresh = true;
        }
      }
      if (fresh) {
        for (int q = l; q < (SB >> 2); q += SQ_W) reinterpret_cast<uint32_t *>(board)[q] = reinterpret_cast<const uint32_t *>(tmpl)[q];
        w = 0;
        filled = 0;
        steps = 0;
        max_t = 0;
        h0 = K0;
        h1k = K1;
        cur = startc = safe;
        phase = SQ_SPLIT_WIRE;
      }
      __syncwarp();
    }

    // ---- one threefry block per lane (everything from here to the rare events below is executed by all 32 lanes together:
    // the phases differ in operands, not in instructions)
    const bool ph_sw = phase == SQ_SPLIT_WIRE, ph_ss = phase == SQ_SPLIT_START, ph_pk = phase == SQ_PICK, ph_swk = phase == SQ_SPLIT_WALK,
               ph_wk = phase == SQ_WALK;
    const int ip = j * SQ_W + l;
    const bool wdraw = ph_wk && draw_lane;
    const uint32_t hk0 = wdraw ? s0 : h0, hk1 = wdraw ? s1 : h1k;
    const uint32_t x0 = ph_pk ? (uint32_t)ip : wdraw ? wx0 : sx0;
    const uint32_t x1 = ph_pk ? ((ip + h1 < n1) ? (uint32_t)(ip + h1) : 0u) : wdraw ? wx1 : sx1;
    uint32_t o0, o1;
    tf_block(hk0, hk1, x0, x1, o0, o1);
    const uint32_t a0 = __shfl_sync(FULL, o0, gbase), a1 = __shfl_sync(FULL, o0, gbase + 1);
    const uint32_t b0 = __shfl_sync(FULL, o1, gbase), b1 = __shfl_sync(FULL, o1, gbase + 1);

    // ---- WALK: SRW:115-140 available_cells of the cell the wire stands on, one direction per draw lane
    const int cand = cur + dirk;
    const uint32_t wbase = 3u * w + 1u;
    const uint32_t vc = board[cand];
    const int touching = (int)own_wire(board[cand - S], wbase) + (int)own_wire(board[cand + S], wbase) + (int)own_wire(board[cand - 1], wbase) +
                         (int)own_wire(board[cand + 1], wbase);
    // :142-156 is_cell_free (the border is never free), :158-191 touches the wire through at most one cell
    const bool av = wdraw && t < L && vc == 0u && touching <= 1;
    const unsigned bal = (__ballot_sync(FULL, av) >> (gbase + 2)) & 0xFu;
    const uint32_t mant = (k_low ? o0 : o1) >> 9;
    // :211-217 choice over the padded list: largest mantissa among the available entries, lowest index on ties
    int pick = -1;
    uint32_t pm = 0;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const uint32_t mk = __shfl_sync(FULL, mant, gbase + 2 + k);
      const bool take = ((bal >> k) & 1u) && (pick < 0 || mk > pm);
      pick = take ? k : pick;
      pm = take ? mk : pm;
    }
    const bool step = ph_wk && bal != 0u;
    const bool wover = ph_wk && bal == 0u;  // :241 can_step False (or max_length steps done): the walk is over
    const int nxt = cur + (pick == 0 ? -S : pick == 1 ? S : pick == 2 ? -1 : 1);
    if (step && l == 0) {
      board[nxt] = (uint8_t)(3 * w + TARGET);  // :221
      board[cur] = (uint8_t)(3 * w + PATH);    // :223-227
    }

    // ---- PICK: the lane's two cells of this pass (words ip and ip + h1 of random_bits(d, (G*G,)))
    {
      const int i1 = ip < cells ? ip : cells - 1, i2 = ip + h1 < cells ? ip + h1 : cells - 1;
      uint32_t q, r;
      divG.divmod((uint32_t)i1, q, r);
      const bool f1 = ph_pk && ip < h1 && board[(q + 2) * S + r + 2] == 0;
      divG.divmod((uint32_t)i2, q, r);
      const bool f2 = ph_pk && ip < h1 && ip + h1 < n1 && board[(q + 2) * S + r + 2] == 0;
      const unsigned long long c1k = ((unsigned long long)(o0 >> 9) << 32) | (unsigned)(0xffff - i1);
      const unsigned long long c2k = ((unsigned long long)(o1 >> 9) << 32) | (unsigned)(0xffff - i2);
      best = (f1 && c1k > best) ? c1k : best;
      best = (f2 && c2k > best) ? c2k : best;
    }
    const bool pick_end = ph_pk && (j + 1 == P);
    j += ph_pk ? 1 : 0;

    // ---- key / phase bookkeeping of the common transitions (selects)
    //   SPLIT_WIRE  -> SPLIT_START: hash the subkey b next                        (SRW:307; the other half is dropped, :306)
    //   SPLIT_START -> PICK:        chain key c = a, hash the draw key d = b next (:51)
    //   SPLIT_WALK  -> WALK:        next chain key a is hashed next, s = b draws the first step (:204)
    //   WALK, step taken:           c <- the key hashed by lanes 0,1 a pass ago; a, b as above for the next step
    const bool can_start = filled < cells;  // SRW:53
    {
      const bool to_b = ph_sw || ph_ss, to_a = ph_swk || step;
      const uint32_t oh0 = h0, oh1 = h1k;
      h0 = to_b ? b0 : to_a ? a0 : h0;
      h1k = to_b ? b1 : to_a ? a1 : h1k;
      c0 = ph_ss ? a0 : step ? oh0 : c0;
      c1 = ph_ss ? a1 : step ? oh1 : c1;
      s0 = to_a ? b0 : s0;
      s1 = to_a ? b1 : s1;
      cur = step ? nxt : cur;
      t += step ? 1 : 0;
      filled += step ? 1 : 0;
      steps += step ? 1 : 0;
      j = ph_ss ? 0 : j;
      best = ph_ss ? 0ull : best;
      phase = ph_sw ? SQ_SPLIT_START : ph_ss ? SQ_PICK : ph_swk ? SQ_WALK : phase;
    }

    // ---- once per wire: the start cell, the end of the walk
    bool failed = ph_ss && !can_start, finished = false;  // can_start False: the attempt cannot succeed
    if (__any_sync(FULL, pick_end)) {
      if (SQ_W == 8) {
#pragma unroll
        for (int off = SQ_W / 2; off > 0; off >>= 1) {
          const unsigned long long ob = __shfl_xor_sync(FULL, best, off);
          best = ob > best ? ob : best;
        }
      } else {  // not a power of two: every lane looks at the other lanes of its group in turn
        const unsigned long long mine = best;
#pragma unroll
        for (int k = 1; k < SQ_W; ++k) {
          int src = l + k;
          src = gbase + (src >= SQ_W ? src - SQ_W : src);
          const unsigned long long ob = __shfl_sync(FULL, mine, src & 31);
          best = ob > best ? ob : best;
        }
      }
      if (pick_end) {
        uint32_t q, r;
        divG.divmod(0xffffu - (uint32_t)(best & 0xffffull), q, r);  // SRW:66 divmod(flat, rows)
        startc = (int)((q + 2) * S + r + 2);
        cur = startc;
        if (l == 0) {
          board[startc] = (uint8_t)(3 * w + POSITION);  // SRW:71
          winfo[4 * w] = c0;
          winfo[4 * w + 1] = c1;
          winfo[4 * w + 2] = (uint32_t)startc;
        }
        filled++;
        t = 0;
        h0 = c0;  // SPLIT_WALK hashes the chain key
        h1k = c1;
        phase = SQ_SPLIT_WALK;
      }
    }
    if (wover) {
      if (t == 0) {
        failed = true;  // :319 the wire did not move
      } else {
        if (l == 0) {
          board[startc] = (uint8_t)(3 * w + POSITION);  // :286
          winfo[4 * w + 3] = (uint32_t)t;
        }
        max_t = t > max_t ? t : max_t;
        ++w;
        h0 = c0;  // the tuple's key: the next wire splits it
        h1k = c1;
        cur = startc = safe;
        if (w == N)
          finished = true;
        else
          phase = SQ_SPLIT_WIRE;
      }
    }

    // ---- rare: a failed attempt, a finished board
    if (__any_sync(FULL, failed || finished)) {
      if (failed) {
        // SRW:342-366: the next attempt walks one step less, from the SAME key.  Every attempt whose max_length is still
        // >= the longest walk of the wires placed before the failing one repeats this attempt exactly (same keys, same
        // board, same steps: max_length only ever truncates a walk) and fails at the same wire, so those attempts are
        // skipped: the next one that can differ has max_length = (longest walk so far) - 1.  No wire placed: nothing
        // can change, every attempt fails.
        L = max_t - 1;
        attempt = 2 * G - L;  // max_length = rows + cols - i
        if (L <= 0) {  // an attempt with max_length 0 cannot move: SRW:389-391 zero board
          attempt = 0;
          steps = 0;
          finished = true;
        } else {
          // The attempt with max_length = L replays this one up to the first wire that walked max_t = L + 1 steps (the
          // wires before it are shorter: untouched by the smaller limit) and walks that wire from the same start cell
          // with the same keys, one step less.  So nothing before that wire is recomputed: the later wires are taken off
          // the board, the wire restarts its walk (its start cell needs no new scan) and the attempt goes on from there.
          __syncwarp(gmask);
          int wm = 0, psum = 0, pmax = 0;
          for (int i = 0; i < w; ++i) {  // w wires were placed before the failing one
            const int ti = (int)winfo[4 * i + 3];
            if (ti == max_t) {
              wm = i;
              break;
            }
            psum += ti;
            pmax = ti > pmax ? ti : pmax;
          }
          const uint32_t keep_below = 3u * wm + 1u;  // codes of the wires before wm: 1 .. 3 wm
          for (int r = 2; r < G + 2; ++r)
            for (int c = 2 + l; c < G + 2; c += SQ_W) {
              const uint32_t v = board[r * S + c];
              if (v >= keep_below) board[r * S + c] = 0;
            }
          w = wm;
          c0 = winfo[4 * wm];
          c1 = winfo[4 * wm + 1];
          startc = (int)winfo[4 * wm + 2];
          cur = startc;
          __syncwarp(gmask);
          if (l == 0) board[startc] = (uint8_t)(3 * wm + POSITION);
          filled = psum + wm + 1;  // a wire holds its steps + its start cell
          steps = psum;
          max_t = pmax;
          t = 0;
          h0 = c0;  // SPLIT_WALK hashes the chain key
          h1k = c1;
          phase = SQ_SPLIT_WALK;
          __syncwarp(gmask);
        }
      }
      if (finished) {
        __syncwarp(gmask);
        uint32_t *ob = reinterpret_cast<uint32_t *>(out_board + (size_t)m * CB);
        for (int qd = l; qd < (CB >> 2); qd += SQ_W) {
          uint32_t word = 0;
          if (attempt != 0) {
#pragma unroll
            for (int b = 0; b < 4; ++b) {
              const int i = 4 * qd + b;
              if (i < cells) {
                uint32_t q, r;
                divG.divmod((uint32_t)i, q, r);
                word |= (uint32_t)board[(q + 2) * S + r + 2] << (8 * b);
              }
            }
          }
          ob[qd] = word;
        }
        if (l == 0 && p.stats) {
          p.stats[2 * e] = attempt;
          p.stats[2 * e + 1] = steps;
        }
        phase = SQ_IDLE;
      }
    }
  }
}

static int env_w() {  // RBG_SEQRW_W=6 | 8: lanes per board
  const char *e = getenv("RBG_SEQRW_W");
  const int v = e ? atoi(e) : 0;
  return v == 6 || v == 8 ? v : 0;
}

int launch_seqrw(SeqRwParams p, int64_t max_boards, cudaStream_t stream) {
  const int G = p.G, N = p.N;
  if (G < 3) return set_error(RBG_EINVAL, "SequentialRandomWalk: rows=%d (available_cells pads with jnp.full(rows - 3, -1): rows >= 3)", G);
  const int S = G + 4, SB = (S * S + 15) & ~15, CB = (G * G + 15) & ~15;
  static int w_env = -1;
  if (w_env < 0) w_env = env_w();
  // 6 lanes per board where the walk dominates (5 boards per warp, every lane of a walk pass busy), 8 where the start-cell
  // scan does (G*G/2 blocks per wire): 10x10/5 74.9 against 66.7 M boards/s, 14x14/7 36.5 / 35.0, 20x20/10 15.8 / 15.7,
  // 32x32/16 2.48 / 2.82
  const int W = w_env ? w_env : (G <= 16 ? 6 : 8);
  const int SQ_GROUPS = W == 6 ? SqShape<6>::GROUPS : SqShape<8>::GROUPS;
  decltype(&seqrw_walk_kernel<8>) fn = W == 6 ? seqrw_walk_kernel<6> : seqrw_walk_kernel<8>;
  const size_t smem = (size_t)(SQ_GROUPS + 1) * SB + (size_t)SQ_GROUPS * 4 * RBG_MAX_N * sizeof(uint32_t);
  const size_t n = (size_t)max_boards;
  const size_t o_gkey = (n * CB + 255) & ~(size_t)255, o_queue = o_gkey + ((n * 8 + 255) & ~(size_t)255), total = o_queue + 256;
  uint8_t *base = nullptr;
  keep_pool_cached();
  cudaError_t ce = cudaMallocAsync(reinterpret_cast<void **>(&base), total, stream);
  if (ce != cudaSuccess) return set_cuda_error(ce, "cudaMallocAsync(SequentialRandomWalk scratch)");
  uint32_t *gkey = reinterpret_cast<uint32_t *>(base + o_gkey);
  int *queue = reinterpret_cast<int *>(base + o_queue);
  int rc = RBG_OK;
  do {
    if ((ce = cudaMemsetAsync(queue, 0, 256, stream)) != cudaSuccess) {
      rc = set_cuda_error(ce, "cudaMemsetAsync(SequentialRandomWalk queue)");
      break;
    }
    if ((rc = opt_in_smem(fn, smem, "seqrw_walk_kernel"))) break;
    int per_sm = 0;
    if ((ce = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, fn, SQ_THREADS, smem)) != cudaSuccess) {
      rc = set_cuda_error(ce, "cudaOccupancyMaxActiveBlocksPerMultiprocessor(seqrw_walk_kernel)");
      break;
    }
    const long long resident = (long long)(per_sm < 1 ? 1 : per_sm) * device_sm_count();
    const long long need = (max_boards + SQ_GROUPS - 1) / SQ_GROUPS;
    const unsigned ctas = (unsigned)(need < resident ? (need < 1 ? 1 : need) : resident);
    if ((rc = launch_kernel(fn, ctas, SQ_THREADS, smem, stream, RBG_K_SEQRW, "seqrw_walk_kernel", false, p, base, gkey, CB, queue,
                            FastDiv::make((uint32_t)G))))
      break;
    SeedExtParams f;
    memset(&f, 0, sizeof(f));
    f.keys = p.keys;
    f.B = p.B;
    f.G = G;
    f.N = N;
    f.mode = p.mode;
    f.solved = p.board;
    f.solved_f32 = p.float_board;
    f.starts = p.starts;
    f.ends = p.ends;
    f.st = p.st;
    f.ts = p.ts;
    f.observe = p.observe;
    f.list = p.list;
    f.list_count = p.list_count;
    rc = launch_board_finish(f, base, gkey, CB, max_boards, RBG_K_SEQRW, stream);
  } while (0);
  cudaFreeAsync(base, stream);
  return rc;
}

}  // namespace rbg
