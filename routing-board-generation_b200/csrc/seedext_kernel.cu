// seedext_kernel.cu -- SeedExtension board generation for sm_100a.
//
// Replaces jit(vmap(SeedExtensionBoard.return_solved_board / generate_starts_ends))
// and jit(vmap(SeedExtensionGenerator.__call__)):
//   reference seed_extension.py:93-304 (seeding, extension/optimise loop, starts/ends),
//   post_processor_utils_jax.py:24-195,200-234,283-429 (extend_wires_jax),
//   grid_utils.py:59-224,242-260,299-346,491-612 (optimise_wire BFS),
//   random_seed_generator.py:28-57 (generator wrapper)
//   (all under /root/reference/routing_board_generation/).
//
// The algorithm is a per-board sequential program whose cost is a threefry2x32
// hash CHAIN: every cell of every sweep advances the key by `key = split(key)[0]`
// (post_processor_utils_jax.py:156), G*G*sweeps dependent 2-block steps that no
// amount of intra-board parallelism can shorten.  So the parallel axis is the
// batch (DESIGN.md "K3"):
//   se_seed_kernel      one warp per board: key derivation, lattice seeding
//                       (the same warp-cooperative top-N selection as the
//                       ParallelRandomWalk start cells), uint8 board -> scratch
//   se_extend_kernel    persistent; one LANE per board, board in that lane's slice of shared
//                       memory (odd word stride: conflict-free when lanes touch the same cell);
//                       lanes take boards from a queue and hand them on when they have converged
//                       (6 .. 45 sweeps).  A sweep has two phases for the whole CTA: (i) the key
//                       chain of the sweep never reads the board, so the boards of the CTA that
//                       still sweep hand their keys to a dense prefix of the CTA's threads, which
//                       run the chain (two independent blocks per cell, nothing else in the loop)
//                       and park the G*G random_keys in a ring in global memory (L2); (ii) every
//                       lane walks the wire ends of its board in traversal order (per-row bit
//                       masks; an end that can no longer move is dropped for good), the lanes
//                       aligned on "k-th visit of the sweep" so that the random picks are computed
//                       by the whole warp from the parked keys.
//                       Flips are coordinate transforms, never data movement
//   se_optimise_kernel  one lane per board: per wire a FIFO breadth-first search
//                       (the reference's argmin/max queue is a FIFO in disguise),
//                       parents as 3-bit direction codes tagged with the wire id; runs on a second
//                       stream WHILE the extend kernel does, on the boards that kernel has finished
//   se_finish_kernel    one warp per board: uint8 -> int32 with 128-bit stores,
//                       starts/ends extraction, State / observation / action mask
// Boards travel between the kernels as uint8 in a stream-ordered scratch
// allocation (1 byte per cell, L2-resident for any realistic batch).
#include <stdlib.h>

#include <mutex>
#include <type_traits>

#include "connector_device.cuh"
#include "rbg_host.h"
#include "select.cuh"

namespace rbg {

struct SeScratch {
  uint8_t *board;   // [B, CB]  row-major G*G codes, CB = cells rounded up to 16
  uint32_t *keys;   // [B, 4]   loop key (2), optkey of the current iteration (2)
  uint32_t *gkey;   // [B, 2]   State.key (random_seed_generator.py:34,57)
  int32_t *status;  // [B]      bit0 BFS ran dry / pop limit (never seen), bits 8.. sweeps
  uint32_t *snap;   // [extend warps, SB2w, 32]  pre-sweep board of every lane, word-interleaved per warp
  uint2 *ring;      // [extend warps, cells + SE_LOOK + 1, 32]  random_key of every cell of the current sweep, per lane
  int CB;
};

struct SeDims {
  int G, N, wires, cells;
  int cnt, K;         // lattice side and size (seed_extension.py:104-117)
  uint32_t thresh;    // selection filter
  int cap;
  int S2, SB2w;       // extend: padded stride (G+4), words per padded board
  int refill_min;     // extend: a warp takes new boards when that many of its lanes are free
  int lane_words_ext; // extend: words per lane (the padded board + the G cell keys of a row), odd
  int S1, SB1;        // optimise: padded stride (G+2), bytes per padded board
  int fifo_bytes;     // optimise: bytes of a lane's FIFO (entries of 1 or 2 bytes), even
  int lane_bytes_opt; // optimise: bytes per lane (board, parents, fifo, pins), multiple of 4 with odd word count
};

__device__ __forceinline__ long long se_total(const SeedExtParams &p) {
  return p.list ? (long long)(*p.list_count) : p.B;
}

// ---------------------------------------------------------------- seeding
constexpr int SE_SEED_WARPS = 4;

__global__ void __launch_bounds__(SE_SEED_WARPS * 32) se_seed_kernel(const SeedExtParams p, const SeDims d, const SeScratch sc) {
  extern __shared__ __align__(16) uint8_t smem_raw[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const long long m = (long long)blockIdx.x * SE_SEED_WARPS + warp;
  if (m >= se_total(p)) return;
  const int nselp = (d.N + 1) & ~1;
  uint64_t *cand = reinterpret_cast<uint64_t *>(smem_raw) + (size_t)warp * d.cap;
  uint16_t *sel = reinterpret_cast<uint16_t *>(smem_raw + sizeof(uint64_t) * (size_t)SE_SEED_WARPS * d.cap) + warp * nselp;

  const long long e = p.list ? (long long)p.list[m] : m;
  uint32_t k0 = p.keys[2 * e], k1 = p.keys[2 * e + 1];
  uint32_t a0, a1, b0, b1;
  for (int sp = 0; sp < p.extra_split; ++sp) {  // generator / auto-reset: key = split(key)[0]
    split2(k0, k1, a0, a1, b0, b1);
    k0 = a0;
    k1 = a1;
  }
  const uint32_t g0 = k0, g1 = k1;
  split2(k0, k1, a0, a1, b0, b1);  // key, seedkey = split(key)            SE:171
  k0 = a0;
  k1 = a1;
  // return_seeded_board(seedkey) SE:93-147: randint, choice(replace=False) and
  // choice(offsets) all consume the SAME key; each starts with split(seedkey)
  // and draws from its second half.
  uint32_t s0, s1;
  split2(b0, b1, a0, a1, s0, s1);
  const int side = (int)(bits_scalar(s0, s1) & 1u);  // randint(key, (), 0, 2)
  const int lo = side ? 1 : 0;
  select_smallest(s0, s1, d.K, d.N, d.thresh, d.cap, cand, sel, lane, false);
  // offsets: randint(key, (N,), 0, 2) = random_bits(k2, (N,)) & 1
  const int h = (d.N + 1) >> 1;
  uint32_t o0 = 0, o1 = 0;
  if (lane < h) tf_block(s0, s1, (uint32_t)lane, (lane + h) < d.N ? (uint32_t)(lane + h) : 0u, o0, o1);
  const int src = lane < h ? lane : lane - h;
  const uint32_t t0 = __shfl_sync(FULL, o0, src & 31), t1 = __shfl_sync(FULL, o1, src & 31);
  const int off = (int)((lane < h ? t0 : t1) & 1u);

  uint8_t *board = sc.board + (size_t)m * sc.CB;
  uint32_t *b32 = reinterpret_cast<uint32_t *>(board);
  for (int q = lane; q < (sc.CB >> 2); q += 32) b32[q] = 0u;
  __syncwarp();
  int hr = 0, hc = 0, tr = 0, tc = 0;
  if (lane < d.N) {
    const int idx = sel[lane];
    hr = lo + 2 * (idx / d.cnt);
    hc = lo + 2 * (idx % d.cnt);
    // side != 0: offsets [(-1,0),(0,-1)]; side == 0: [(0,1),(1,0)]   SE:106-112
    const int dr = side ? (off ? 0 : -1) : (off ? 1 : 0);
    const int dc = side ? (off ? -1 : 0) : (off ? 0 : 1);
    tr = hr + dr;
    tc = hc + dc;
    board[hr * d.G + hc] = (uint8_t)(3 * lane + TARGET);  // heads carry TARGET codes  SE:145
  }
  __syncwarp();
  if (lane < d.N) board[tr * d.G + tc] = (uint8_t)(3 * lane + POSITION);  // SE:146
  if (lane == 0) {
    sc.keys[4 * m] = k0;
    sc.keys[4 * m + 1] = k1;
    sc.gkey[2 * m] = g0;
    sc.gkey[2 * m + 1] = g1;
    sc.status[m] = 0;
  }
}

// ------------------------------------------------------------ extension
// split(key, 3): blocks (0,3), (1,4), (2,5); flat = [o0_0, o0_1, o0_2, o1_0, o1_1, o1_2]
__device__ __forceinline__ void split3(uint32_t k0, uint32_t k1, uint32_t out[6]) {
  tf_block(k0, k1, 0u, 3u, out[0], out[3]);
  tf_block(k0, k1, 1u, 4u, out[1], out[4]);
  tf_block(k0, k1, 2u, 5u, out[2], out[5]);
}

// The random pick of extend_wires_jax (PPU:127-144): repeat `k, ck = split(k); pos = list[randint(ck, 0, 4)]`
// until the drawn candidate is valid, starting from the cell's key, which the loop does NOT advance.  The k of
// that loop is the cell chain itself (key = split(key)[0], PPU:156), so draw t of the cell at chain position j
// is a function of the random_key r_{j+t} = split(key_{j+t})[1] alone:
//     D(j + t) = random_bits(split(r_{j+t})[1]) & 3            (randint over a span of 4: the low draw)
// and the pick is the first t whose D lands on a valid candidate.  The row burst parks r for the row's cells
// and SE_LOOK cells beyond, so a pick needs no chain at all: the lanes of the warp evaluate, for every lane that
// needs a pick, `per` consecutive draws at once (two dependent threefry levels for the whole warp), and a
// ballot finds each lane's first hit.  A pick that outruns the parked keys (about 1 % of them) continues the
// chain on its own lane.
constexpr int SE_LOOK = 8;

__device__ __forceinline__ uint32_t se_draw(uint32_t r0, uint32_t r1) {
  uint32_t a0, a1, b0, b1;
  tf_block(r0, r1, 0u, 2u, a0, b0);
  tf_block(r0, r1, 1u, 3u, a1, b1);
  return bits_scalar(b0, b1) & 3u;  // candidate index in list order up, left, down, right
}

// ring + col: this lane's column of the sweep's parked random_keys in global memory (L2), position j at [j * 32];
// position ring_n holds the chain KEY behind the last parked position.  idx: this lane's position.
__device__ __forceinline__ uint32_t warp_pick(uint32_t needm, bool need, const uint2 *ring, uint32_t col, int ring_n, int idx, uint32_t ok, uint32_t pick, int lane) {
  const int n = __popc(needm);
  const int per = 32 / n;                      // draws evaluated per needing lane and pass
  const int slot = lane / per, j = lane - slot * per;
  const bool worker = slot < n;
  int owner = 0;  // the lane this worker draws for: the slot-th set bit of needm (few bits are set; __fns is a long software sequence)
  {
    uint32_t mk = needm;
    for (int k = 0; k < slot && mk; ++k) mk &= mk - 1u;
    owner = worker ? __ffs((int)mk) - 1 : 0;
  }
  const uint32_t own_ok = __shfl_sync(FULL, ok, owner);
  const int own_idx = __shfl_sync(FULL, idx, owner);
  const int avail = ring_n - idx, own_avail = ring_n - own_idx;
  const uint2 *rb = ring + __shfl_sync(FULL, col, owner);
  const int my_slot = __popc(needm & ((1u << lane) - 1u));
  const uint32_t my_range = (per == 32 ? FULL : ((1u << per) - 1u)) << (my_slot * per);  // the lanes that draw for me
  bool pending = need;
  for (int t0 = 0;; t0 += per) {
    const uint32_t pendm = __ballot_sync(FULL, pending && t0 < avail);
    if (!pendm) break;
    const int t = t0 + j;
    uint32_t d = 0;
    bool hit = false;
    if (worker && ((pendm >> owner) & 1u) && t < own_avail) {
      const uint2 r = __ldcg(rb + (size_t)(own_idx + t) * 32);
      d = se_draw(r.x, r.y);
      hit = ((own_ok >> d) & 1u) != 0u;
    }
    const uint32_t hits = __ballot_sync(FULL, hit) & my_range;
    const uint32_t dd = __shfl_sync(FULL, d, hits ? __ffs((int)hits) - 1 : 0);
    if (pending && hits) {
      pick = 1u << dd;
      pending = false;
    }
  }
  if (pending) {  // outran the parked keys: the chain goes on from the key behind them (draws avail, avail + 1, ...)
    const uint2 kk = __ldcg(ring + col + (size_t)ring_n * 32);
    uint32_t k0 = kk.x, k1 = kk.y;
    for (;;) {
      uint32_t n0, r0, n1, r1;
      tf_block(k0, k1, 0u, 2u, n0, r0);
      tf_block(k0, k1, 1u, 3u, n1, r1);
      const uint32_t d = se_draw(r0, r1);
      if ((ok >> d) & 1u) {
        pick = 1u << d;
        break;
      }
      k0 = n0;
      k1 = n1;
    }
  }
  return pick;
}

// extend_wires_jax's sweep loop (PPU:47-195) as a PERSISTENT kernel: a lane takes a board from the queue, sweeps it until
// it has converged, hands it on and takes the next one (sweeps per board at 14x14/7: mean 9.9, p99 23, max 45).  A sweep
// has two phases for the whole CTA.  (i) The key chain of the sweep (`key, random_key = split(key)` per cell, 57 % of the
// kernel's instructions) never reads the board, so it is not tied to the lane that owns the board: the boards of the CTA
// that still sweep hand their keys to a dense prefix of the CTA's threads, ceil(active / 32) warps run the chain at
// 32 / 32 lanes and park the random_keys in a ring in global memory (L2); warps beyond the prefix skip the phase.
// (ii) Every lane walks the wire ends of its own board (in its slice of shared memory) in traversal order.
struct SeQueue {
  int32_t *head;       // next scratch slot to hand out (zeroed by the host before the launch)
  int32_t *done_list;  // optional: scratch slots in completion order, -1 until published (consumed by se_optimise_kernel
  int32_t *done_head;  //           running at the same time), and its reservation counter
  int32_t *resident;   // optional: counts the CTAs of this launch that have started
};

__device__ __forceinline__ bool se_extendable(uint32_t v, bool two_sided) {
  if (v == 0u || v == 0xFFu) return false;
  const uint32_t wv = v - 1u, ctype = wv - 3u * ((wv * 171u) >> 9) + 1u;  // x / 3 == (x * 171) >> 9 for x < 256
  return two_sided ? ctype != PATH : ctype == TARGET;                       // PPU:109-116
}

// WIDE: G > 32, a row's mask of wire ends takes two words
template <bool WIDE>
__global__ void __launch_bounds__(256) se_extend_kernel(const SeedExtParams p, const SeDims d, const SeScratch sc, const SeQueue qu) {
  typedef typename std::conditional<WIDE, unsigned long long, uint32_t>::type mask_t;
  extern __shared__ __align__(16) uint8_t smem_raw[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (threadIdx.x == 0 && qu.resident) atomicAdd(qu.resident, 1);
  const long long total = se_total(p);
  const long long wg = (long long)blockIdx.x * (blockDim.x >> 5) + warp;
  const long long grid_warps = (long long)gridDim.x * (blockDim.x >> 5);
  // A batch that does not fill the grid is spread over its warps, `lanes_used` boards per warp: a sweep's latency (a
  // sequential hash chain per board plus, per row, as many head-extension passes as the busiest lane needs) falls
  // with fewer boards per warp.
  int lanes_used = (int)((total + grid_warps - 1) / grid_warps);
  lanes_used = lanes_used < 1 ? 1 : (lanes_used > 32 ? 32 : lanes_used);
  const int G = d.G, S = d.S2;
  // shared memory: [cnt: 8 ints][kx: one key per thread][per-lane slices]
  const int nwarps = blockDim.x >> 5;
  int *cnt = reinterpret_cast<int *>(smem_raw);
  uint2 *kx = reinterpret_cast<uint2 *>(smem_raw + 32);
  uint8_t *mine = smem_raw + 32 + (size_t)blockDim.x * 8 + ((size_t)warp * 32 + lane) * d.lane_words_ext * 4;
  uint8_t *board = mine;
  // rm[r]: bit c set = cell (r, c) holds an extendable wire end; for G > 32 the bits 32.. of row r are in rm[G + r]
  uint32_t *rm = reinterpret_cast<uint32_t *>(mine) + d.SB2w;
  constexpr bool wide = WIDE;
  // the sweep's random_keys, parked in global memory (L2) by the chain phase: position j of lane L at ring[j * 32 + L]
  const int ring_n = d.cells + SE_LOOK;
  uint2 *ring = sc.ring + (size_t)blockIdx.x * nwarps * (ring_n + 1) * 32;  // the CTA's rings, one per chain warp
  // the pre-sweep snapshot lives in global memory (L2), word q of this lane at [q * 32 + lane] of
  // its warp's region: written and read once per mirrored sweep, coalesced
  uint32_t *snap = sc.snap + (size_t)wg * d.SB2w * 32 + lane;

  uint32_t key0 = 0, key1 = 0;
  long long step_num = 0;
  long long m = -1;       // scratch slot of this lane's board, -1: none
  bool again = false;     // the board changed in its last sweep (or has not been swept yet)
  int sweeps = 0;
  bool queue_open = true;  // warp-uniform: the queue may still hold boards
  const bool two_sided = p.two_sided != 0;
  const bool use_rand = p.randomness > 0.0f;
  // The sweep is warp-synchronous: all 32 lanes walk the rows together, so that the chain bursts run at 32 / 32 lanes
  // and the random picks can be computed by the whole warp.
  for (;;) {
    // ---- boards that have converged (or reached the step limit) go back to the scratch
    const bool fin = m >= 0 && !(again && (p.ext_steps < 0 || step_num < p.ext_steps));
    const uint32_t finm = __ballot_sync(FULL, fin);
    if (finm) {
      if (fin) {
        uint32_t *dst = reinterpret_cast<uint32_t *>(sc.board + (size_t)m * sc.CB);
        int r = 0, c = 0;
        for (int q = 0; q < (d.cells + 3) >> 2; ++q) {
          uint32_t w = 0;
#pragma unroll
          for (int bb = 0; bb < 4; ++bb) {
            if (r < G) w |= (uint32_t)board[(r + 2) * S + (c + 2)] << (8 * bb);
            if (++c == G) {
              c = 0;
              ++r;
            }
          }
          dst[q] = w;
        }
        sc.status[m] += sweeps << 8;
      }
      if (qu.done_list) {  // publish: the lane's own board stores are ordered before the release store of its list entry
        int base = 0;
        if (lane == 0) base = atomicAdd(qu.done_head, __popc(finm));
        base = __shfl_sync(FULL, base, 0);
        if (fin) {
          __threadfence();
          st_release_s32(qu.done_list + base + __popc(finm & ((1u << lane) - 1u)), (int)m);
        }
      }
      if (fin) m = -1;
    }
    // ---- free lanes take the next boards of the queue
    bool fresh = false;
    if (queue_open) {
      // Boards are taken in batches (d.refill_min free lanes at least): boards of one age sweep together, and a
      // board's first sweeps are the long ones (its ends run across the empty grid: ~50 visits against ~10 later), so a
      // warp pays for them once per batch instead of in every sweep; idle lanes cost nothing in the chain phase.
      const bool want = lane < lanes_used && m < 0;
      uint32_t wantm = __ballot_sync(FULL, want);
      if (__popc(wantm) < (lanes_used < d.refill_min ? lanes_used : d.refill_min)) wantm = 0u;
      if (wantm) {
        long long base = 0;
        if (lane == 0) base = (long long)atomicAdd(qu.head, __popc(wantm));
        base = __shfl_sync(FULL, base, 0);
        const long long t = base + __popc(wantm & ((1u << lane) - 1u));
        if (want && t < total) {
          m = t;
          fresh = true;
        }
        if (base + __popc(wantm) >= total) queue_open = false;
      }
    }
    if (__any_sync(FULL, fresh)) {
      if (fresh) {
        // key, extkey, optkey = split(key, 3)   SE:189
        uint32_t f[6];
        split3(sc.keys[4 * m], sc.keys[4 * m + 1], f);
        sc.keys[4 * m] = f[0];
        sc.keys[4 * m + 1] = f[1];
        sc.keys[4 * m + 2] = f[4];
        sc.keys[4 * m + 3] = f[5];
        key0 = f[2];
        key1 = f[3];
        step_num = 0;
        sweeps = 0;
        again = true;  // prev_layout differs from the board by construction  PPU:47
        // padded board: 0xFF outside the grid (never EMPTY, never anybody's wire)
        uint32_t *w = reinterpret_cast<uint32_t *>(board);
        for (int q = 0; q < d.SB2w; ++q) w[q] = 0xFFFFFFFFu;
        const uint4 *src = reinterpret_cast<const uint4 *>(sc.board + (size_t)m * sc.CB);  // CB is a multiple of 16
        int r = 0, c = 0;
        for (int q = 0; q < (sc.CB >> 4); q += 2) {  // two 128-bit loads in flight
          const uint4 a = src[q];
          const uint4 b = q + 1 < (sc.CB >> 4) ? src[q + 1] : make_uint4(0, 0, 0, 0);
          const uint32_t ws[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
#pragma unroll
          for (int k = 0; k < 8; ++k)
#pragma unroll
            for (int bb = 0; bb < 4; ++bb) {
              if (r < G) board[(r + 2) * S + (c + 2)] = (uint8_t)(ws[k] >> (8 * bb));
              if (++c == G) {
                c = 0;
                ++r;
              }
            }
        }
        // the extendable cells (wire ends) of every row
        for (int r2 = 0; r2 < G; ++r2) {
          unsigned long long mk = 0ull;
          const uint8_t *rowp = board + (r2 + 2) * S + 2;
          for (int c2 = 0; c2 < G; ++c2) mk |= (unsigned long long)(se_extendable(rowp[c2], two_sided) ? 1u : 0u) << c2;
          rm[r2] = (uint32_t)mk;
          if (wide) rm[G + r2] = (uint32_t)(mk >> 32);
        }
      }
    }
    if (!__syncthreads_or(m >= 0)) break;  // no board in the CTA and none left in the queue
    const bool act = m >= 0 && again && (p.ext_steps < 0 || step_num < p.ext_steps);  // false only with extension_steps == 0
    bool flip = false, flop = false;
    if (act) {
      ++step_num;
      ++sweeps;
      // key, flipkey, flopkey = split(key, 3); choice over [True, False]  PPU:63-67
      uint32_t f[6];
      split3(key0, key1, f);
      key0 = f[0];
      key1 = f[1];
      flip = randint_pow2(f[2], f[3], 2u) == 0u;
      flop = randint_pow2(f[4], f[5], 2u) == 0u;
    }
    const bool mirrored = flip || flop;
    if (mirrored) {  // the convergence test needs the pre-sweep board  PPU:70,186-189
      const uint32_t *a = reinterpret_cast<const uint32_t *>(board);
      for (int q = 0; q < d.SB2w; ++q) snap[q * 32] = a[q];
    }
    bool modified = false;
    int mod_idx = 0;
    uint32_t mod_v = 0;
    // walking the FLIPPED board row-major == walking the board with mirrored
    // coordinates and mirrored neighbour directions
    const int sr = flip ? -S : S, scol = flop ? -1 : 1;
    // ---- (i) the chain of the sweep: key, random_key = split(key) for EVERY cell (PPU:156) never reads the board.
    // The sweeping boards of the CTA are ranked; thread t of the CTA runs the chain of the board of rank t: two
    // independent blocks per cell, nothing else in the loop.  random_key is parked for the sweep's cells and SE_LOOK
    // cells beyond (the random picks read ahead, see warp_pick), then the key behind them.
    const uint32_t actm = __ballot_sync(FULL, act);
    if (lane == 0) cnt[warp] = __popc(actm);
    __syncthreads();
    int rank = __popc(actm & ((1u << lane) - 1u)), nact = 0;
    for (int w2 = 0; w2 < nwarps; ++w2) {
      const int c2 = cnt[w2];
      rank += w2 < warp ? c2 : 0;
      nact += c2;
    }
    if (act) kx[rank] = make_uint2(key0, key1);
    __syncthreads();
    if (warp * 32 < nact) {  // a chain warp (lanes beyond nact run along on a stale key: harmless)
      const uint2 k = kx[threadIdx.x];
      uint32_t c0 = k.x, c1 = k.y, e0 = c0, e1 = c1;
      uint2 *rp = ring + (size_t)warp * (ring_n + 1) * 32 + lane;
      for (int i = 0; i < ring_n; ++i, rp += 32) {
        uint32_t n0, r0, n1, r1;
        tf_block(c0, c1, 0u, 2u, n0, r0);
        tf_block(c0, c1, 1u, 3u, n1, r1);
        __stcg(rp, make_uint2(r0, r1));
        c0 = n0;
        c1 = n1;
        if (i == d.cells - 1) {
          e0 = c0;
          e1 = c1;
        }
      }
      __stcg(rp, make_uint2(c0, c1));
      kx[threadIdx.x] = make_uint2(e0, e1);  // the loop key after the sweep's G*G cells
    }
    __syncthreads();  // parked keys (global) and end keys (shared) are visible to the whole CTA
    uint32_t end0 = key0, end1 = key1;
    if (act) {
      const uint2 e = kx[rank];
      end0 = e.x;
      end1 = e.y;
    }
    const uint32_t col = (uint32_t)(((rank >> 5) * (ring_n + 1)) * 32 + (rank & 31));  // this board's column of the ring
    // ---- (ii) the extendable cells of the sweep in traversal order, the lanes aligned on "k-th visit of the sweep".
    // The wire ends are the only extendable cells; rm holds them per row.  A row's mask is read when the walk
    // reaches the row (an end that moved down into it is there, one that moved up is behind the walk), an end that
    // grows along the row is added to the mask in hand and visited again, exactly as in the cell-by-cell walk.
    auto trav_mask = [&](int rowt) -> mask_t {
      const int r = flip ? G - 1 - rowt : rowt;
      if (wide) {
        const unsigned long long mk = (unsigned long long)rm[r] | ((unsigned long long)rm[G + r] << 32);
        return (mask_t)(flop ? (__brevll(mk) >> (64 - G)) : mk);
      }
      const uint32_t mk = rm[r];
      return (mask_t)(flop ? (__brev(mk) >> (32 - G)) : mk);
    };
    int rowt = 0;
    mask_t emask = act ? trav_mask(0) : (mask_t)0;
    for (;;) {
      while (act && emask == 0 && rowt < G - 1) emask = trav_mask(++rowt);
      const bool have = emask != 0;
      if (!__any_sync(FULL, have)) break;
      const int colt = have ? (wide ? __ffsll((long long)emask) : __ffs((int)emask)) - 1 : 0;
      emask &= emask - 1;
      const int r_act = flip ? G - 1 - rowt : rowt, c_act = flop ? G - 1 - colt : colt;
      uint8_t *pc = board + (r_act + 2) * S + (c_act + 2);
      const uint32_t v = have ? pc[0] : 0u;
      const int pos = rowt * G + colt;  // chain position of this cell
      uint32_t b3 = 0, ok = 0, pick = 0;
      bool need = false;
      if (have) {
        const uint32_t wv = v - 1u;
        b3 = 3u * ((wv * 171u) >> 9) + 1u;  // the wire's PATH code
        // candidates in list order up, left, down, right (PPU:322-369); a
        // candidate is dropped when it touches the wire anywhere but through
        // the current cell (PPU:86-97)
        const uint32_t u = pc[-sr], l = pc[-scol], dn = pc[sr], r = pc[scol];
        const bool oul = own_wire(pc[-sr - scol], b3), our = own_wire(pc[-sr + scol], b3);
        const bool odl = own_wire(pc[sr - scol], b3), odr = own_wire(pc[sr + scol], b3);
        ok |= (u == 0u && !own_wire(pc[-2 * sr], b3) && !oul && !our) ? 1u : 0u;
        ok |= (l == 0u && !own_wire(pc[-2 * scol], b3) && !oul && !odl) ? 2u : 0u;
        ok |= (dn == 0u && !own_wire(pc[2 * sr], b3) && !odl && !odr) ? 4u : 0u;
        ok |= (r == 0u && !own_wire(pc[2 * scol], b3) && !our && !odr) ? 8u : 0u;
        if (ok) {
          // previous neighbour: last match among up, down, left (PPU:200-234);
          // the priority cell mirrors it through the current cell (PPU:99-103)
          uint32_t pri = 0;
          if (own_wire(u, b3)) pri = 4u;   // came from above -> continue down
          if (own_wire(dn, b3)) pri = 1u;  // from below -> up
          if (own_wire(l, b3)) pri = 8u;   // from the left -> right
          bool take_pri = (ok & pri) != 0u;
          if (take_pri && use_rand) {  // PPU:157-162: random_key = split(key)[1] of this cell
            const uint2 rk = __ldcg(ring + col + (size_t)pos * 32);
            const float uni = bits_to_uniform(bits_scalar(rk.x, rk.y));
            take_pri = !(p.randomness > uni);
          }
          pick = pri;
          need = !take_pri;
        }
      }
      // repeat `k, ck = split(k); pos = list[randint(ck, 0, 4)]` until valid, from the cell's
      // key, which is NOT advanced by this loop (PPU:127-144): the whole warp computes the draws
      // of the lanes that need one (warp_pick)
      const uint32_t needm = __ballot_sync(FULL, need);
      if (needm) pick = warp_pick(needm, need, ring, col, ring_n, pos, ok, pick, lane);
      if (ok) {
        const int delta = pick == 1u ? -sr : (pick == 2u ? -scol : (pick == 4u ? sr : scol));
        pc[delta] = (uint8_t)v;   // the head / target moves      PPU:165-167
        pc[0] = (uint8_t)b3;      // and leaves PATH behind       PPU:168-173
        modified = true;
        mod_idx = (int)(pc + delta - board);  // the last write of the sweep survives it
        mod_v = v;
        // the end's bit moves with it
        const int dr = pick == 1u ? -1 : (pick == 4u ? 1 : 0), dc = pick == 2u ? -1 : (pick == 8u ? 1 : 0);  // in walk coordinates
        const int r_new = flip ? r_act - dr : r_act + dr, c_new = flop ? c_act - dc : c_act + dc;
        {
          uint32_t *w0 = rm + (wide && c_act >= 32 ? G : 0) + r_act;
          *w0 &= ~(1u << (c_act & 31));
          uint32_t *w1 = rm + (wide && c_new >= 32 ? G : 0) + r_new;
          *w1 |= 1u << (c_new & 31);
        }
        if (pick == 8u) emask |= (mask_t)1 << (colt + 1);  // grew along the row: visited again further on, as in the cell-by-cell walk
      } else if (have) {
        // No candidate left.  Cells are only ever filled during the extension (EMPTY -> end -> PATH) and a wire's
        // cells only grow, so a candidate that is taken or touches the own wire stays so: this end will never move
        // again and need not be visited any more.
        rm[(wide && c_act >= 32 ? G : 0) + r_act] &= ~(1u << (c_act & 31));
      }
    }
    if (act) {
      key0 = end0;
      key1 = end1;
    }
    // PPU:186-189: un-flip the board (a no-op here) and loop while the FLIPPED
    // pre-sweep layout differs from the un-flipped result
    if (act) {
      // flipped pre-sweep cell that faces cell (r, c) of the result: (flip ? G-1-r : r, flop ? G-1-c : c)
      auto mirror_idx = [&](int idx) {
        const int r = idx / S - 2, c = idx - (r + 2) * S - 2;
        return ((flip ? G - 1 - r : r) + 2) * S + 2 + (flop ? G - 1 - c : c);
      };
      if (!mirrored) {
        again = modified;
      } else if (!modified) {
        // nothing moved: the result IS the pre-sweep board, the loop goes on unless that board is its own mirror image
        bool diff = false;
        for (int r = 0; r < G && !diff; ++r) {
          const uint8_t *a = board + (r + 2) * S + 2;
          const uint8_t *b = board + ((flip ? G - 1 - r : r) + 2) * S + 2 + (flop ? G - 1 : 0);
          for (int c = 0; c < G; ++c) diff |= a[c] != b[c * scol];
        }
        again = diff;
      } else {
        // the cell written last holds a wire-end code, which occurs once on a board: the mirrored pre-sweep board
        // matches there only if that very end sat on the facing cell.  One snapshot word decides nearly always.
        const int o = mirror_idx(mod_idx);
        bool diff = ((snap[(o >> 2) * 32] >> (8 * (o & 3))) & 0xffu) != mod_v;
        if (!diff) {
          for (int r = 0; r < G && !diff; ++r) {
            const uint8_t *a = board + (r + 2) * S + 2;
            int oo = ((flip ? G - 1 - r : r) + 2) * S + 2 + (flop ? G - 1 : 0);  // byte offset in the snapshot
            for (int c = 0; c < G; ++c, oo += scol) {
              const uint32_t w = snap[(oo >> 2) * 32];
              diff |= (uint32_t)a[c] != ((w >> (8 * (oo & 3))) & 0xffu);
            }
          }
        }
        again = diff;
      }
    }
  }
}

// ------------------------------------------------------- optimise_wire (BFS)
// FIFO_T: uint8_t when a padded board has at most 256 cells (G <= 14), which takes a lane's footprint from 940 to
// 740 bytes at 14x14 and two more warps onto an SM; the kernel is latency-bound, so warps per SM are what it runs on
// done_list != NULL: the kernel runs WHILE se_extend_kernel does; a warp takes 32 consecutive entries of the list of
// finished boards, waits until they are published (acquire loads, pairs with the extend kernel's release stores),
// optimises them and takes the next 32.  Lanes never synchronise with each other.
// ext_resident != NULL (the launch that runs beside the extend kernel): a warp takes work only once all ext_ctas CTAs
// of the extend kernel have started, and leaves if that does not happen within a millisecond.  CTAs of this kernel
// that spin on the list while CTAs of the extend kernel wait for their shared memory would never get an entry; a
// second launch of this kernel behind the extend kernel takes whatever the first one has left.
template <typename FIFO_T>
__global__ void __launch_bounds__(128)
    se_optimise_kernel(const SeedExtParams p, const SeDims d, const SeScratch sc, const int32_t *done_list, int32_t *take_head, const int32_t *ext_resident, int ext_ctas) {
  extern __shared__ __align__(16) uint8_t smem_raw[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (ext_resident) {
    int seen = 0;
    for (int tries = 0; tries < 1000; ++tries) {
      if (lane == 0) seen = ld_acquire_s32(ext_resident);
      seen = __shfl_sync(FULL, seen, 0);
      if (seen >= ext_ctas) break;
      __nanosleep(1000);
    }
    if (seen < ext_ctas) return;
  }
  const long long total = se_total(p);
  const int G = d.G, S = d.S1, cells = d.cells;
  uint8_t *mine = smem_raw + ((size_t)warp * 32 + lane) * d.lane_bytes_opt;
  uint8_t *board = mine;                                      // [(G+2)^2] 0xFF border
  uint8_t *par = mine + d.SB1;                                // parents: (wire << 3) | (dir + 1)
  FIFO_T *fifo = reinterpret_cast<FIFO_T *>(mine + 2 * d.SB1);  // [cells + 2]
  uint16_t *pins = reinterpret_cast<uint16_t *>(mine + 2 * d.SB1 + d.fifo_bytes);  // [2N] first POSITION / TARGET per wire
  for (bool first_trip = true;; first_trip = false) {
  long long m;
  if (done_list) {
    int base = 0;
    if (lane == 0) base = atomicAdd(take_head, 32);
    base = __shfl_sync(FULL, base, 0);
    if (base >= total) return;
    if (base + lane >= total) continue;  // (the next trip ends this lane: the head is beyond the list)
    int v;
    while ((v = ld_acquire_s32(done_list + base + lane)) < 0) __nanosleep(200);
    m = v;
  } else {
    if (!first_trip) return;
    m = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (m >= total) return;
  }
  for (int q = 0; q < (d.SB1 >> 2); ++q) {
    reinterpret_cast<uint32_t *>(board)[q] = 0xFFFFFFFFu;
    reinterpret_cast<uint32_t *>(par)[q] = 0u;
  }
  for (int i = 0; i < 2 * d.N; ++i) pins[i] = 0xFFFFu;
  uint8_t *gb = sc.board + (size_t)m * sc.CB;
  for (int r = 0; r < G; ++r)
    for (int c = 0; c < G; ++c) {
      const uint32_t v = gb[r * G + c];
      const int idx = (r + 1) * S + (c + 1);
      board[idx] = (uint8_t)v;
      if (v) {  // argmax of (board == code): the first cell in row-major order  GU:512-517
        const uint32_t w = (v - 1u) / 3u, t = v - 3u * w;
        if (t == POSITION && pins[2 * w] == 0xFFFFu) pins[2 * w] = (uint16_t)idx;
        if (t == TARGET && pins[2 * w + 1] == 0xFFFFu) pins[2 * w + 1] = (uint16_t)idx;
      }
    }
  const uint32_t ok0 = sc.keys[4 * m + 2], ok1 = sc.keys[4 * m + 3];
  const int origin = S + 1;  // cell (0,0): what argmax returns when the code is absent
  int bad = 0;
  for (int w = 0; w < d.wires; ++w) {
    // optkeys = split(optkey, wires); this wire's key = flat[2w], flat[2w+1]   SE:194
    uint32_t wk[2];
#pragma unroll
    for (int t = 0; t < 2; ++t) {
      const int f = 2 * w + t;
      uint32_t x0, x1;
      if (f < d.wires) {
        tf_block(ok0, ok1, (uint32_t)f, (uint32_t)(f + d.wires), x0, x1);
        wk[t] = x0;
      } else {
        tf_block(ok0, ok1, (uint32_t)(f - d.wires), (uint32_t)f, x0, x1);
        wk[t] = x1;
      }
    }
    // neighbour order: permutation(key, arange(4)) = one _shuffle round  GU:91
    uint32_t a0, a1, s0, s1, bits[4];
    split2(wk[0], wk[1], a0, a1, s0, s1);
    tf_block(s0, s1, 0u, 2u, bits[0], bits[2]);
    tf_block(s0, s1, 1u, 3u, bits[1], bits[3]);
    int delta[4];
    {
      const int dlt[4] = {-S, 1, S, -1};  // rows [-1,0,1,0], cols [0,1,0,-1]  GU:87-88
#pragma unroll
      for (int i = 0; i < 4; ++i) {  // stable rank of bits[i]
        int rank = 0;
#pragma unroll
        for (int j = 0; j < 4; ++j) rank += (bits[j] < bits[i] || (bits[j] == bits[i] && j < i)) ? 1 : 0;
#pragma unroll
        for (int q = 0; q < 4; ++q)
          if (rank == q) delta[q] = dlt[i];
      }
    }
    const uint32_t path_num = 3u * w + PATH, start_num = 3u * w + POSITION, end_num = 3u * w + TARGET;
    const int start = pins[2 * w] == 0xFFFFu ? origin : (int)pins[2 * w];
    const int end = pins[2 * w + 1] == 0xFFFFu ? origin : (int)pins[2 * w + 1];
    board[start] = (uint8_t)path_num;  // GU:519-520
    board[end] = (uint8_t)path_num;
    const uint32_t tag = (uint32_t)w << 3;
    int head = 0, tail = 0, pops = 0;
    fifo[tail++] = (FIFO_T)start;
    auto seen = [&](int q) { const uint32_t b = par[q]; return (b & 7u) != 0u && (b & ~7u) == tag; };
    bool dry = false;
    while (pops < cells && !seen(end)) {  // GU:560-566
      if (head == tail) {
        dry = true;
        break;
      }
      const int cur = fifo[head++];
      ++pops;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int q = cur + delta[j];
        const uint32_t bv = board[q];
        if ((bv == path_num || bv == 0u) && !seen(q)) {  // GU:118-160
          par[q] = (uint8_t)(tag | (uint32_t)(j + 1));
          fifo[tail++] = (FIFO_T)q;
        }
      }
    }
    if (dry || !seen(end)) {  // not reachable on boards this pipeline makes
      board[start] = (uint8_t)start_num;
      board[end] = (uint8_t)end_num;
      bad = 1;
      continue;
    }
    // remove_path + jax_fill_grid: the wire becomes the BFS path   GU:242-346
    for (int r = 0; r < G; ++r) {
      uint8_t *rowp = board + (r + 1) * S + 1;
      for (int c = 0; c < G; ++c)
        if (rowp[c] == path_num) rowp[c] = 0;
    }
    int cur = end, n = 0, last = end;
    for (;;) {
      board[cur] = (uint8_t)path_num;
      last = cur;
      ++n;
      if (cur == start || n >= cells) break;
      cur -= delta[(par[cur] & 7u) - 1u];
    }
    board[last] = (uint8_t)start_num;
    board[end] = (uint8_t)end_num;
  }
  for (int r = 0; r < G; ++r)
    for (int c = 0; c < G; ++c) gb[r * G + c] = board[(r + 1) * S + (c + 1)];
  if (bad) sc.status[m] |= 1;
  }
}

// ------------------------------------------------------------------ outputs
constexpr int SE_FIN_WARPS = 8;

__global__ void __launch_bounds__(SE_FIN_WARPS * 32) se_finish_kernel(const SeedExtParams p, const SeDims d, const SeScratch sc, const FastDiv divG) {
  extern __shared__ __align__(16) uint8_t smem_raw[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const long long m = (long long)blockIdx.x * SE_FIN_WARPS + warp;
  if (m >= se_total(p)) return;
  const int G = d.G, N = d.N, cells = d.cells, CB = sc.CB;
  uint8_t *mine = smem_raw + (size_t)warp * (2 * CB + 8 * RBG_MAX_N);
  uint8_t *grid = mine;        // solved board
  uint8_t *pinsg = mine + CB;  // pins-only board (training grid)
  int *first = reinterpret_cast<int *>(mine + 2 * CB);  // [2N] first POSITION / TARGET cell per wire
  const long long e = p.list ? (long long)p.list[m] : m;

  const uint32_t *src = reinterpret_cast<const uint32_t *>(sc.board + (size_t)m * CB);
  for (int q = lane; q < (CB >> 2); q += 32) {
    reinterpret_cast<uint32_t *>(grid)[q] = src[q];
    reinterpret_cast<uint32_t *>(pinsg)[q] = 0u;
  }
  if (lane < N) first[2 * lane] = first[2 * lane + 1] = cells;
  __syncwarp();

  if (p.mode == 0) {  // return_solved_board: int32[G,G]
    int32_t *out = p.solved + e * cells;
    if (p.solved_f32) {  // SequentialRandomWalkBoard.generate: the same codes as float32
      float *fo = reinterpret_cast<float *>(out);
      if ((cells & 3) == 0) {
        for (int q = lane; q < (cells >> 2); q += 32) {
          const int4 v = bytes_to_int4(reinterpret_cast<const uint32_t *>(grid)[q]);
          reinterpret_cast<float4 *>(fo)[q] = make_float4((float)v.x, (float)v.y, (float)v.z, (float)v.w);
        }
      } else {
        for (int i = lane; i < cells; i += 32) fo[i] = (float)grid[i];
      }
    } else if ((cells & 3) == 0) {
      int4 *o = reinterpret_cast<int4 *>(out);
      for (int q = lane; q < (cells >> 2); q += 32) o[q] = bytes_to_int4(reinterpret_cast<const uint32_t *>(grid)[q]);
    } else {
      for (int i = lane; i < cells; i += 32) out[i] = grid[i];
    }
    return;
  }
  // generate_starts_ends SE:282-293: first POSITION / TARGET cell per wire in
  // row-major order, (0,0) when absent (argwhere(size=2) fill value)
  for (int i = lane; i < cells; i += 32) {
    const uint32_t v = grid[i];
    if (v == 0u || v > 3u * N) continue;
    const uint32_t w = (v - 1u) / 3u, t = v - 3u * w;
    if (t == POSITION) atomicMin(&first[2 * w], i);
    if (t == TARGET) atomicMin(&first[2 * w + 1], i);
  }
  __syncwarp();
  int sr = 0, scol = 0, tr = 0, tc = 0;
  if (lane < N) {
    const int fs = first[2 * lane] == cells ? 0 : first[2 * lane];
    const int ft = first[2 * lane + 1] == cells ? 0 : first[2 * lane + 1];
    uint32_t q, r;
    divG.divmod((uint32_t)fs, q, r);
    sr = (int)q;
    scol = (int)r;
    divG.divmod((uint32_t)ft, q, r);
    tr = (int)q;
    tc = (int)r;
  }
  if (p.mode == 1) {
    if (lane < N) {
      p.starts[e * 2 * N + lane] = sr;
      p.starts[e * 2 * N + N + lane] = scol;
      p.ends[e * 2 * N + lane] = tr;
      p.ends[e * 2 * N + N + lane] = tc;
    }
    return;
  }
  // SeedExtensionGenerator.__call__ RSG:34-57: pins-only grid (heads, then targets), Agent pytree
  // `grid.at[starts].set(...)`, `grid.at[targets].set(...)`: when several wires share a cell (a failed
  // SequentialRandomWalk generation leaves every pin at (0,0)) the last one stays (sequential scatter)
  {
    const unsigned act = __ballot_sync(FULL, lane < N);
    if (lane < N) {
      const unsigned peers = __match_any_sync(act, sr * G + scol);
      if ((31 - __clz(peers)) == lane) pinsg[sr * G + scol] = (uint8_t)(3 * lane + POSITION);
    }
    __syncwarp();
    if (lane < N) {
      const unsigned peers = __match_any_sync(act, tr * G + tc);
      if ((31 - __clz(peers)) == lane) pinsg[tr * G + tc] = (uint8_t)(3 * lane + TARGET);
    }
    __syncwarp();
  }
  int32_t *gout = p.st.grid + e * cells;
  if ((cells & 3) == 0) {
    int4 *o = reinterpret_cast<int4 *>(gout);
    for (int q = lane; q < (cells >> 2); q += 32) o[q] = bytes_to_int4(reinterpret_cast<const uint32_t *>(pinsg)[q]);
  } else {
    for (int i = lane; i < cells; i += 32) gout[i] = pinsg[i];
  }
  if (lane < N) {
    p.st.agent_id[e * N + lane] = lane;
    reinterpret_cast<int2 *>(p.st.start)[e * N + lane] = make_int2(sr, scol);
    reinterpret_cast<int2 *>(p.st.target)[e * N + lane] = make_int2(tr, tc);
    reinterpret_cast<int2 *>(p.st.position)[e * N + lane] = make_int2(sr, scol);
    if (p.observe) {
      SmemGrid sg{pinsg, G, 0, G};
      store_mask5(p.ts.action_mask + (e * N + lane) * 5, move_mask(sg, sr, scol, lane, sr == tr && scol == tc));
    }
  }
  if (lane == 0) {
    p.st.step_count[e] = 0;
    p.st.key[2 * e] = sc.gkey[2 * m];
    p.st.key[2 * e + 1] = sc.gkey[2 * m + 1];
    if (p.observe) p.ts.obs_step_count[e] = 0;
  }
  if (p.observe) {
    SmemGrid sg{pinsg, G, 0, G};
    warp_write_obs(sg, N, divG, p.ts.obs_grid + (size_t)e * N * cells, lane);
  }
}

// ---------------------------------------------------------------- host side
static size_t round_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

static int set_smem(const void *fn, size_t bytes, const char *name) {
  if (bytes > 227 * 1024) return set_error(RBG_EINVAL, "%s needs %zu bytes of shared memory per CTA", name, bytes);
  if (bytes > 48 * 1024) {
    cudaError_t e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
    if (e != cudaSuccess) return set_cuda_error(e, name);
  }
  return RBG_OK;
}

// second stream + fork / join events of the overlapped optimise kernel, one set per device
struct SeOverlap {
  cudaStream_t side = nullptr;
  cudaEvent_t fork = nullptr, join = nullptr;
  std::mutex mu;  // a record + wait pair on the shared events is made under it (callers on several host threads)
};
static SeOverlap *se_overlap() {
  static SeOverlap per_dev[64];
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return nullptr;
  SeOverlap &o = per_dev[dev];
  if (!o.side) {
    if (cudaStreamCreateWithFlags(&o.side, cudaStreamNonBlocking) != cudaSuccess) return nullptr;
    if (cudaEventCreateWithFlags(&o.fork, cudaEventDisableTiming) != cudaSuccess || cudaEventCreateWithFlags(&o.join, cudaEventDisableTiming) != cudaSuccess) {
      o.side = nullptr;
      return nullptr;
    }
  }
  return &o;
}

// keep the stream-ordered pool's memory cached between calls (default: released at every sync); once per device
void keep_pool_cached() {
  static bool ready[64] = {false};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64 || ready[dev]) return;
  cudaMemPool_t pool;
  if (cudaDeviceGetDefaultMemPool(&pool, dev) == cudaSuccess) {
    uint64_t thr = ~0ull;
    cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thr);
  }
  ready[dev] = true;
}

int launch_seedext(SeedExtParams p, int64_t max_boards, cudaStream_t stream) {
  const int G = p.G, N = p.N;
  SeDims d;
  d.G = G;
  d.N = N;
  d.cells = G * G;
  d.wires = N < d.cells / 3 ? N : d.cells / 3;  // SE:60-63
  d.cnt = G / 2;
  d.K = d.cnt * d.cnt;
  if (N > d.K)
    return set_error(RBG_EINVAL, "SeedExtension: %d agents need %d seed cells but the %dx%d lattice has %d (choice(replace=False) would raise)", N, N, G, G, d.K);
  if (p.iterations < 0) return set_error(RBG_EINVAL, "SeedExtension: extension_iterations=%d", p.iterations);
  d.cap = 4 * N + 32;
  {
    const double frac = (2.0 * N + 16.0) / (double)d.K;
    d.thresh = frac >= 1.0 ? 0xffffffffu : (uint32_t)(frac * 4294967296.0);
  }
  d.S2 = G + 4;
  d.SB2w = (int)(round_up((size_t)d.S2 * d.S2, 4) / 4);
  d.lane_words_ext = (d.SB2w + (G > 32 ? 2 : 1) * G) | 1;  // board + one mask of wire ends per row; odd: lanes on the same cell hit 32 different banks
  d.S1 = G + 2;
  d.SB1 = (int)round_up((size_t)d.S1 * d.S1, 4);
  {
    const bool byte_fifo = d.S1 * d.S1 <= 256;
    d.fifo_bytes = (int)((byte_fifo ? 1 : 2) * (size_t)((d.cells + 3) & ~1));
    size_t b = 2 * (size_t)d.SB1 + (size_t)d.fifo_bytes + 2 * (size_t)(2 * N);
    b = round_up(b, 4);
    if (((b / 4) & 1) == 0) b += 4;
    d.lane_bytes_opt = (int)b;
  }
  // lane-per-board kernels: small CTAs (2 warps / 1 warp), so that the boards spread evenly over the SMs
  auto warps_for = [](size_t per_warp, int w) {
    while (w > 1 && per_warp * w > 100 * 1024) --w;
    return w;
  };
  const size_t ext_warp = (size_t)32 * d.lane_words_ext * 4 + 32 * 8, opt_warp = (size_t)32 * d.lane_bytes_opt;  // extend: + one exchanged key per thread
  int ext_w = warps_for(ext_warp, 4), opt_w = warps_for(opt_warp, 1);
  // A batch that is a single wave of the extend kernel ends in a long tail of half-empty CTAs: 3-warp CTAs leave
  // shared memory for the optimise kernel to move in beside them (14x14/7, 65 536 boards: 4.17 -> 3.84 ms; bigger
  // batches are faster with 4-warp CTAs: 262 144 boards 12.7 against 13.0 ms)
  bool one_wave = false;
  if (ext_w == 4 && ext_warp * 4 + 1024 <= device_smem_per_sm() / 4) {
    one_wave = max_boards <= (int64_t)device_sm_count() * 4 * 128;
    if (one_wave) ext_w = 3;
  }
  if (const char *ex = getenv("RBG_SE_EXT_WARPS")) {
    if (atoi(ex) >= 1 && atoi(ex) <= 8) {
      ext_w = warps_for(ext_warp, atoi(ex));
      one_wave = false;
    }
  }
  int rc = RBG_OK;
  const bool wide = G > 32;
  const void *ext_fn = wide ? reinterpret_cast<const void *>(se_extend_kernel<true>) : reinterpret_cast<const void *>(se_extend_kernel<false>);
  if ((rc = set_smem(ext_fn, ext_warp * ext_w + 32, "se_extend_kernel"))) return rc;
  const bool byte_fifo = d.S1 * d.S1 <= 256;
  if ((rc = set_smem(byte_fifo ? reinterpret_cast<const void *>(se_optimise_kernel<uint8_t>) : reinterpret_cast<const void *>(se_optimise_kernel<uint16_t>), opt_warp * opt_w,
                     "se_optimise_kernel")))
    return rc;
  {
    static int rmin = -1;
    if (rmin < 0) {
      const char *ex = getenv("RBG_SE_REFILL_MIN");
      rmin = ex ? atoi(ex) : 1;
      if (rmin < 1) rmin = 1;
      if (rmin > 32) rmin = 32;
    }
    d.refill_min = rmin;
  }
  // se_extend_kernel is persistent: as many CTAs as are resident at once (RBG_SE_CTAS_PER_SM: fewer), never more than the batch needs
  unsigned ext_ctas = 1;
  {
    int per_sm = 0;
    cudaError_t oe = wide ? cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, se_extend_kernel<true>, ext_w * 32, ext_warp * ext_w + 32)
                          : cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, se_extend_kernel<false>, ext_w * 32, ext_warp * ext_w + 32);
    if (oe != cudaSuccess) return set_cuda_error(oe, "cudaOccupancyMaxActiveBlocksPerMultiprocessor(se_extend_kernel)");
    if (per_sm < 1) return set_error(RBG_EINVAL, "se_extend_kernel: a CTA of %d warps does not fit an SM (%zu bytes of shared memory)", ext_w, ext_warp * ext_w + 32);
    static int cap = -1;
    if (cap < 0) {
      const char *ex = getenv("RBG_SE_CTAS_PER_SM");
      cap = ex ? atoi(ex) : 0;
      if (cap < 0) cap = 0;
    }
    if (one_wave && per_sm > 4) per_sm = 4;
    if (cap > 0 && per_sm > cap) per_sm = cap;
    const long long resident = (long long)per_sm * device_sm_count();
    const long long need = (max_boards + ext_w * 32 - 1) / (ext_w * 32);
    ext_ctas = (unsigned)(need < resident ? need : resident);
    if (ext_ctas < 1) ext_ctas = 1;
  }
  static int overlap_env = -1;
  if (overlap_env < 0) {
    const char *ex = getenv("RBG_SE_OVERLAP");
    overlap_env = ex ? (atoi(ex) != 0 ? 1 : 0) : 1;
  }
  const bool overlap = overlap_env == 1 && !kernel_timing_on();  // per-kernel timing wants one kernel at a time
  unsigned opt_resident = 1;
  {
    int per_sm = 0;
    cudaError_t oe = byte_fifo ? cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, se_optimise_kernel<uint8_t>, opt_w * 32, opt_warp * opt_w)
                               : cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, se_optimise_kernel<uint16_t>, opt_w * 32, opt_warp * opt_w);
    if (oe != cudaSuccess) return set_cuda_error(oe, "cudaOccupancyMaxActiveBlocksPerMultiprocessor(se_optimise_kernel)");
    opt_resident = (unsigned)((per_sm < 1 ? 1 : per_sm) * device_sm_count());
  }
  SeScratch sc;
  sc.CB = (int)round_up((size_t)d.cells, 16);
  const size_t n = (size_t)max_boards;
  const size_t o_keys = round_up(n * sc.CB, 256), o_gkey = o_keys + round_up(n * 16, 256), o_status = o_gkey + round_up(n * 8, 256);
  const size_t o_snap = o_status + round_up(n * 4, 256);
  const size_t o_ring = o_snap + round_up((size_t)ext_ctas * ext_w * 32 * (size_t)d.SB2w * 4, 256);  // one snapshot region per extend warp
  const size_t o_done = o_ring + round_up((size_t)ext_ctas * ext_w * 32 * (size_t)(d.cells + SE_LOOK + 1) * 8, 256);  // and one ring of parked keys
  const size_t o_queue = o_done + round_up(n * 4, 256);  // list of finished boards (overlapped optimise)
  const size_t total = o_queue + 1024;  // queue counters: three ints per extension iteration
  uint8_t *base = nullptr;
  keep_pool_cached();
  cudaError_t ce = cudaMallocAsync(reinterpret_cast<void **>(&base), total, stream);
  if (ce != cudaSuccess) return set_cuda_error(ce, "cudaMallocAsync(SeedExtension scratch)");
  sc.board = base;
  sc.keys = reinterpret_cast<uint32_t *>(base + o_keys);
  sc.gkey = reinterpret_cast<uint32_t *>(base + o_gkey);
  sc.status = reinterpret_cast<int32_t *>(base + o_status);
  sc.snap = reinterpret_cast<uint32_t *>(base + o_snap);
  sc.ring = reinterpret_cast<uint2 *>(base + o_ring);
  int32_t *queue = reinterpret_cast<int32_t *>(base + o_queue);  // [0, 64) queue heads, [64, 128) done-list heads, [128, 192) take heads
  int32_t *done_list = reinterpret_cast<int32_t *>(base + o_done);
  if (p.iterations > 64) {
    cudaFreeAsync(base, stream);
    return set_error(RBG_EINVAL, "SeedExtension: extension_iterations=%d (max 64)", p.iterations);
  }

  do {
    cudaError_t me = cudaMemsetAsync(queue, 0, 1024, stream);
    if (me != cudaSuccess) {
      rc = set_cuda_error(me, "cudaMemsetAsync(SeedExtension queue)");
      break;
    }
    {  // seeding: one warp per board
      const size_t smem = sizeof(uint64_t) * SE_SEED_WARPS * d.cap + sizeof(uint16_t) * SE_SEED_WARPS * ((N + 1) & ~1);
      const unsigned ctas = (unsigned)((max_boards + SE_SEED_WARPS - 1) / SE_SEED_WARPS);
      LaunchScope scope(RBG_K_SEEDEXT, stream);
      se_seed_kernel<<<ctas, SE_SEED_WARPS * 32, smem, stream>>>(p, d, sc);
    }
    if ((rc = check_launch("se_seed_kernel"))) break;
    for (int it = 0; it < p.iterations && rc == RBG_OK; ++it) {  // SE:180-200 while_loop over extension_iterations
      // The optimise kernel runs WHILE the extend kernel does (on a second stream), on the boards the extend kernel
      // has finished: extension ends in a long tail (a board needs 6 .. 45 sweeps and every sweep is a sequential hash
      // chain), during which most SMs would idle, and the optimise kernel is latency-bound at a few warps per SM.
      // Neither kernel waits for the other to become resident: the extend kernel's CTAs take boards from a queue, so
      // it completes with whatever share of the SMs it gets, and the optimise warps only wait for list entries.
      SeOverlap *ov = overlap ? se_overlap() : nullptr;
      SeQueue qu;
      qu.head = queue + it;
      qu.done_list = ov ? done_list : nullptr;
      qu.done_head = ov ? queue + 64 + it : nullptr;
      qu.resident = ov ? queue + 192 + it : nullptr;
      cudaError_t ce2 = cudaSuccess;
      std::unique_lock<std::mutex> ovlock;
      if (ov) ovlock = std::unique_lock<std::mutex>(ov->mu);  // held for the iteration: the side stream's work is enqueued in one piece
      if (ov) {
        if ((ce2 = cudaMemsetAsync(done_list, 0xFF, n * 4, stream)) != cudaSuccess || (ce2 = cudaEventRecord(ov->fork, stream)) != cudaSuccess ||
            (ce2 = cudaStreamWaitEvent(ov->side, ov->fork, 0)) != cudaSuccess) {
          rc = set_cuda_error(ce2, "SeedExtension: fork to the optimise stream");
          break;
        }
      }
      {
        LaunchScope scope(RBG_K_SEEDEXT, stream);
        if (wide)
          se_extend_kernel<true><<<ext_ctas, ext_w * 32, ext_warp * ext_w + 32, stream>>>(p, d, sc, qu);
        else
          se_extend_kernel<false><<<ext_ctas, ext_w * 32, ext_warp * ext_w + 32, stream>>>(p, d, sc, qu);
      }
      if ((rc = check_launch("se_extend_kernel"))) break;
      if (ov) {  // beside the extend kernel: as many CTAs as the device holds; they move in as the extend CTAs leave
        unsigned ctas = (unsigned)((max_boards + opt_w * 32 - 1) / (opt_w * 32));
        if (ctas > opt_resident) ctas = opt_resident;
        LaunchScope scope(RBG_K_SEEDEXT, ov->side);
        if (byte_fifo)
          se_optimise_kernel<uint8_t><<<ctas, opt_w * 32, opt_warp * opt_w, ov->side>>>(p, d, sc, done_list, queue + 128 + it, qu.resident, (int)ext_ctas);
        else
          se_optimise_kernel<uint16_t><<<ctas, opt_w * 32, opt_warp * opt_w, ov->side>>>(p, d, sc, done_list, queue + 128 + it, qu.resident, (int)ext_ctas);
        if ((rc = check_launch("se_optimise_kernel"))) break;
      }
      {  // behind the extend kernel: everything (no overlap), or what the first launch has not taken
        unsigned ctas = (unsigned)((max_boards + opt_w * 32 - 1) / (opt_w * 32));
        if (ov && ctas > opt_resident) ctas = opt_resident;
        LaunchScope scope(RBG_K_SEEDEXT, stream);
        if (byte_fifo)
          se_optimise_kernel<uint8_t><<<ctas, opt_w * 32, opt_warp * opt_w, stream>>>(p, d, sc, ov ? done_list : nullptr, queue + 128 + it, nullptr, 0);
        else
          se_optimise_kernel<uint16_t><<<ctas, opt_w * 32, opt_warp * opt_w, stream>>>(p, d, sc, ov ? done_list : nullptr, queue + 128 + it, nullptr, 0);
      }
      if ((rc = check_launch("se_optimise_kernel"))) break;
      if (ov) {
        if ((ce2 = cudaEventRecord(ov->join, ov->side)) != cudaSuccess || (ce2 = cudaStreamWaitEvent(stream, ov->join, 0)) != cudaSuccess) {
          rc = set_cuda_error(ce2, "SeedExtension: join of the optimise stream");
          break;
        }
      }
    }
    if (rc) break;
    {
      const size_t smem = (size_t)SE_FIN_WARPS * (2 * sc.CB + 8 * RBG_MAX_N);
      const unsigned ctas = (unsigned)((max_boards + SE_FIN_WARPS - 1) / SE_FIN_WARPS);
      LaunchScope scope(RBG_K_SEEDEXT, stream);
      se_finish_kernel<<<ctas, SE_FIN_WARPS * 32, smem, stream>>>(p, d, sc, FastDiv::make((uint32_t)G));
    }
    rc = check_launch("se_finish_kernel");
  } while (0);
  cudaFreeAsync(base, stream);
  return rc;
}

int launch_board_finish(const SeedExtParams &p, const uint8_t *boards, const uint32_t *gkey, int CB, int64_t max_boards, int kernel_id,
                        cudaStream_t stream) {
  SeDims d;
  memset(&d, 0, sizeof(d));
  d.G = p.G;
  d.N = p.N;
  d.cells = p.G * p.G;
  SeScratch sc;
  memset(&sc, 0, sizeof(sc));
  sc.board = const_cast<uint8_t *>(boards);
  sc.gkey = const_cast<uint32_t *>(gkey);
  sc.CB = CB;
  const size_t smem = (size_t)SE_FIN_WARPS * (2 * sc.CB + 8 * RBG_MAX_N);
  const unsigned ctas = (unsigned)((max_boards + SE_FIN_WARPS - 1) / SE_FIN_WARPS);
  {
    LaunchScope scope(kernel_id, stream);
    se_finish_kernel<<<ctas < 1 ? 1 : ctas, SE_FIN_WARPS * 32, smem, stream>>>(p, d, sc, FastDiv::make((uint32_t)p.G));
  }
  return check_launch("se_finish_kernel");
}

}  // namespace rbg
