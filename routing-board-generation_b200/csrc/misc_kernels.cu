// misc_kernels.cu -- key derivation for sharded batches and the on-device
// board validity check.
#include "rbg_host.h"

namespace rbg {

// rows [offset, offset+count) of jax.random.split(key, B) (SURVEY A.2):
// flat word f of the split output is o0(f, f+B) for f < B, o1(f-B, f) otherwise.
// Reference convention: keys = split(PRNGKey(0), B) (dataset_generator_jax.py:76),
// per-device contiguous slices (rl_training/setup_train.py:397-399).
__global__ void __launch_bounds__(256) split_keys_kernel(uint32_t k0, uint32_t k1, long long B,
                                                         long long offset, long long count,
                                                         uint32_t *__restrict__ out) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= 2 * count) return;
  const long long f = 2 * offset + i;
  uint32_t o0, o1;
  if (f < B) {
    tf_block(k0, k1, (uint32_t)f, (uint32_t)(f + B), o0, o1);
    out[i] = o0;
  } else {
    tf_block(k0, k1, (uint32_t)(f - B), (uint32_t)f, o0, o1);
    out[i] = o1;
  }
}

int launch_split_keys(uint32_t k0, uint32_t k1, int64_t B, int64_t offset, int64_t count,
                      uint32_t *out, cudaStream_t stream) {
  if (count <= 0) return RBG_OK;
  const int64_t n = 2 * count;
  return launch_kernel(split_keys_kernel, (unsigned)((n + 255) / 256), 256, 0, stream, RBG_K_SPLIT, "split_keys_kernel", false, k0, k1, B, offset, count, out);
}

// jax.vmap(lambda k: jax.random.split(k, num))(keys): out[b, i] = (flat[2i], flat[2i+1]) of
// threefry_2x32(keys[b], iota(2 * num)) (SURVEY A.2); one thread per output word.
__global__ void __launch_bounds__(256) split_each_kernel(const uint32_t *__restrict__ keys, long long B, int num,
                                                         uint32_t *__restrict__ out) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B * 2 * num) return;
  const long long b = i / (2 * num);
  const uint32_t f = (uint32_t)(i - b * 2 * num);
  uint32_t o0, o1;
  if (f < (uint32_t)num) {
    tf_block(keys[2 * b], keys[2 * b + 1], f, f + (uint32_t)num, o0, o1);
    out[i] = o0;
  } else {
    tf_block(keys[2 * b], keys[2 * b + 1], f - (uint32_t)num, f, o0, o1);
    out[i] = o1;
  }
}

int launch_split_each(const uint32_t *keys, int64_t B, int num, uint32_t *out, cudaStream_t stream) {
  const int64_t n = B * 2 * num;
  if (n <= 0) return RBG_OK;
  return launch_kernel(split_each_kernel, (unsigned)((n + 255) / 256), 256, 0, stream, RBG_K_SPLIT, "split_each_kernel", false, keys, B, num, out);
}

// BoardDatasetGeneratorJAX.__call__ (dataset_generator_jax.py:112-141), one warp per env:
// key, _ = split(key); which = randint(key, (), 0, K) with jax's two-draw formula
// (SURVEY A.9); pins-only grid from heads[which] / targets[which] (heads first, then targets).
constexpr int DS_WARPS = 8;

__global__ void __launch_bounds__(DS_WARPS * 32) dataset_state_kernel(const uint32_t *__restrict__ keys, long long B, int G, int N,
                                                                      const int32_t *__restrict__ heads, const int32_t *__restrict__ targets,
                                                                      uint32_t K, rbg_state st) {
  const int lane = threadIdx.x & 31;
  const long long e = (long long)blockIdx.x * DS_WARPS + (threadIdx.x >> 5);
  if (e >= B) return;
  const int cells = G * G;
  uint32_t k0, k1;
  const uint32_t which = dataset_pick(keys[2 * e], keys[2 * e + 1], K, k0, k1);
  int32_t *grid = st.grid + e * cells;
  for (int i = lane; i < cells; i += 32) grid[i] = 0;
  int sr = 0, sc = 0, tr = 0, tc = 0;
  if (lane < N) {
    const int32_t *h = heads + (size_t)which * 2 * N, *t = targets + (size_t)which * 2 * N;
    sr = h[lane];
    sc = h[N + lane];
    tr = t[lane];
    tc = t[N + lane];
  }
  __syncwarp();
  if (lane < N && (unsigned)sr < (unsigned)G && (unsigned)sc < (unsigned)G) grid[sr * G + sc] = 3 * lane + POSITION;
  __syncwarp();
  if (lane < N && (unsigned)tr < (unsigned)G && (unsigned)tc < (unsigned)G) grid[tr * G + tc] = 3 * lane + TARGET;
  if (lane < N) {
    st.agent_id[e * N + lane] = lane;
    reinterpret_cast<int2 *>(st.start)[e * N + lane] = make_int2(sr, sc);
    reinterpret_cast<int2 *>(st.target)[e * N + lane] = make_int2(tr, tc);
    reinterpret_cast<int2 *>(st.position)[e * N + lane] = make_int2(sr, sc);
  }
  if (lane == 0) {
    st.step_count[e] = 0;
    st.key[2 * e] = k0;
    st.key[2 * e + 1] = k1;
  }
}

int launch_dataset_state(const uint32_t *keys, int64_t B, int G, int N, const int32_t *heads, const int32_t *targets, int64_t K,
                         const rbg_state &st, cudaStream_t stream) {
  if (B <= 0) return RBG_OK;
  return launch_kernel(dataset_state_kernel, (unsigned)((B + DS_WARPS - 1) / DS_WARPS), DS_WARPS * 32, 0, stream, RBG_K_VALIDATE, "dataset_state_kernel", false,
                       keys, B, G, N, heads, targets, (uint32_t)K, st);
}

// Board validity, one warp per board.  The rules are the reference's NumPy functions
// (numpy_implementation/utils/post_processor_utils_numpy.py:34-155 = UP,
// numpy_implementation/utils/board_processor.py:111-162,391-487 = BP); flag bits as in
// include/rbg_b200.h rbg_validate.  tests/golden/validity_reference.npz holds the reference's own
// verdicts on 2 400 boards.
constexpr int VAL_WARPS = 4;

struct ValSmem {
  uint8_t *grid, *reached;
  int *heads, *targets, *paths, *hpos, *tpos;
};

// flood `reached` from the cells already marked, through cells whose wire id matches their own
// (strict = wire cells only, every wire at once) or, for one wire `w`, through its cells and EMPTY
__device__ __forceinline__ void val_flood(const ValSmem &s, int G, int cells, int lane, int w, int stop_at) {
  for (int it = 0; it < cells; ++it) {
    bool changed = false;
    for (int i = lane; i < cells; i += 32) {
      const int v = s.grid[i];
      if (s.reached[i]) continue;
      int cw;  // the wire whose flood may enter this cell
      if (w < 0) {
        if (v == 0) continue;
        cw = (v - 1) / 3;
      } else {
        if (v != 0 && (v - 1) / 3 != w) continue;
        cw = w;
      }
      const int r = i / G, c = i - r * G;
      auto from = [&](int k) {
        if (!s.reached[k]) return false;
        const int u = s.grid[k];
        return w < 0 ? (u > 0 && (u - 1) / 3 == cw) : true;  // (with w >= 0 only passable cells are ever marked)
      };
      if ((r > 0 && from(i - G)) || (r < G - 1 && from(i + G)) || (c > 0 && from(i - 1)) || (c < G - 1 && from(i + 1))) {
        s.reached[i] = 1;
        changed = true;
      }
    }
    __syncwarp();
    if (!__any_sync(FULL, changed)) break;
    if (stop_at >= 0 && s.reached[stop_at]) break;
  }
}

__global__ void __launch_bounds__(VAL_WARPS * 32) validate_kernel(const int32_t *__restrict__ boards, long long B,
                                                                  int G, int N, int32_t *__restrict__ flags) {
  extern __shared__ __align__(16) uint8_t smem_raw[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int cells = G * G;
  const int cp = (cells + 15) & ~15;
  ValSmem s;
  s.grid = smem_raw + (size_t)warp * (2 * cp + 5 * 4 * RBG_MAX_N);
  s.reached = s.grid + cp;
  s.heads = reinterpret_cast<int *>(s.reached + cp);
  s.targets = s.heads + RBG_MAX_N;
  s.paths = s.targets + RBG_MAX_N;
  s.hpos = s.paths + RBG_MAX_N;
  s.tpos = s.hpos + RBG_MAX_N;
  for (long long b = (long long)blockIdx.x * VAL_WARPS + warp; b < B; b += (long long)gridDim.x * VAL_WARPS) {
    const int32_t *src = boards + b * cells;
    int fl = 0;
    if (lane < N) {
      s.heads[lane] = s.targets[lane] = s.paths[lane] = 0;
      s.hpos[lane] = s.tpos[lane] = cells;
    }
    __syncwarp();
    // verify_encodings_range (BP:406-416); is_valid_board raises there, so nothing else is evaluated
    for (int i = lane; i < cells; i += 32) {
      const int v = __ldg(src + i);
      if (v < 0 || v > 3 * N) fl |= 1;
      s.grid[i] = (uint8_t)v;
      s.reached[i] = 0;
    }
    fl = __reduce_or_sync(FULL, fl);
    if (fl) {
      if (lane == 0) flags[b] = fl;
      __syncwarp();
      continue;
    }
    __syncwarp();
    // per wire: code counts, FIRST head / target in row-major order (np.argwhere(...)[0], BP:79-82)
    for (int i = lane; i < cells; i += 32) {
      const int v = s.grid[i];
      if (v == 0) continue;
      const int w = (v - 1) / 3, t = (v - 1) % 3 + 1;
      if (t == PATH) atomicAdd(&s.paths[w], 1);
      if (t == POSITION) {
        atomicAdd(&s.heads[w], 1);
        atomicMin(&s.hpos[w], i);
      }
      if (t == TARGET) {
        atomicAdd(&s.targets[w], 1);
        atomicMin(&s.tpos[w], i);
      }
    }
    __syncwarp();
    // verify_number_heads_tails (BP:419-431): absence only (its counts run over unique values)
    bool eligible = false, zl = false;
    if (lane < N) {
      const int nh = s.heads[lane], nt = s.targets[lane];
      zl = nh == 0 && nt == 1 && s.paths[lane] == 0;  // zero-length wire: a lone TARGET
      if (zl) fl |= 16;
      if (nh < 1 || nt < 1) fl |= zl ? 2 : (2 | 128);
      if (nh > 1 || nt > 1) fl |= 32;
      eligible = nh >= 1 && nt >= 1;
    }
    const uint32_t zmask = __ballot_sync(FULL, zl);
    // verify_wire_validity (UP:88-121) with num_wire_neighbors (UP:124-155)
    auto same = [&](int i, int w) { const int v = s.grid[i]; return v > 0 && (v - 1) / 3 == w; };
    bool struct_bad = false;  // ... at a cell that does not belong to a zero-length wire
    for (int i = lane; i < cells; i += 32) {
      const int v = s.grid[i];
      if (v == 0) continue;
      const int w = (v - 1) / 3, t = (v - 1) % 3 + 1;
      const int r = i / G, c = i - r * G;
      int nb = 0;
      nb += (r > 0 && same(i - G, w));
      nb += (r < G - 1 && same(i + G, w));
      nb += (c > 0 && same(i - 1, w));
      nb += (c < G - 1 && same(i + 1, w));
      if (t == PATH ? nb != 2 : nb != 1) {
        const bool excused = (zmask >> w) & 1u;
        fl |= excused ? 4 : (4 | 128);
        struct_bad |= !excused;
      }
    }
    // first head -> first target through the wire's own cells.  When the neighbour rule holds for every
    // cell of the wires that have a head (warp-uniform test), such a wire is a set of simple chains and
    // lane w just walks the one that starts at its head; otherwise flood from every first head at once.
    bool connected = false;
    if (!__any_sync(FULL, struct_bad)) {
      // A wire with exactly one head and one target whose cells all obey the neighbour rule has exactly two cells of
      // degree one, its head and its target: the chain that starts at one ends at the other (whatever cycles of PATH
      // cells may lie beside it), so there is nothing to walk.  Only duplicated heads / targets need the walk.
      const bool single = eligible && s.heads[lane] == 1 && s.targets[lane] == 1;
      connected = single;
      if (eligible && !single) {
        int cur = s.hpos[lane], prev = -1;
        const int goal = s.tpos[lane];
        for (int step = 0; step < cells && cur != goal; ++step) {
          const int r = cur / G, c = cur - r * G;
          int nxt = -1;
          if (r > 0 && cur - G != prev && same(cur - G, lane)) nxt = cur - G;
          if (r < G - 1 && cur + G != prev && same(cur + G, lane)) nxt = cur + G;
          if (c > 0 && cur - 1 != prev && same(cur - 1, lane)) nxt = cur - 1;
          if (c < G - 1 && cur + 1 != prev && same(cur + 1, lane)) nxt = cur + 1;
          if (nxt < 0) break;
          prev = cur;
          cur = nxt;
        }
        connected = cur == goal;
      }
    } else {
      if (eligible) s.reached[s.hpos[lane]] = 1;
      __syncwarp();
      val_flood(s, G, cells, lane, -1, -1);
      if (eligible) connected = s.reached[s.tpos[lane]] != 0;
    }
    if (eligible && !connected) fl |= 8;
    // get_path_from_head_and_target (BP:111-162) for the wires that are not connected through their own
    // cells: the same search through own cells AND EMPTY ones; PathNotFoundError when it fails
    uint32_t todo = __ballot_sync(FULL, eligible && !connected);
    while (todo) {
      const int w = __ffs(todo) - 1;
      todo &= todo - 1;
      for (int i = lane; i < cells; i += 32) s.reached[i] = 0;
      __syncwarp();
      const int goal = s.tpos[w];
      if (lane == 0) s.reached[s.hpos[w]] = 1;
      __syncwarp();
      val_flood(s, G, cells, lane, w, goal);
      if (!s.reached[goal]) fl |= 64;
      __syncwarp();
    }
    fl = __reduce_or_sync(FULL, fl);
    if (lane == 0) flags[b] = fl;
    __syncwarp();
  }
}

// ---------------------------------------------------------------------------------------------------
// Board statistics: EvaluateEmptyBoard (benchmarking/benchmarks/empty_board_evaluation.py:31-155), the
// deterministic part -- score_from_neighbours (:56-88: 3x3 weighted window of the per-cell scores times the
// number of distinct wire labels in the window, with _change_heads_to_wire_ids' label map :90-97),
// count_detours (:99-137) and heatmap_score_diversity (:155, the number of distinct scores).  One warp per
// board, the board as bytes in shared memory with a one-cell border; 4 B read and (optionally) 4 B written per
// cell.  tests/golden/board_stats_reference.npz holds the reference class's own outputs.
constexpr int STAT_WARPS = 4;
constexpr int STAT_SCORE_BITS = 1024;  // scores lie in [-9 * 32, 9 * 48]; bit = score + 320

__global__ void __launch_bounds__(STAT_WARPS * 32) board_stats_kernel(const int32_t *__restrict__ boards, long long B, int G, int count_current_wire,
                                                                     int32_t *__restrict__ scored, int32_t *__restrict__ detours,
                                                                     int32_t *__restrict__ diversity, int32_t *__restrict__ status) {
  extern __shared__ __align__(16) uint8_t smem_raw[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int P = G + 2, PB = (P * P + 15) & ~15, cells = G * G;
  uint8_t *raw = smem_raw + (size_t)warp * (3 * PB + STAT_SCORE_BITS / 8);  // codes, 0 on the border
  uint8_t *lab = raw + PB;                                                  // _change_heads_to_wire_ids labels
  int8_t *ind = reinterpret_cast<int8_t *>(lab + PB);                       // assess_board scores, 0 on the border
  uint32_t *bits = reinterpret_cast<uint32_t *>(ind + PB);
  for (long long b = (long long)blockIdx.x * STAT_WARPS + warp; b < B; b += (long long)gridDim.x * STAT_WARPS) {
    const int32_t *src = boards + b * cells;
    for (int i = lane; i < PB; i += 32) raw[i] = lab[i] = 0, ind[i] = 0;
    if (lane < STAT_SCORE_BITS / 32) bits[lane] = 0u;
    __syncwarp();
    // codes must fit the label / wire-number bit sets: 0 .. 96 (32 wires); anything else is reported, not scored
    int bad = 0;
    uint32_t plo = 0;  // POSITION codes present: unique(filled_board[filled_board % 3 == 2])  (:92), bit w for code 3w + 2
    for (int i = lane; i < cells; i += 32) {
      const int v = __ldg(src + i);
      if (v < 0 || v > 3 * RBG_MAX_N) {
        bad = 1;
        continue;
      }
      const int r = i / G, c = i - r * G;
      raw[(r + 1) * P + c + 1] = (uint8_t)v;
      if (v % 3 == 2) plo |= 1u << (v / 3);
    }
    bad = __reduce_or_sync(FULL, bad);
    plo = __reduce_or_sync(FULL, plo);
    if (bad) {
      if (lane == 0) {
        detours[b] = -1;
        diversity[b] = -1;
        if (status) atomicOr(status, 1);
      }
      __syncwarp();
      continue;
    }
    __syncwarp();
    for (int i = lane; i < cells; i += 32) {
      const int r = i / G, c = i - r * G, idx = (r + 1) * P + c + 1;
      int v = raw[idx];
      ind[idx] = (int8_t)(v == 0 ? -2 : (v % 3 == 1 ? 2 : 3));  // assess_board (:41-54)
      // for every head code id present: cells == id + 1 -> id, cells == id + 2 -> id  (:94-96)
      if (v > 0 && v % 3 == 0 && ((plo >> ((v - 1) / 3)) & 1u)) v -= 1;
      else if (v >= 4 && v % 3 == 1 && ((plo >> ((v - 2) / 3)) & 1u)) v -= 2;
      lab[idx] = (uint8_t)v;
    }
    __syncwarp();
    // score_from_neighbours (:56-88)
    for (int i = lane; i < cells; i += 32) {
      const int r = i / G, c = i - r * G, idx = (r + 1) * P + c + 1;
      int sum = 0, nseen = 0;
      uint32_t seen[9];
#pragma unroll
      for (int dr = -1; dr <= 1; ++dr)
#pragma unroll
        for (int dc = -1; dc <= 1; ++dc) {
          const int q = idx + dr * P + dc;
          sum += (int)ind[q] * ((dr == 0 ? 2 : 1) * (dc == 0 ? 2 : 1));
          const uint32_t l = lab[q];
          bool dup = l == 0u;
#pragma unroll
          for (int k = 0; k < 9; ++k) dup |= k < nseen && seen[k] == l;
          if (!dup) {
#pragma unroll
            for (int k = 0; k < 9; ++k)
              if (k == nseen) seen[k] = l;
            ++nseen;
          }
        }
      const int sc = sum * nseen;
      if (scored) scored[b * cells + i] = sc;
      atomicOr(&bits[(sc + 320) >> 5], 1u << ((sc + 320) & 31));
    }
    // count_detours (:99-137): wire numbers by get_wire_num (:139-151), -1 .. 31 as bits 0 .. 32
    int det = 0;
    for (int i = lane; i < cells; i += 32) {
      const int x = i / G, y = i - x * G;
      const int v = raw[(x + 1) * P + y + 1];
      if (v < 2 || v % 3 == 2) continue;
      const int cur = (v - 2) / 3;
      unsigned long long above = 0, below = 0, left = 0, right = 0;
      for (int t = 0; t < G; ++t) {
        const int u = raw[(t + 1) * P + y + 1], h = raw[(x + 1) * P + t + 1];
        const int wu = u < 2 ? -1 : (u - 2) / 3, wh = h < 2 ? -1 : (h - 2) / 3;
        if (t != x && u != 0 && (count_current_wire || wu != cur)) (t < x ? above : below) |= 1ull << (wu + 1);
        if (t != y && h != 0 && (count_current_wire || wh != cur)) (t < y ? left : right) |= 1ull << (wh + 1);
      }
      det += __popcll(above & below) + __popcll(left & right);
    }
    det = __reduce_add_sync(FULL, det);
    __syncwarp();
    int nd = lane < STAT_SCORE_BITS / 32 ? __popc(bits[lane]) : 0;
    nd = __reduce_add_sync(FULL, nd);
    if (lane == 0) {
      detours[b] = det;
      diversity[b] = nd;
    }
    __syncwarp();
  }
}

int launch_board_stats(const int32_t *boards, int64_t B, int G, int count_current_wire, int32_t *scored, int32_t *detours, int32_t *diversity,
                       cudaStream_t stream) {
  if (B <= 0) return RBG_OK;
  const int P = G + 2, PB = (P * P + 15) & ~15;
  const size_t smem = (size_t)STAT_WARPS * (3 * PB + STAT_SCORE_BITS / 8);
  int64_t ctas = (B + STAT_WARPS - 1) / STAT_WARPS;
  if (ctas > (int64_t)device_sm_count() * 32) ctas = (int64_t)device_sm_count() * 32;
  return launch_kernel(board_stats_kernel, (unsigned)ctas, STAT_WARPS * 32, smem, stream, RBG_K_VALIDATE, "board_stats_kernel", false, boards, B, G,
                       count_current_wire, scored, detours, diversity, nullptr);
}

int launch_validate(const int32_t *boards, int64_t B, int G, int N, int32_t *flags, cudaStream_t stream) {
  if (B <= 0) return RBG_OK;
  const int cells = G * G, cp = (cells + 15) & ~15;
  const size_t smem = (size_t)VAL_WARPS * (2 * cp + 5 * 4 * RBG_MAX_N);
  int64_t ctas = (B + VAL_WARPS - 1) / VAL_WARPS;
  if (ctas > (int64_t)device_sm_count() * 64) ctas = (int64_t)device_sm_count() * 64;
  return launch_kernel(validate_kernel, (unsigned)ctas, VAL_WARPS * 32, smem, stream, RBG_K_VALIDATE, "validate_kernel", false, boards, B, G, N, flags);
}

// ---- host transport of the observation (rbg_connector_step_host_io) -------------------------------------
// Codes are <= 3 * RBG_MAX_N < 256: the int32 observation crosses the bus as bytes (4x fewer) and is widened back
// to the API's int32 by the host threads of the call (host_pool.cpp).  16 codes per thread: four 128-bit loads in
// flight, one 128-bit store.
__global__ void __launch_bounds__(256) narrow_codes_kernel(const int32_t *__restrict__ src, uint8_t *__restrict__ dst, long long n) {
  const long long n16 = n >> 4;
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x; q < n16; q += stride) {
    const int4 *s = reinterpret_cast<const int4 *>(src) + 4 * q;
    const int4 a = s[0], b = s[1], c = s[2], d = s[3];
    uint4 o;
    o.x = (uint32_t)a.x | ((uint32_t)a.y << 8) | ((uint32_t)a.z << 16) | ((uint32_t)a.w << 24);
    o.y = (uint32_t)b.x | ((uint32_t)b.y << 8) | ((uint32_t)b.z << 16) | ((uint32_t)b.w << 24);
    o.z = (uint32_t)c.x | ((uint32_t)c.y << 8) | ((uint32_t)c.z << 16) | ((uint32_t)c.w << 24);
    o.w = (uint32_t)d.x | ((uint32_t)d.y << 8) | ((uint32_t)d.z << 16) | ((uint32_t)d.w << 24);
    reinterpret_cast<uint4 *>(dst)[q] = o;
  }
  const long long t = (n16 << 4) + (long long)blockIdx.x * blockDim.x + threadIdx.x;  // the last n % 16 codes
  if (t < n) dst[t] = (uint8_t)src[t];
}

// two codes < 16 per byte (low nibble first): the observation of boards with at most 5 agents (codes <= 3 N).  8 codes per
// thread: two 128-bit loads, one 32-bit store; n is even.
__global__ void __launch_bounds__(256) narrow_codes4_kernel(const int32_t *__restrict__ src, uint8_t *__restrict__ dst, long long n) {
  const long long n8 = n >> 3;
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x; q < n8; q += stride) {
    const int4 *s = reinterpret_cast<const int4 *>(src) + 2 * q;
    const int4 a = s[0], b = s[1];
    reinterpret_cast<uint32_t *>(dst)[q] = (uint32_t)(a.x & 15) | ((uint32_t)(a.y & 15) << 4) | ((uint32_t)(a.z & 15) << 8) | ((uint32_t)(a.w & 15) << 12) |
                                           ((uint32_t)(b.x & 15) << 16) | ((uint32_t)(b.y & 15) << 20) | ((uint32_t)(b.z & 15) << 24) | ((uint32_t)(b.w & 15) << 28);
  }
  const long long t = (n8 << 3) + 2 * ((long long)blockIdx.x * blockDim.x + threadIdx.x);  // the last n % 8 codes, a pair per thread
  if (t + 1 < n) dst[t >> 1] = (uint8_t)((src[t] & 15) | ((src[t + 1] & 15) << 4));
}

// src and dst 16-byte aligned; bits = 8 (a code per byte) or 4 (two per byte, n even)
int launch_narrow_codes(const int32_t *src, uint8_t *dst, int64_t n, cudaStream_t stream, int bits) {
  if (n <= 0) return RBG_OK;
  if (bits == 4) {
    int64_t ctas4 = ((n >> 3) + 255) / 256;
    const int64_t cap4 = (int64_t)device_sm_count() * 8;
    if (ctas4 > cap4) ctas4 = cap4;
    if (ctas4 < 1) ctas4 = 1;
    return launch_kernel(narrow_codes4_kernel, (unsigned)ctas4, 256, 0, stream, -1, "narrow_codes4_kernel", false, src, dst, (long long)n);
  }
  int64_t ctas = ((n >> 4) + 255) / 256;
  const int64_t cap = (int64_t)device_sm_count() * 8;
  if (ctas > cap) ctas = cap;
  if (ctas < 1) ctas = 1;
  return launch_kernel(narrow_codes_kernel, (unsigned)ctas, 256, 0, stream, -1, "narrow_codes_kernel", false, src, dst, (long long)n);
}

// The last node of a device-side evaluation loop's body: counts the iteration and sets the WHILE node's condition.
// max_steps bounds the loop whatever the count says.
__global__ void __launch_bounds__(1) eval_loop_cond_kernel(cudaGraphConditionalHandle cond, const int32_t *__restrict__ live_count,
                                                           int32_t *__restrict__ steps, int max_steps) {
  const int s = ++*steps;
  cudaGraphSetConditional(cond, (*live_count > 0 && s < max_steps) ? 1u : 0u);
}

int launch_eval_loop_cond(unsigned long long cond, const int32_t *live_count, int32_t *steps, int max_steps, cudaStream_t stream) {
  return launch_kernel(eval_loop_cond_kernel, 1, 1, 0, stream, RBG_K_EVAL_LOOP, "eval_loop_cond_kernel", false, (cudaGraphConditionalHandle)cond,
                       live_count, steps, max_steps);
}

}  // namespace rbg
