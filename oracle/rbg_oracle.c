/*
 * rbg_oracle.c -- CPU ORACLE (TEST INFRASTRUCTURE, NOT PRODUCT CODE).
 * See rbg_oracle.h for the scope, the pinning status and the citation key.
 *
 * Style: one small function per reference function, same order of
 * evaluation, same quirks; no cleverness.  int32 everywhere the reference
 * uses `int` with x64 disabled.
 */
#include "rbg_oracle.h"

#include <math.h>
#include <stdlib.h>
#include <string.h>
#ifdef _OPENMP
#include <omp.h>
#endif

enum { EMPTY = 0, PATH = 1, POSITION = 2, TARGET = 3 };
enum { NOOP = 0, UP = 1, RIGHT = 2, DOWN = 3, LEFT = 4 };

/* ======================================================================== */
/* jax.random, jax==0.4.8 (requirements.txt:4), threefry_partitionable=False */
/* ======================================================================== */

static inline uint32_t rotl32(uint32_t x, int r) {
  return (x << r) | (x >> (32 - r));
}

/* jax/_src/prng.py threefry2x32 (Random123 Threefry-2x32, 20 rounds). */
void orc_threefry2x32(uint32_t k0, uint32_t k1, uint32_t x0, uint32_t x1,
                      uint32_t *o0, uint32_t *o1) {
  static const int R0[4] = {13, 15, 26, 6};
  static const int R1[4] = {17, 29, 16, 24};
  uint32_t ks[3] = {k0, k1, k0 ^ k1 ^ 0x1BD11BDAu};
  x0 += ks[0];
  x1 += ks[1];
  for (int g = 0; g < 5; ++g) {
    const int *R = (g & 1) ? R1 : R0;
    for (int i = 0; i < 4; ++i) {
      x0 += x1;
      x1 = rotl32(x1, R[i]);
      x1 ^= x0;
    }
    x0 += ks[(g + 1) % 3];
    x1 += ks[(g + 2) % 3] + (uint32_t)(g + 1);
  }
  *o0 = x0;
  *o1 = x1;
}

void orc_prng_key(uint64_t seed, uint32_t key[2]) {
  key[0] = (uint32_t)(seed >> 32);
  key[1] = (uint32_t)(seed & 0xffffffffu);
}

/* threefry_2x32(key, iota(n)): odd n is padded with one 0, the counter array
 * is cut into halves x0 = [0,h), x1 = [h,2h), out = concat(o0, o1)[:n]. */
static void tf_iota(const uint32_t key[2], int64_t n, uint32_t *out) {
  int64_t h = (n + 1) / 2;
  for (int64_t j = 0; j < h; ++j) {
    uint32_t c1 = (j + h < n) ? (uint32_t)(j + h) : 0u; /* the pad */
    uint32_t a, b;
    orc_threefry2x32(key[0], key[1], (uint32_t)j, c1, &a, &b);
    out[j] = a;
    if (j + h < n) out[j + h] = b;
  }
}

/* jax.random.split(key, num) = threefry(key, iota(2*num)).reshape(num, 2) */
void orc_split(const uint32_t key[2], int num, uint32_t *out) {
  tf_iota(key, 2 * (int64_t)num, out);
}

/* _random_bits(key, 32, (n,)) ; shape () is n = 1 */
void orc_random_bits(const uint32_t key[2], int n, uint32_t *out) {
  tf_iota(key, n, out);
}

static inline float bits_to_uniform(uint32_t bits) {
  uint32_t fb = (bits >> 9) | 0x3F800000u;
  float f;
  memcpy(&f, &fb, 4);
  return f - 1.0f;
}

/* jax.random.uniform(key, (), float32) in [0,1) */
float orc_uniform(const uint32_t key[2]) {
  uint32_t b;
  orc_random_bits(key, 1, &b);
  return bits_to_uniform(b);
}

static int cmp_u64(const void *a, const void *b) {
  uint64_t x = *(const uint64_t *)a, y = *(const uint64_t *)b;
  return (x > y) - (x < y);
}

/* jax.random._shuffle(key, arange(n), 0): rounds of
 * `key, sub = split(key); sort_key_val(random_bits(sub, (n,)), x)` with a
 * STABLE sort (lax.sort default). */
void orc_shuffle_iota(const uint32_t key_in[2], int n, int32_t *out) {
  uint32_t key[2] = {key_in[0], key_in[1]};
  for (int i = 0; i < n; ++i) out[i] = i;
  if (n <= 1) return;
  int rounds = (int)ceil(3.0 * log((double)n) / log(4294967295.0));
  uint32_t *bits = (uint32_t *)malloc(sizeof(uint32_t) * (size_t)n);
  uint64_t *comp = (uint64_t *)malloc(sizeof(uint64_t) * (size_t)n);
  int32_t *tmp = (int32_t *)malloc(sizeof(int32_t) * (size_t)n);
  for (int r = 0; r < rounds; ++r) {
    uint32_t ks[4];
    orc_split(key, 2, ks);
    key[0] = ks[0];
    key[1] = ks[1];
    orc_random_bits(&ks[2], n, bits);
    /* stable: ties on the 32-bit sort key keep the current order */
    for (int i = 0; i < n; ++i) comp[i] = ((uint64_t)bits[i] << 32) | (uint32_t)i;
    qsort(comp, (size_t)n, sizeof(uint64_t), cmp_u64);
    for (int i = 0; i < n; ++i) tmp[i] = out[(uint32_t)(comp[i] & 0xffffffffu)];
    memcpy(out, tmp, sizeof(int32_t) * (size_t)n);
  }
  free(bits);
  free(comp);
  free(tmp);
}

/* jax.random.randint int32: two 32-bit draws, multiplier trick. */
static inline int32_t randint_from_bits(uint32_t hi_bits, uint32_t lo_bits,
                                        int32_t lo, int32_t hi) {
  uint32_t span = (uint32_t)(hi - lo);
  if (hi <= lo) span = 1;
  uint32_t mult = (uint32_t)(65536u % span);
  /* jax squares in the span's dtype, uint32: for span > 2^16 the square 2^32
   * wraps to 0, so the value is lo + lo_bits % span. */
  mult = (mult * mult) % span;
  uint32_t off = (hi_bits % span) * mult + (lo_bits % span); /* uint32 wrap */
  off = off % span;
  return lo + (int32_t)off;
}

void orc_randint_vec(const uint32_t key[2], int n, int32_t lo, int32_t hi,
                     int32_t *out) {
  uint32_t ks[4];
  orc_split(key, 2, ks);
  uint32_t *hb = (uint32_t *)malloc(sizeof(uint32_t) * (size_t)n * 2);
  uint32_t *lb = hb + n;
  orc_random_bits(&ks[0], n, hb);
  orc_random_bits(&ks[2], n, lb);
  for (int i = 0; i < n; ++i) out[i] = randint_from_bits(hb[i], lb[i], lo, hi);
  free(hb);
}

int32_t orc_randint(const uint32_t key[2], int32_t lo, int32_t hi) {
  int32_t v;
  orc_randint_vec(key, 1, lo, hi, &v);
  return v;
}

/* jax.random.choice(key, a[4], (), replace=True, p=mask):
 *   p_cuml = cumsum(float32(p)); r = p_cuml[-1] * (1 - uniform(key));
 *   ind = searchsorted(p_cuml, r)  (side='left' = #(p_cuml < r)) */
int32_t orc_choice_p4(const uint32_t key[2], const int32_t a[4],
                      const uint8_t p[4]) {
  float pc[4];
  float acc = 0.0f;
  for (int i = 0; i < 4; ++i) {
    acc = acc + (p[i] ? 1.0f : 0.0f);
    pc[i] = acc;
  }
  volatile float one_minus_u = 1.0f - orc_uniform(key);
  volatile float r = pc[3] * one_minus_u;
  int ind = 0;
  for (int i = 0; i < 4; ++i) ind += (pc[i] < r);
  if (ind > 3) ind = 3; /* gather clamps; unreachable since r <= pc[3] */
  return a[ind];
}

/* ======================================================================== */
/* ParallelRandomWalk  (PRW:49-447)                                          */
/* ======================================================================== */

/* floor divmod as jnp.divmod */
static inline void fdivmod(int a, int b, int *q, int *r) {
  int qq = a / b, rr = a % b;
  if (rr != 0 && ((rr < 0) != (b < 0))) {
    qq -= 1;
    rr += b;
  }
  *q = qq;
  *r = rr;
}

/* gather with jnp semantics: negative indices wrap once, then clamp */
static inline int32_t gather2(const int32_t *grid, int G, int r, int c) {
  if (r < 0) r += G;
  if (c < 0) c += G;
  if (r < 0) r = 0;
  if (r > G - 1) r = G - 1;
  if (c < 0) c = 0;
  if (c > G - 1) c = G - 1;
  return grid[r * G + c];
}

/* PRW:262-291 _adjacent_cells: order up, down, left, right; -1 padding.
 * (strides by rows, divmods by cols: square grids only) */
void orc_prw_adjacent_cells(int G, int cell, int32_t out[4]) {
  const int dirs[4] = {-G, G, -1, 1};
  int r0, c0;
  fdivmod(cell, G, &r0, &c0);
  for (int i = 0; i < 4; ++i) {
    int c = cell + dirs[i];
    int ok = (0 <= c) && (c < G * G);
    int r, cc;
    fdivmod(c, G, &r, &cc);
    ok = ok && (r == r0 || cc == c0);
    out[i] = ok ? c : -1;
  }
}

/* PRW:321-338 _is_cell_free */
int orc_prw_is_cell_free(int G, const int32_t *grid, int cell) {
  int r, c;
  fdivmod(cell, G, &r, &c);
  int32_t v = gather2(grid, G, r, c);
  return (cell == -1) ? 0 : (v == 0);
}

/* PRW:340-374 _is_cell_doubling_back: True when the candidate touches the
 * wire at most once. */
static int prw_not_doubling_back(int G, const int32_t *grid, int wire_id,
                                 int cell) {
  int32_t adj[4];
  orc_prw_adjacent_cells(G, cell, adj);
  int sum = 0;
  for (int i = 0; i < 4; ++i) {
    int r, c;
    fdivmod(adj[i], G, &r, &c);
    int32_t v = gather2(grid, G, r, c);
    int touching = (v == 3 * wire_id + POSITION) || (v == 3 * wire_id + PATH) ||
                   (v == 3 * wire_id + TARGET);
    sum += (adj[i] == -1) ? 0 : touching;
  }
  return sum > 1 ? 0 : 1;
}

/* PRW:293-319 _available_cells */
void orc_prw_available_cells(int G, const int32_t *grid, int cell,
                             int32_t out[4]) {
  int32_t adj[4];
  orc_prw_adjacent_cells(G, cell, adj);
  int r, c;
  fdivmod(cell, G, &r, &c);
  int32_t value = gather2(grid, G, r, c);
  int q, rem;
  fdivmod(value - 1, 3, &q, &rem);
  int wire_id = q;
  for (int i = 0; i < 4; ++i) {
    int free_ = orc_prw_is_cell_free(G, grid, adj[i]);
    int ok = prw_not_doubling_back(G, grid, wire_id, adj[i]);
    out[i] = (free_ && ok) ? adj[i] : -1;
  }
}

/* PRW:238-260 _action_from_positions / _action_from_tuple */
int orc_prw_action_from_positions(int G, int p1, int p2) {
  int r1, c1, r2, c2;
  fdivmod(p1, G, &r1, &c1);
  fdivmod(p2, G, &r2, &c2);
  int dr = r2 - r1, dc = c2 - c1;
  int a = 0;
  a += (dr == -1 && dc == 0) * UP;
  a += (dr == 1 && dc == 0) * DOWN;
  a += (dr == 0 && dc == -1) * LEFT;
  a += (dr == 0 && dc == 1) * RIGHT;
  a += (dr == 0 && dc == 0) * NOOP;
  return a;
}

/* jumanji connector utils.move_position: lax.switch clamps the index */
static inline void move_position(int r, int c, int action, int *nr, int *nc) {
  if (action < 0) action = 0;
  if (action > 4) action = 4;
  static const int dr[5] = {0, -1, 0, 1, 0};
  static const int dc[5] = {0, 0, 1, 0, -1};
  *nr = r + dr[action];
  *nc = c + dc[action];
}

/* PRW:401-429 _is_valid_position == jumanji utils.is_valid_position */
static inline int is_valid_position(int G, const int32_t *grid, int agent_id,
                                    int connected, int row, int col) {
  int in_bounds = (0 <= row) && (row < G) && (0 <= col) && (col < G);
  int32_t v = gather2(grid, G, row, col);
  int open_cell = (v == EMPTY) || (v == 3 * agent_id + TARGET);
  return in_bounds && open_cell && !connected;
}

/* PRW:101-145 _step_agents with the actions supplied (also jumanji
 * Connector._step_agents).  Every agent moves on a private copy of `grid`,
 * the copies are max-joined, an agent whose head value is absent from the
 * join has collided and is put back (get_correction_mask: +1 on its old
 * head cell, which the join holds as PATH).  Returns #collided. */
static int step_agents_with_actions(int G, int N, int32_t *grid,
                                    const int32_t *target /* [N,2] or NULL */,
                                    int32_t *pos /* [N,2] */,
                                    const int32_t *actions) {
  const int cells = G * G;
  int32_t *joined = (int32_t *)calloc((size_t)cells, sizeof(int32_t));
  int32_t *priv = (int32_t *)malloc(sizeof(int32_t) * (size_t)cells);
  int32_t newpos[ORC_MAX_N][2];
  for (int i = 0; i < N; ++i) {
    int r = pos[2 * i], c = pos[2 * i + 1];
    int connected = target ? (r == target[2 * i] && c == target[2 * i + 1]) : 0;
    int nr, nc;
    move_position(r, c, actions[i], &nr, &nc);
    int ok = is_valid_position(G, grid, i, connected, nr, nc) &&
             (actions[i] != NOOP);
    memcpy(priv, grid, sizeof(int32_t) * (size_t)cells);
    newpos[i][0] = r;
    newpos[i][1] = c;
    if (ok) { /* move_agent */
      priv[r * G + c] = 3 * i + PATH;
      priv[nr * G + nc] = 3 * i + POSITION;
      newpos[i][0] = nr;
      newpos[i][1] = nc;
    }
    /* get_agent_grid + max join */
    for (int k = 0; k < cells; ++k) {
      int32_t v = priv[k];
      int32_t own = (v == 3 * i + POSITION || v == 3 * i + TARGET ||
                     v == 3 * i + PATH) ? v : 0;
      if (own > joined[k]) joined[k] = own;
    }
  }
  int collided_total = 0;
  int32_t *corr = (int32_t *)calloc((size_t)cells, sizeof(int32_t));
  for (int i = 0; i < N; ++i) {
    int present = 0;
    for (int k = 0; k < cells; ++k) present |= (joined[k] == 3 * i + POSITION);
    int collided = !present;
    if (collided) {
      for (int k = 0; k < cells; ++k) corr[k] += (grid[k] == 3 * i + POSITION);
      collided_total++;
    } else {
      pos[2 * i] = newpos[i][0];
      pos[2 * i + 1] = newpos[i][1];
    }
  }
  for (int k = 0; k < cells; ++k) grid[k] = joined[k] + corr[k];
  free(joined);
  free(priv);
  free(corr);
  return collided_total;
}

/* PRW:147-190 _initialise_agents */
void orc_prw_initialise_agents(const uint32_t key[2], int G, int N,
                               int32_t *grid, int32_t *pos) {
  int32_t *perm = (int32_t *)malloc(sizeof(int32_t) * (size_t)(G * G));
  orc_shuffle_iota(key, G * G, perm); /* choice(replace=False) = permutation[:N] */
  memset(grid, 0, sizeof(int32_t) * (size_t)(G * G));
  for (int i = 0; i < N; ++i) {
    int r, c;
    fdivmod(perm[i], G, &r, &c);
    pos[2 * i] = r;
    pos[2 * i + 1] = c;
    int32_t v = 3 * i + POSITION;
    if (v > grid[r * G + c]) grid[r * G + c] = v; /* max over per-agent grids */
  }
  free(perm);
}

/* PRW:192-203 */
int orc_prw_continue_stepping(int G, int N, const int32_t *grid,
                              const int32_t *pos) {
  int all_done = 1;
  for (int i = 0; i < N; ++i) {
    int32_t av[4];
    orc_prw_available_cells(G, grid, pos[2 * i] * G + pos[2 * i + 1], av);
    int done = (av[0] == -1 && av[1] == -1 && av[2] == -1 && av[3] == -1);
    all_done = all_done && done;
  }
  return !all_done;
}

/* PRW:92-99 _step (+ :205-230 _select_action) */
int orc_prw_step(const uint32_t key[2], int G, int N, int32_t *grid,
                 int32_t *pos, int32_t *actions_out, uint32_t next_key[2]) {
  uint32_t keys[2 * ORC_MAX_N];
  int32_t actions[ORC_MAX_N];
  orc_split(key, N, keys);
  for (int i = 0; i < N; ++i) {
    int cell = pos[2 * i] * G + pos[2 * i + 1];
    int32_t av[4];
    uint8_t p[4];
    orc_prw_available_cells(G, grid, cell, av);
    for (int k = 0; k < 4; ++k) p[k] = (av[k] != -1);
    int32_t dest = orc_choice_p4(&keys[2 * i], av, p);
    actions[i] = orc_prw_action_from_positions(G, cell, dest);
  }
  int coll = step_agents_with_actions(G, N, grid, NULL, pos, actions);
  if (actions_out) memcpy(actions_out, actions, sizeof(int32_t) * (size_t)N);
  uint32_t ks[4];
  orc_split(key, 2, ks);
  next_key[0] = ks[2];
  next_key[1] = ks[3];
  return coll;
}

/* PRW:60-90 generate_board */
int orc_prw_generate(const uint32_t key[2], int G, int N, int32_t *heads,
                     int32_t *targets, int32_t *solved, int32_t *stats) {
  if (G < 2 || G > ORC_MAX_G || N < 1 || N > ORC_MAX_N || N > G * G) return -1;
  uint32_t ks[4];
  orc_split(key, 2, ks); /* key, step_key = split(key) */
  int32_t start[2 * ORC_MAX_N], pos[2 * ORC_MAX_N];
  orc_prw_initialise_agents(&ks[0], G, N, solved, pos);
  memcpy(start, pos, sizeof(int32_t) * 2 * (size_t)N);
  uint32_t k[2] = {ks[2], ks[3]};
  int trips = 0, colls = 0;
  while (orc_prw_continue_stepping(G, N, solved, pos)) {
    uint32_t nk[2];
    colls += orc_prw_step(k, G, N, solved, pos, NULL, nk);
    k[0] = nk[0];
    k[1] = nk[1];
    trips++;
  }
  for (int i = 0; i < N; ++i) { /* heads = start.T, targets = position.T */
    heads[i] = start[2 * i];
    heads[N + i] = start[2 * i + 1];
    targets[i] = pos[2 * i];
    targets[N + i] = pos[2 * i + 1];
  }
  /* PRW:435-447: heads first, then targets */
  for (int i = 0; i < N; ++i) solved[start[2 * i] * G + start[2 * i + 1]] = 3 * i + POSITION;
  for (int i = 0; i < N; ++i) solved[pos[2 * i] * G + pos[2 * i + 1]] = 3 * i + TARGET;
  if (stats) {
    stats[0] = trips;
    stats[1] = colls;
  }
  return 0;
}

/* ======================================================================== */
/* SeedExtension (SE:93-304, PPU:24-195,200-234,283-429, GU:59-178,491-612)  */
/* ======================================================================== */

/* PPU:373-407 position_to_wire_num_jax: -1 when empty or out of bounds */
static inline int se_wire_num(int G, const int32_t *b, int r, int c) {
  if (!(0 <= r && r < G && 0 <= c && c < G)) return -1;
  int32_t v = b[r * G + c];
  return v == 0 ? -1 : (v - 1) / 3;
}

/* PPU:411-429 */
static inline int se_cell_type(int32_t v) { return v == 0 ? 0 : ((v - 1) % 3) + 1; }

/* PPU:283-317 */
static inline int se_num_adj(int G, const int32_t *b, int r, int c, int wire) {
  return (se_wire_num(G, b, r - 1, c) == wire) + (se_wire_num(G, b, r + 1, c) == wire) +
         (se_wire_num(G, b, r, c - 1) == wire) + (se_wire_num(G, b, r, c + 1) == wire);
}

#define SE_INVALID (-999)

/* SE:93-147 return_seeded_board. The SAME key feeds randint, choice (heads)
 * and choice (offsets). */
int orc_seedext_seeded_board(const uint32_t key[2], int G, int N, int32_t *board) {
  int side = orc_randint(key, 0, 2);
  int lo = side ? 1 : 0;
  int cnt = 0; /* len(arange(1,G,2)) or len(arange(0,G-1,2)) */
  for (int v = lo; v < (side ? G : G - 1); v += 2) cnt++;
  int K = cnt * cnt;
  if (N > K) return -2; /* jax raises at trace time */
  int32_t *perm = (int32_t *)malloc(sizeof(int32_t) * (size_t)K);
  int32_t offs[ORC_MAX_N];
  orc_shuffle_iota(key, K, perm);      /* choice(key, index_choice, (N,), replace=False) */
  orc_randint_vec(key, N, 0, 2, offs); /* choice(key, offset_array, (N,)) */
  memset(board, 0, sizeof(int32_t) * (size_t)(G * G));
  static const int off_one[2][2] = {{-1, 0}, {0, -1}};
  static const int off_other[2][2] = {{0, 1}, {1, 0}};
  int hr[ORC_MAX_N], hc[ORC_MAX_N], tr[ORC_MAX_N], tc[ORC_MAX_N];
  for (int i = 0; i < N; ++i) {
    int idx = perm[i];
    hr[i] = lo + 2 * (idx / cnt);
    hc[i] = lo + 2 * (idx % cnt);
    const int *o = side ? off_one[offs[i]] : off_other[offs[i]];
    tr[i] = hr[i] + o[0];
    tc[i] = hc[i] + o[1];
  }
  for (int i = 0; i < N; ++i) board[hr[i] * G + hc[i]] = 3 * i + TARGET;
  for (int i = 0; i < N; ++i) board[tr[i] * G + tc[i]] = 3 * i + POSITION;
  free(perm);
  return 0;
}

static void flip_rows(int G, int32_t *b) {
  for (int r = 0; r < G / 2; ++r)
    for (int c = 0; c < G; ++c) {
      int32_t t = b[r * G + c];
      b[r * G + c] = b[(G - 1 - r) * G + c];
      b[(G - 1 - r) * G + c] = t;
    }
}
static void flip_cols(int G, int32_t *b) {
  for (int r = 0; r < G; ++r)
    for (int c = 0; c < G / 2; ++c) {
      int32_t t = b[r * G + c];
      b[r * G + c] = b[r * G + (G - 1 - c)];
      b[r * G + (G - 1 - c)] = t;
    }
}

/* PPU:24-195 extend_wires_jax */
void orc_extend_wires(int G, int32_t *board, const uint32_t key_in[2],
                      float randomness, int two_sided, int64_t ext_steps,
                      int32_t *sweeps_out) {
  const int cells = G * G;
  uint32_t key[2] = {key_in[0], key_in[1]};
  int32_t *prev = (int32_t *)malloc(sizeof(int32_t) * (size_t)cells);
  memcpy(prev, board, sizeof(int32_t) * (size_t)cells);
  prev[0] += 1; /* PPU:47 */
  int64_t step_num = 0;
  while (memcmp(prev, board, sizeof(int32_t) * (size_t)cells) != 0 &&
         (ext_steps < 0 || step_num < ext_steps)) {
    step_num++;
    uint32_t ks[6];
    orc_split(key, 3, ks); /* key, flipkey, flopkey */
    key[0] = ks[0];
    key[1] = ks[1];
    int do_flip = (orc_randint(&ks[2], 0, 2) == 0); /* choice over [True, False] */
    int do_flop = (orc_randint(&ks[4], 0, 2) == 0);
    if (do_flip) flip_rows(G, board);
    if (do_flop) flip_cols(G, board);
    memcpy(prev, board, sizeof(int32_t) * (size_t)cells); /* the FLIPPED copy */
    for (int row = 0; row < G; ++row) {
      for (int col = 0; col < G; ++col) {
        /* PPU:322-369 candidates in order up, left, down, right */
        int list[4][2];
        const int cand[4][2] = {{row - 1, col}, {row, col - 1}, {row + 1, col}, {row, col + 1}};
        for (int k = 0; k < 4; ++k) {
          int r = cand[k][0], c = cand[k][1];
          int inb = (k == 0) ? (r >= 0) : (k == 1) ? (c >= 0) : (k == 2) ? (r < G) : (c < G);
          int open_ = inb && board[r * G + c] == EMPTY;
          list[k][0] = open_ ? r : SE_INVALID;
          list[k][1] = open_ ? c : SE_INVALID;
        }
        int cur_wire = se_wire_num(G, board, row, col);
        for (int k = 0; k < 4; ++k) { /* PPU:86-97 */
          int na = se_num_adj(G, board, list[k][0], list[k][1], cur_wire);
          if (na > 1) list[k][0] = list[k][1] = SE_INVALID;
        }
        /* PPU:200-234 get_previous_neighbor_jax: only up, down, left */
        int prev_r = SE_INVALID, prev_c = SE_INVALID;
        const int nb[3][2] = {{row - 1, col}, {row + 1, col}, {row, col - 1}};
        for (int k = 0; k < 3; ++k) {
          int r = nb[k][0], c = nb[k][1];
          int inb = (r >= 0 && r < G && c >= 0 && c < G);
          if (inb && se_wire_num(G, board, r, c) == cur_wire) {
            prev_r = r;
            prev_c = c;
          }
        }
        int pri_r = row + (row - prev_r), pri_c = col + (col - prev_c);
        int ctype = se_cell_type(board[row * G + col]);
        int extendable = two_sided ? (ctype == POSITION || ctype == TARGET) : (ctype == TARGET);
        if (!extendable)
          for (int k = 0; k < 4; ++k) list[k][0] = list[k][1] = SE_INVALID;
        int stop = 1;
        for (int k = 0; k < 4; ++k) stop = stop && (list[k][0] == SE_INVALID && list[k][1] == SE_INVALID);
        if (stop)
          for (int k = 0; k < 4; ++k) {
            list[k][0] = row;
            list[k][1] = col;
          }
        /* PPU:127-144 random pick until valid, from `key` without advancing it */
        int ext_r = SE_INVALID, ext_c = SE_INVALID;
        uint32_t lk[2] = {key[0], key[1]};
        while (ext_r == SE_INVALID && ext_c == SE_INVALID) {
          uint32_t s2[4];
          orc_split(lk, 2, s2);
          lk[0] = s2[0];
          lk[1] = s2[1];
          int ind = orc_randint(&s2[2], 0, 4);
          ext_r = list[ind][0];
          ext_c = list[ind][1];
        }
        int pri_avail = 0;
        for (int k = 0; k < 4; ++k) pri_avail |= (list[k][0] == pri_r && list[k][1] == pri_c);
        uint32_t s3[4];
        orc_split(key, 2, s3); /* key, random_key = split(key) */
        key[0] = s3[0];
        key[1] = s3[1];
        int use_random = randomness > orc_uniform(&s3[2]);
        if (pri_avail && !use_random) {
          ext_r = pri_r;
          ext_c = pri_c;
        }
        board[ext_r * G + ext_c] = board[row * G + col];
        int ct2 = se_cell_type(board[row * G + col]);
        int offset = stop ? 0 : (PATH - ct2);
        board[row * G + col] += offset;
      }
    }
    if (do_flip) flip_rows(G, board);
    if (do_flop) flip_cols(G, board);
  }
  if (sweeps_out) *sweeps_out = (int32_t)step_num;
  free(prev);
}

/* GU:491-612 optimise_wire (+ GU:59-178 update_queue_and_visited,
 * GU:186-224 get_path, GU:242-260 remove_path, GU:299-346 jax_fill_grid).
 * Returns 0, or 1 if the degenerate branch (queue ran dry / end not reached)
 * was hit -- never observed for boards made by this pipeline. */
int orc_optimise_wire(const uint32_t key[2], int G, int32_t *board, int wire,
                      int32_t *pops_out) {
  const int cells = G * G;
  const int32_t start_num = 3 * wire + POSITION, end_num = 3 * wire + TARGET,
                path_num = 3 * wire + PATH;
  int flat_start = 0, flat_end = 0;
  for (int k = cells - 1; k >= 0; --k) { /* argmax -> first index of the max */
    if (board[k] == start_num) flat_start = k;
    if (board[k] == end_num) flat_end = k;
  }
  board[flat_start] = path_num;
  board[flat_end] = path_num;
  int32_t *queue = (int32_t *)calloc((size_t)cells, sizeof(int32_t));
  int32_t *visited = (int32_t *)malloc(sizeof(int32_t) * (size_t)cells);
  int32_t *path = (int32_t *)malloc(sizeof(int32_t) * (size_t)cells);
  for (int k = 0; k < cells; ++k) visited[k] = -1, path[k] = -1;
  queue[flat_start] = 1;
  int32_t perm[4];
  orc_shuffle_iota(key, 4, perm); /* GU:91 permutation(key, arange(4), independent=True) */
  static const int drow[4] = {-1, 0, 1, 0}, dcol[4] = {0, 1, 0, -1};
  int degenerate = 0, pops = 0;
  for (int it = 0; it < cells && visited[flat_end] == -1; ++it) {
    int cur = 0;
    int32_t best = 0;
    for (int k = 0; k < cells; ++k) /* argmin over positive entries, first index */
      if (queue[k] > 0 && (best == 0 || queue[k] < best)) {
        best = queue[k];
        cur = k;
      }
    if (best == 0) { /* all inf -> argmin 0; max over -inf -> INT_MIN order number */
      degenerate = 1;
      cur = 0;
    }
    int cr = cur / G, cc = cur % G;
    for (int j = 0; j < 4; ++j) {
      int nr = cr + drow[perm[j]], nc = cc + dcol[perm[j]];
      int inb = (0 <= nr && nr < G && 0 <= nc && nc < G);
      if (!inb) continue;
      int p = nr * G + nc;
      int ok = visited[p] == -1 && queue[p] == 0 &&
               (board[p] == path_num || board[p] == EMPTY);
      if (!ok) continue;
      int32_t mx = 0;
      int any = 0;
      for (int k = 0; k < cells; ++k)
        if (queue[k] > 0 && (!any || queue[k] > mx)) {
          mx = queue[k];
          any = 1;
        }
      queue[p] = any ? mx + 1 : INT32_MIN;
      visited[p] = cur;
    }
    queue[cur] = 0;
    pops++;
  }
  if (pops_out) *pops_out = pops;
  if (visited[flat_end] == -1) { /* unreachable for pipeline boards */
    board[flat_start] = start_num;
    board[flat_end] = end_num;
    free(queue);
    free(visited);
    free(path);
    return 1;
  }
  int n = 0, cur = flat_end;
  while (n == 0 || path[n - 1] != flat_start) {
    path[n++] = cur;
    cur = visited[cur];
    if (n >= cells) break;
  }
  for (int k = 0; k < cells; ++k)
    if (board[k] == path_num) board[k] = 0;
  for (int k = 0; k < n; ++k) board[path[k]] = path_num;
  board[path[n - 1]] = start_num;
  board[path[0]] = end_num;
  free(queue);
  free(visited);
  free(path);
  return degenerate;
}

/* SE:149-227 return_solved_board */
int orc_seedext_solved(const uint32_t key_in[2], int G, int N, float randomness,
                       int two_sided, int iterations, int64_t ext_steps,
                       int32_t *board, int32_t *stats) {
  if (G < 2 || G > ORC_MAX_G || N < 1 || N > ORC_MAX_N) return -1;
  uint32_t ks[4];
  orc_split(key_in, 2, ks); /* key, seedkey */
  uint32_t key[2] = {ks[0], ks[1]};
  int rc = orc_seedext_seeded_board(&ks[2], G, N, board);
  if (rc) return rc;
  int wires = N > (G * G) / 3 ? (G * G) / 3 : N; /* SE:60-63 */
  int sweeps_total = 0, pops_total = 0, degenerate = 0;
  for (int it = 0; it < iterations; ++it) {
    uint32_t k3[6];
    orc_split(key, 3, k3); /* key, extkey, optkey */
    key[0] = k3[0];
    key[1] = k3[1];
    int32_t sweeps = 0;
    orc_extend_wires(G, board, &k3[2], randomness, two_sided, ext_steps, &sweeps);
    sweeps_total += sweeps;
    uint32_t optkeys[2 * ORC_MAX_N];
    orc_split(&k3[4], wires, optkeys);
    for (int w = 0; w < wires; ++w) {
      int32_t pops = 0;
      degenerate |= orc_optimise_wire(&optkeys[2 * w], G, board, w, &pops);
      pops_total += pops;
    }
  }
  if (stats) {
    stats[0] = sweeps_total;
    stats[1] = pops_total;
    stats[2] = degenerate;
  }
  return 0;
}

/* SE:257-304 generate_starts_ends: first POSITION / TARGET cell per wire in
 * row-major order, (0,0) when absent (argwhere(size=2) fill value 0). */
int orc_seedext_starts_ends(const uint32_t key[2], int G, int N, float randomness,
                            int two_sided, int iterations, int64_t ext_steps,
                            int32_t *starts, int32_t *ends) {
  int32_t *board = (int32_t *)malloc(sizeof(int32_t) * (size_t)(G * G));
  int rc = orc_seedext_solved(key, G, N, randomness, two_sided, iterations, ext_steps, board, NULL);
  if (rc) {
    free(board);
    return rc;
  }
  for (int w = 0; w < N; ++w) {
    int s = 0, e = 0, fs = 0, fe = 0;
    for (int k = 0; k < G * G; ++k) {
      if (!fs && board[k] == 3 * w + POSITION) s = k, fs = 1;
      if (!fe && board[k] == 3 * w + TARGET) e = k, fe = 1;
    }
    starts[w] = s / G;
    starts[N + w] = s % G;
    ends[w] = e / G;
    ends[N + w] = e % G;
  }
  free(board);
  return 0;
}

/* ======================================================================== */
/* SequentialRandomWalkBoard  (SRW = routing_board_generation/board_generation_methods/
 *   jax_implementation/board_generation/sequential_random_walk.py)              */
/* ======================================================================== */
/* jax.random.choice(key, a, shape=(), replace=False, p) with p in {0,1}^n, as SRW:57-63 and :211-217
 * call it: jax 0.4.8 evaluates g = -gumbel(key, (n,)) - log(p) and takes argsort(g)[0] (stable).  log(1) = 0 and
 * log(0) = -inf, so an entry with p = 0 gets g = +inf and an entry with p = 1 gets
 * g = log(-log(u)), u = uniform(key, (n,), minval=tiny, maxval=1) = max(tiny, m * 2^-23) with m the top 23 bits of
 * the entry's random word.  That map is decreasing in m, so the pick is the candidate with the LARGEST m, the
 * lowest index among equal m (stable sort).  The only assumption is that float32 log is strictly monotone over
 * the 2^23 values u takes and over their negated logs, so that two different m never tie: NumPy's is (checked
 * exhaustively by tests/tools/make_seqrw_fixtures.py, which also checks this integer rule against the float
 * formula on every draw of every fixture); XLA's cannot be run here.  Returns the index (0 when no entry has
 * p = 1: argsort of all +inf). */
static int choice_gumbel01(const uint32_t key[2], int n, const uint8_t *p) {
  uint32_t *bits = (uint32_t *)malloc(sizeof(uint32_t) * (size_t)(n + 1));
  orc_random_bits(key, n, bits);
  int best = -1;
  uint32_t bm = 0;
  for (int i = 0; i < n; ++i) {
    if (!p[i]) continue;
    uint32_t m = bits[i] >> 9;
    if (best < 0 || m > bm) best = i, bm = m;
  }
  free(bits);
  return best < 0 ? 0 : best;
}

/* SRW:85-113 adjacent_cells: [up, down, left, right] as flat indices, -1 when off the board */
static void seqrw_adjacent(int G, int cell, int out[4]) {
  int r = cell / G, c = cell % G;
  out[0] = r > 0 ? cell - G : -1;
  out[1] = r < G - 1 ? cell + G : -1;
  out[2] = c > 0 ? cell - 1 : -1;
  out[3] = c < G - 1 ? cell + 1 : -1;
}

/* SRW:115-140 available_cells: an adjacent cell is available when it is free (:142-156) and touches at most one
 * cell of the wire (:158-191; the cell the wire stands on is that one) */
static int seqrw_available(int G, const int32_t *board, int cell, int w, int out[4]) {
  int adj[4], any = 0;
  seqrw_adjacent(G, cell, adj);
  for (int k = 0; k < 4; ++k) {
    out[k] = -1;
    if (adj[k] < 0 || board[adj[k]] != 0) continue;
    int nb[4], touching = 0;
    seqrw_adjacent(G, adj[k], nb);
    for (int j = 0; j < 4; ++j)
      if (nb[j] >= 0 && board[nb[j]] >= 3 * w + 1 && board[nb[j]] <= 3 * w + 3) touching++;
    if (touching > 1) continue;
    out[k] = adj[k];
    any = 1;
  }
  return any;
}

/* SRW:290-322 add_agents with :34-83 pick_start, :193-228 one_step, :230-288 walk_randomly */
static int seqrw_add_agents(const uint32_t key_in[2], int G, int N, int max_length, int32_t *board, int32_t *steps_out) {
  const int cells = G * G;
  uint32_t key[2] = {key_in[0], key_in[1]};
  uint8_t *p = (uint8_t *)malloc((size_t)(cells > G + 1 ? cells : G + 1));
  int success = 1, steps = 0;
  memset(board, 0, sizeof(int32_t) * (size_t)cells);
  for (int w = 0; w < N; ++w) {
    uint32_t ks[4], ps[4];
    orc_split(key, 2, ks);     /* :307 key, subkey = split(key); that `key` is dropped (:306 reads the tuple's) */
    orc_split(&ks[2], 2, ps);  /* :51  key, subkey = split(key) inside pick_start(subkey) */
    key[0] = ps[0];
    key[1] = ps[1];            /* the tuple's key from here on */
    int can_start = 0;
    for (int i = 0; i < cells; ++i) can_start |= (p[i] = (uint8_t)(board[i] == 0));
    if (!can_start) {          /* :315 lambda x: (x, False) */
      success = 0;
      continue;
    }
    const int start = choice_gumbel01(&ps[2], cells, p); /* :57-63; divmod(flat, rows) :66 */
    board[start] = 3 * w + POSITION;                       /* :71 */
    int cur = start, moved = 0;
    for (int t = 0; t < max_length; ++t) {                 /* :280 fori_loop(0, max_length) */
      int avail[4];
      if (!seqrw_available(G, board, cur, w, avail)) break; /* can_step False: the board no longer changes */
      moved = 1;
      uint32_t ss[4];
      orc_split(key, 2, ss);                               /* :204 */
      key[0] = ss[0];
      key[1] = ss[1];
      /* :138-140 available_cells is padded with -1 to rows + 1 entries; choice draws one word per entry */
      memset(p, 0, (size_t)(G + 1));
      for (int k = 0; k < 4; ++k) p[k] = (uint8_t)(avail[k] >= 0);
      const int nxt = avail[choice_gumbel01(&ss[2], G + 1, p)]; /* :211-217 */
      board[nxt] = 3 * w + TARGET;                          /* :221 */
      board[cur] = 3 * w + PATH;                            /* :223-227 */
      cur = nxt;
      steps++;
    }
    board[start] = 3 * w + POSITION;                        /* :286 */
    success &= moved;                                       /* :319 */
  }
  free(p);
  if (steps_out) *steps_out = steps;
  return success;
}

/* SRW:324-392 generate: attempts with max_length = rows + cols - i, i = 1 .. rows + cols, ALL from the same key,
 * until one places every wire and moves it at least once; a zero board otherwise.  The reference returns the
 * codes as float32 (jnp.zeros default dtype, :350); they are given as int32 here.
 * stats (may be NULL): [0] = i of the attempt that succeeded (0 = none), [1] = its steps. */
int orc_seqrw_generate(const uint32_t key[2], int G, int N, int32_t *board, int32_t *stats) {
  if (G < 3 || G > ORC_MAX_G || N < 1 || N > ORC_MAX_N) return -1; /* :138-140 jnp.full(rows - 3) needs rows >= 3 */
  const int L0 = 2 * G;
  int success = 0, steps = 0, i;
  for (i = 1; i <= L0 && !success; ++i) success = seqrw_add_agents(key, G, N, L0 - i, board, &steps);
  if (!success) memset(board, 0, sizeof(int32_t) * (size_t)(G * G)); /* :389-391 */
  if (stats) {
    stats[0] = success ? i - 1 : 0;
    stats[1] = success ? steps : 0;
  }
  return 0;
}

/* SRW:394-431 generate_starts_ends: first POSITION / TARGET cell of every wire in row-major order, (0,0) when
 * absent (argwhere(size=2) fill value): starts[2,N], ends[2,N] */
int orc_seqrw_starts_ends(const uint32_t key[2], int G, int N, int32_t *starts, int32_t *ends) {
  int32_t *board = (int32_t *)malloc(sizeof(int32_t) * (size_t)(G * G));
  int rc = orc_seqrw_generate(key, G, N, board, NULL);
  if (rc) {
    free(board);
    return rc;
  }
  for (int w = 0; w < N; ++w) {
    int s = 0, e = 0, fs = 0, fe = 0;
    for (int k = 0; k < G * G; ++k) {
      if (!fs && board[k] == 3 * w + POSITION) s = k, fs = 1;
      if (!fe && board[k] == 3 * w + TARGET) e = k, fe = 1;
    }
    starts[w] = s / G;
    starts[N + w] = s % G;
    ends[w] = e / G;
    ends[N + w] = e % G;
  }
  free(board);
  return 0;
}

/* ======================================================================== */
/* Generator.__call__(key) -> State  (PRWG:46-77, UG:70-109, RSG:28-57)      */
/* ======================================================================== */
int orc_state(int kind, const uint32_t key_in[2], int G, int N, int32_t *grid,
              int32_t *step_count, int32_t *agent_id, int32_t *start,
              int32_t *target, int32_t *position, uint32_t key_out[2]) {
  if (G < 2 || G > ORC_MAX_G || N < 1 || N > ORC_MAX_N) return -1;
  uint32_t ks[4];
  orc_split(key_in, 2, ks); /* key, pos_key = split(key) */
  int32_t a[2 * ORC_MAX_N], b[2 * ORC_MAX_N]; /* [2,N] rows then cols */
  int rc = 0;
  if (kind == ORC_GEN_PRW) {
    int32_t *solved = (int32_t *)malloc(sizeof(int32_t) * (size_t)(G * G));
    rc = orc_prw_generate(&ks[0], G, N, a, b, solved, NULL);
    free(solved);
  } else if (kind == ORC_GEN_UNIFORM) {
    if (2 * N > G * G) return -2;
    int32_t *perm = (int32_t *)malloc(sizeof(int32_t) * (size_t)(G * G));
    orc_shuffle_iota(&ks[2], G * G, perm); /* choice(pos_key, arange(G*G), (2,N), replace=False) */
    for (int i = 0; i < N; ++i) {
      a[i] = perm[i] / G;
      a[N + i] = perm[i] % G;
      b[i] = perm[N + i] / G;
      b[N + i] = perm[N + i] % G;
    }
    free(perm);
  } else if (kind == ORC_GEN_SEEDEXT) {
    rc = orc_seedext_starts_ends(&ks[0], G, N, 0.0f, 1, 1, -1, a, b);
  } else if (kind == ORC_GEN_SEQRW) {
    /* rl_training/online_generators/sequential_random_walk_generator.py:36-62: key, pos_key = split(key);
     * generate_starts_ends(key); a failed generation leaves every pin at (0,0) and the scatters below
     * keep the last one */
    rc = orc_seqrw_starts_ends(&ks[0], G, N, a, b);
  } else {
    return -3;
  }
  if (rc) return rc;
  memset(grid, 0, sizeof(int32_t) * (size_t)(G * G));
  for (int i = 0; i < N; ++i) grid[a[i] * G + a[N + i]] = 3 * i + POSITION;
  for (int i = 0; i < N; ++i) grid[b[i] * G + b[N + i]] = 3 * i + TARGET;
  for (int i = 0; i < N; ++i) {
    agent_id[i] = i;
    start[2 * i] = a[i];
    start[2 * i + 1] = a[N + i];
    target[2 * i] = b[i];
    target[2 * i + 1] = b[N + i];
    position[2 * i] = a[i];
    position[2 * i + 1] = a[N + i];
  }
  *step_count = 0;
  key_out[0] = ks[0];
  key_out[1] = ks[1];
  return 0;
}

/* BoardDatasetGeneratorJAX.__call__ (rl_training/offline_generation/
 * dataset_generator_jax.py:112-141): key, _ = split(key); which = randint(key, (), 0, K);
 * State from heads[which] / targets[which] (each [2,N], rows then cols). */
int orc_dataset_state(const uint32_t key_in[2], int G, int N, const int32_t *heads,
                      const int32_t *targets, int64_t K, int32_t *grid,
                      int32_t *step_count, int32_t *agent_id, int32_t *start,
                      int32_t *target, int32_t *position, uint32_t key_out[2]) {
  uint32_t ks[4];
  orc_split(key_in, 2, ks);
  int32_t which = orc_randint(&ks[0], 0, (int32_t)K);
  const int32_t *h = heads + (size_t)which * 2 * N, *t = targets + (size_t)which * 2 * N;
  memset(grid, 0, sizeof(int32_t) * (size_t)(G * G));
  for (int i = 0; i < N; ++i) grid[h[i] * G + h[N + i]] = 3 * i + POSITION;
  for (int i = 0; i < N; ++i) grid[t[i] * G + t[N + i]] = 3 * i + TARGET;
  for (int i = 0; i < N; ++i) {
    agent_id[i] = i;
    start[2 * i] = h[i];
    start[2 * i + 1] = h[N + i];
    target[2 * i] = t[i];
    target[2 * i + 1] = t[N + i];
    position[2 * i] = h[i];
    position[2 * i + 1] = h[N + i];
  }
  *step_count = 0;
  key_out[0] = ks[0];
  key_out[1] = ks[1];
  return 0;
}

/* ======================================================================== */
/* Connector (jumanji==0.2.2 environments/routing/connector/{env,utils,       */
/* reward}.py -- UPSTREAM, not under /root/reference; call sites             */
/* rl_training/setup_train.py:158-166, demos/board_generator_demo.py:80-97)  */
/* ======================================================================== */

/* env._get_action_mask: [True, valid(UP), valid(RIGHT), valid(DOWN), valid(LEFT)] */
void orc_connector_action_mask(int G, int N, const int32_t *grid,
                               const int32_t *target, const int32_t *position,
                               uint8_t *mask) {
  for (int i = 0; i < N; ++i) {
    int r = position[2 * i], c = position[2 * i + 1];
    int connected = (r == target[2 * i] && c == target[2 * i + 1]);
    mask[5 * i] = 1;
    for (int a = 1; a < 5; ++a) {
      int nr, nc;
      move_position(r, c, a, &nr, &nc);
      mask[5 * i + a] = (uint8_t)is_valid_position(G, grid, i, connected, nr, nc);
    }
  }
}

/* env._obs_from_grid: agent a sees ids shifted so that its own codes are 1,2,3 */
void orc_connector_obs(int G, int N, const int32_t *grid, int32_t *obs) {
  const int cells = G * G;
  for (int a = 0; a < N; ++a)
    for (int k = 0; k < cells; ++k) {
      int32_t v = grid[k];
      int32_t o = 0;
      if (v != 0) {
        int32_t m = (v - 1 - 3 * a) % (3 * N);
        if (m < 0) m += 3 * N;
        o = m + 1;
      }
      obs[a * cells + k] = o;
    }
}

/* env._get_extras */
void orc_connector_extras(int G, int N, const int32_t *grid,
                          const int32_t *target, const int32_t *position,
                          int32_t *num_connections, float *ratio_connections,
                          int32_t *total_path_length) {
  int conn = 0;
  for (int i = 0; i < N; ++i)
    conn += (position[2 * i] == target[2 * i] && position[2 * i + 1] == target[2 * i + 1]);
  int paths = 0;
  for (int k = 0; k < G * G; ++k) paths += (grid[k] > 0 && (grid[k] - 1) % 3 == 0);
  *num_connections = conn;
  *ratio_connections = (float)conn / (float)N;
  *total_path_length = paths + N; /* path cells + one head per agent */
}

void orc_connector_step(int G, int N, int32_t *grid, int32_t *step_count,
                        const int32_t *target, int32_t *position,
                        const int32_t *action, int time_limit,
                        float timestep_reward, float connected_reward,
                        int32_t *obs, uint8_t *mask, float *reward,
                        float *discount, int8_t *step_type,
                        int32_t *num_connections, float *ratio_connections,
                        int32_t *total_path_length) {
  int was[ORC_MAX_N];
  for (int i = 0; i < N; ++i)
    was[i] = (position[2 * i] == target[2 * i] && position[2 * i + 1] == target[2 * i + 1]);
  step_agents_with_actions(G, N, grid, target, position, action);
  *step_count += 1;
  /* DenseRewardFn */
  for (int i = 0; i < N; ++i) {
    int now = (position[2 * i] == target[2 * i] && position[2 * i + 1] == target[2 * i + 1]);
    volatile float cr = connected_reward * ((!was[i] && now) ? 1.0f : 0.0f);
    volatile float tr = timestep_reward * ((!was[i]) ? 1.0f : 0.0f);
    reward[i] = cr + tr;
  }
  orc_connector_action_mask(G, N, grid, target, position, mask);
  orc_connector_obs(G, N, grid, obs);
  int all_done = 1;
  for (int i = 0; i < N; ++i) {
    int now = (position[2 * i] == target[2 * i] && position[2 * i + 1] == target[2 * i + 1]);
    int any = mask[5 * i + 1] | mask[5 * i + 2] | mask[5 * i + 3] | mask[5 * i + 4];
    int done = now || !any; /* connected_or_blocked */
    discount[i] = done ? 0.0f : 1.0f;
    all_done = all_done && done;
  }
  orc_connector_extras(G, N, grid, target, position, num_connections,
                       ratio_connections, total_path_length);
  if (all_done || *step_count >= time_limit) { /* termination */
    *step_type = 2;
    for (int i = 0; i < N; ++i) discount[i] = 0.0f;
  } else { /* transition */
    *step_type = 1;
  }
}

/* ======================================================================== */
/* validity rules: the reference's NumPy code, function by function           */
/*   UP = numpy_implementation/utils/post_processor_utils_numpy.py            */
/*   BP = numpy_implementation/utils/board_processor.py                       */
/* Pinned by tests/golden/validity_reference.npz = verdicts of those very     */
/* functions (imported unmodified) on 2 400 boards,                           */
/* tests/tools/make_validity_fixtures.py.                                     */
/* ======================================================================== */

/* num_wire_neighbors (UP:124-155, BP:456-487): adjacent cells whose code lies in
 * [3w+1, 3w+3], w = (label-1)//3, order up, left, down, right */
static int val_wire_neighbours(int G, const int32_t *board, int k) {
  const int w = (board[k] - 1) / 3, lo = 3 * w + PATH, hi = 3 * w + TARGET;
  const int r = k / G, c = k % G;
  int nb = 0;
  if (r > 0 && board[k - G] >= lo && board[k - G] <= hi) nb++;
  if (c > 0 && board[k - 1] >= lo && board[k - 1] <= hi) nb++;
  if (r < G - 1 && board[k + G] >= lo && board[k + G] <= hi) nb++;
  if (c < G - 1 && board[k + 1] >= lo && board[k + 1] <= hi) nb++;
  return nb;
}

/* breadth-first search from `from` to `to` through cells whose code passes `ok`:
 * with_empty = 0: the wire's own codes only (the invariant "a wire connects its own
 * start and target"); with_empty = 1: own codes and EMPTY = the valid_cells list of
 * BoardProcessor.get_path_from_head_and_target (BP:111-162), whose PathNotFoundError
 * is raised exactly when this search fails (the shuffled move order picks among
 * shortest paths, it cannot change whether one exists). */
static int val_reachable(int G, const int32_t *board, int w, int from, int to, int with_empty,
                         int32_t *queue, uint8_t *seen) {
  const int cells = G * G, lo = 3 * w + PATH, hi = 3 * w + TARGET;
  memset(seen, 0, (size_t)cells);
  int qh = 0, qt = 0;
  queue[qt++] = from;
  seen[from] = 1;
  while (qh < qt) {
    const int k = queue[qh++];
    if (k == to) return 1;
    const int r = k / G, c = k % G;
    const int nbk[4] = {c < G - 1 ? k + 1 : -1, c > 0 ? k - 1 : -1, r < G - 1 ? k + G : -1, r > 0 ? k - G : -1};
    for (int j = 0; j < 4; ++j) {
      const int p = nbk[j];
      if (p < 0 || seen[p]) continue;
      const int32_t v = board[p];
      if ((v >= lo && v <= hi) || (with_empty && v == EMPTY)) {
        seen[p] = 1;
        queue[qt++] = p;
      }
    }
  }
  return 0;
}

/* Flags (0 = valid by every rule):
 *   1   EncodingOutOfRangeError: a code < 0 or > 3N (verify_encodings_range BP:406-416); as in
 *       is_valid_board (BP:391-404, UP:34-48) nothing else is evaluated then
 *   2   MissingHeadTailError: some wire has no POSITION or no TARGET code
 *       (verify_number_heads_tails BP:419-431, UP:72-85)
 *   4   InvalidWireStructureError: verify_wire_validity (UP:88-121, BP:433-454) is False
 *   8   a wire's first head and first target are not connected through its own cells
 *  16   zero-length wire: a lone TARGET, no head, no path (ParallelRandomWalk quirk, SURVEY A.7.3);
 *       the reference reports it as 2 | 4
 *  32   a wire has more than one head or target (the DuplicateHeadsTailsError the reference means to
 *       raise; its counts run over np.setdiff1d(...) = unique values, so it never can)
 *  64   PathNotFoundError: get_path_from_head_and_target (BP:111-162) finds no path for some wire
 * 128   rule 2 or 4 is broken by something OTHER than a zero-length wire */
int orc_validate_board(int G, int N, const int32_t *board) {
  const int cells = G * G;
  int flags = 0;
  for (int k = 0; k < cells; ++k)
    if (board[k] < 0 || board[k] > 3 * N) flags |= 1;
  if (flags) return flags;
  int heads[ORC_MAX_N] = {0}, targets[ORC_MAX_N] = {0}, paths[ORC_MAX_N] = {0}, hpos[ORC_MAX_N], tpos[ORC_MAX_N];
  for (int k = 0; k < cells; ++k) { /* row-major: the first hit is np.argwhere(...)[0] (BP:79-82) */
    const int32_t v = board[k];
    if (v == 0) continue;
    const int w = (v - 1) / 3, t = (v - 1) % 3 + 1;
    if (t == PATH) paths[w]++;
    if (t == POSITION && heads[w]++ == 0) hpos[w] = k;
    if (t == TARGET && targets[w]++ == 0) tpos[w] = k;
  }
  int zero_len[ORC_MAX_N];
  for (int w = 0; w < N; ++w) {
    zero_len[w] = (heads[w] == 0 && targets[w] == 1 && paths[w] == 0);
    if (zero_len[w]) flags |= 16;
    if (heads[w] < 1 || targets[w] < 1) flags |= zero_len[w] ? 2 : (2 | 128);
    if (heads[w] > 1 || targets[w] > 1) flags |= 32;
  }
  for (int k = 0; k < cells; ++k) {
    const int32_t v = board[k];
    if (v <= 0) continue;
    const int t = (v - 1) % 3 + 1, nb = val_wire_neighbours(G, board, k);
    if (t == PATH ? nb != 2 : nb != 1) flags |= zero_len[(v - 1) / 3] ? 4 : (4 | 128);
  }
  int32_t *queue = (int32_t *)malloc(sizeof(int32_t) * (size_t)cells);
  uint8_t *seen = (uint8_t *)malloc((size_t)cells);
  for (int w = 0; w < N; ++w) {
    if (heads[w] < 1 || targets[w] < 1) continue;
    if (val_reachable(G, board, w, hpos[w], tpos[w], 0, queue, seen)) continue; /* then a path through own + EMPTY cells exists too */
    flags |= 8;
    if (!val_reachable(G, board, w, hpos[w], tpos[w], 1, queue, seen)) flags |= 64;
  }
  free(queue);
  free(seen);
  return flags;
}

/* ======================================================================== */
/* batched wrappers                                                          */
/* ======================================================================== */
int orc_max_threads(void) {
#ifdef _OPENMP
  return omp_get_max_threads();
#else
  return 1;
#endif
}

static int pick_threads(int nthreads) {
  int mx = orc_max_threads();
  if (nthreads <= 0 || nthreads > mx) return mx;
  return nthreads;
}

/* rows [offset, offset+count) of jax.random.split(key, B) */
void orc_split_batch_slice(const uint32_t key[2], int64_t B, int64_t offset,
                           int64_t count, uint32_t *out) {
  for (int64_t i = 0; i < 2 * count; ++i) {
    int64_t f = 2 * offset + i; /* flat word index in [0, 2B) */
    uint32_t a, b;
    if (f < B) {
      orc_threefry2x32(key[0], key[1], (uint32_t)f, (uint32_t)(f + B), &a, &b);
      out[i] = a;
    } else {
      orc_threefry2x32(key[0], key[1], (uint32_t)(f - B), (uint32_t)f, &a, &b);
      out[i] = b;
    }
  }
}

int orc_prw_generate_batch(const uint32_t *keys, int64_t B, int G, int N,
                           int32_t *heads, int32_t *targets, int32_t *solved,
                           int32_t *stats, int nthreads) {
  int rc_all = 0;
  int nt = pick_threads(nthreads);
  (void)nt;
#pragma omp parallel for num_threads(nt) schedule(dynamic, 64)
  for (int64_t b = 0; b < B; ++b) {
    int rc = orc_prw_generate(&keys[2 * b], G, N, &heads[b * 2 * N], &targets[b * 2 * N],
                              &solved[b * G * G], stats ? &stats[2 * b] : NULL);
    if (rc) rc_all = rc;
  }
  return rc_all;
}

int orc_seedext_solved_batch(const uint32_t *keys, int64_t B, int G, int N,
                             float randomness, int two_sided, int iterations,
                             int64_t ext_steps, int32_t *boards, int32_t *stats,
                             int nthreads) {
  int rc_all = 0;
  int nt = pick_threads(nthreads);
  (void)nt;
#pragma omp parallel for num_threads(nt) schedule(dynamic, 16)
  for (int64_t b = 0; b < B; ++b) {
    int rc = orc_seedext_solved(&keys[2 * b], G, N, randomness, two_sided, iterations,
                                ext_steps, &boards[b * G * G], stats ? &stats[3 * b] : NULL);
    if (rc) rc_all = rc;
  }
  return rc_all;
}

int orc_state_batch(int kind, const uint32_t *keys, int64_t B, int G, int N,
                    int32_t *grid, int32_t *step_count, int32_t *agent_id,
                    int32_t *start, int32_t *target, int32_t *position,
                    uint32_t *key_out, int nthreads) {
  int rc_all = 0;
  int nt = pick_threads(nthreads);
  (void)nt;
#pragma omp parallel for num_threads(nt) schedule(dynamic, 64)
  for (int64_t b = 0; b < B; ++b) {
    int rc = orc_state(kind, &keys[2 * b], G, N, &grid[b * G * G], &step_count[b],
                       &agent_id[b * N], &start[b * 2 * N], &target[b * 2 * N],
                       &position[b * 2 * N], &key_out[2 * b]);
    if (rc) rc_all = rc;
  }
  return rc_all;
}

int orc_seqrw_generate_batch(const uint32_t *keys, int64_t B, int G, int N, int32_t *boards, int32_t *stats, int nthreads) {
  int rc_all = 0;
  int nt = pick_threads(nthreads);
  (void)nt;
#pragma omp parallel for num_threads(nt) schedule(dynamic, 16)
  for (int64_t b = 0; b < B; ++b) {
    int rc = orc_seqrw_generate(&keys[2 * b], G, N, &boards[b * G * G], stats ? &stats[2 * b] : NULL);
    if (rc) rc_all = rc;
  }
  return rc_all;
}

void orc_connector_observe_batch(int64_t B, int G, int N, const int32_t *grid,
                                 const int32_t *target, const int32_t *position,
                                 int32_t *obs, uint8_t *mask,
                                 int32_t *num_connections,
                                 float *ratio_connections,
                                 int32_t *total_path_length, int nthreads) {
  int nt = pick_threads(nthreads);
  (void)nt;
#pragma omp parallel for num_threads(nt) schedule(static)
  for (int64_t b = 0; b < B; ++b) {
    const int32_t *g = &grid[b * G * G];
    orc_connector_action_mask(G, N, g, &target[b * 2 * N], &position[b * 2 * N], &mask[b * 5 * N]);
    orc_connector_obs(G, N, g, &obs[b * (int64_t)N * G * G]);
    orc_connector_extras(G, N, g, &target[b * 2 * N], &position[b * 2 * N],
                         &num_connections[b], &ratio_connections[b], &total_path_length[b]);
  }
}

/* autoreset_kind 3 = BoardDatasetGeneratorJAX over ds_heads / ds_targets [ds_K,2,N]
 * (rl_training/setup_train.py:119-133,158: Connector(generator=BoardDatasetGeneratorJAX(...))) */
void orc_connector_step_batch_ds(int64_t B, int G, int N, int32_t *grid,
                                 int32_t *step_count, int32_t *start,
                                 int32_t *target, int32_t *position,
                                 uint32_t *key, const int32_t *action,
                                 int time_limit, float timestep_reward,
                                 float connected_reward, int autoreset_kind,
                                 const int32_t *ds_heads, const int32_t *ds_targets, int64_t ds_K,
                                 int32_t *obs, uint8_t *mask, float *reward,
                                 float *discount, int8_t *step_type,
                                 int32_t *num_connections,
                                 float *ratio_connections,
                                 int32_t *total_path_length,
                                 int32_t *obs_step_count, int nthreads) {
  int nt = pick_threads(nthreads);
  (void)nt;
#pragma omp parallel for num_threads(nt) schedule(dynamic, 64)
  for (int64_t b = 0; b < B; ++b) {
    int32_t *g = &grid[b * G * G];
    int32_t *ob = &obs[b * (int64_t)N * G * G];
    orc_connector_step(G, N, g, &step_count[b], &target[b * 2 * N], &position[b * 2 * N],
                       &action[b * N], time_limit, timestep_reward, connected_reward, ob,
                       &mask[b * 5 * N], &reward[b * N], &discount[b * N], &step_type[b],
                       &num_connections[b], &ratio_connections[b], &total_path_length[b]);
    if (autoreset_kind >= 0 && step_type[b] == 2) {
      /* jumanji VmapAutoResetWrapper._auto_reset: key, _ = split(state.key);
       * state, reset_ts = env.reset(key); keep reward/discount/step_type/extras,
       * replace the observation. */
      uint32_t ks[4];
      int32_t ids[ORC_MAX_N];
      orc_split(&key[2 * b], 2, ks);
      if (autoreset_kind == 3)
        orc_dataset_state(&ks[0], G, N, ds_heads, ds_targets, ds_K, g, &step_count[b], ids, &start[b * 2 * N],
                          &target[b * 2 * N], &position[b * 2 * N], &key[2 * b]);
      else
        orc_state(autoreset_kind, &ks[0], G, N, g, &step_count[b], ids, &start[b * 2 * N],
                  &target[b * 2 * N], &position[b * 2 * N], &key[2 * b]);
      orc_connector_action_mask(G, N, g, &target[b * 2 * N], &position[b * 2 * N], &mask[b * 5 * N]);
      orc_connector_obs(G, N, g, ob);
    }
    if (obs_step_count) obs_step_count[b] = step_count[b];
  }
}

void orc_connector_step_batch(int64_t B, int G, int N, int32_t *grid,
                              int32_t *step_count, int32_t *start,
                              int32_t *target, int32_t *position,
                              uint32_t *key, const int32_t *action,
                              int time_limit, float timestep_reward,
                              float connected_reward, int autoreset_kind,
                              int32_t *obs, uint8_t *mask, float *reward,
                              float *discount, int8_t *step_type,
                              int32_t *num_connections,
                              float *ratio_connections,
                              int32_t *total_path_length,
                              int32_t *obs_step_count, int nthreads) {
  orc_connector_step_batch_ds(B, G, N, grid, step_count, start, target, position, key, action, time_limit,
                              timestep_reward, connected_reward, autoreset_kind, NULL, NULL, 0, obs, mask, reward,
                              discount, step_type, num_connections, ratio_connections, total_path_length,
                              obs_step_count, nthreads);
}

/* ======================================================================== */
/* board statistics: EvaluateEmptyBoard (benchmarking/benchmarks/                */
/* empty_board_evaluation.py:31-155), the deterministic part; pinned by          */
/* tests/golden/board_stats_reference.npz = that class executed unmodified        */
/* ======================================================================== */

/* assess_board (:41-54): empty -2, head (v % 3 == 2) 3, target (v % 3 == 0, v != 0) 3, route (v % 3 == 1) 2 */
static int stat_cell_score(int32_t v) {
  if (v == 0) return -2;
  return v % 3 == 1 ? 2 : 3;
}

/* get_wire_num (:139-151): -1 below 2, else (label - 2) // 3 -- so PATH cells of wire w > 0 count as wire w - 1 */
static int stat_wire_num(int32_t v) { return v < 2 ? -1 : (v - 2) / 3; }

/* scored [G,G] (score_from_neighbours :56-88), *detours (count_detours :99-137),
 * *diversity (heatmap_score_diversity :155 = number of distinct scores) */
void orc_board_statistics(int G, const int32_t *board, int count_current_wire, int32_t *scored, int32_t *detours,
                          int32_t *diversity) {
  const int P = G + 2;
  int32_t *lab = (int32_t *)calloc((size_t)P * P, sizeof(int32_t));   /* _change_heads_to_wire_ids on the padded board */
  int32_t *ind = (int32_t *)calloc((size_t)P * P, sizeof(int32_t));   /* np.pad(individual_score, 1): zeros, not -2 */
  int maxv = 0;
  for (int k = 0; k < G * G; ++k)
    if (board[k] > maxv) maxv = board[k];
  uint8_t *present = (uint8_t *)calloc((size_t)maxv + 4, 1);          /* unique(filled_board[filled_board % 3 == 2]) */
  for (int k = 0; k < G * G; ++k)
    if (board[k] > 0 && board[k] % 3 == 2) present[board[k]] = 1;
  for (int r = 0; r < G; ++r)
    for (int c = 0; c < G; ++c) {
      int32_t v = board[r * G + c];
      /* for wire_id in unique ids (ascending): cells == id + 1 -> id, cells == id + 2 -> id (:90-97); the values it
       * produces are ids (2 mod 3) and no later id looks for those, so this is a per-cell map */
      if (v > 0 && v % 3 == 0 && present[v - 1]) v = v - 1;
      else if (v >= 4 && v % 3 == 1 && present[v - 2]) v = v - 2;
      lab[(r + 1) * P + c + 1] = v;
      ind[(r + 1) * P + c + 1] = stat_cell_score(board[r * G + c]);
    }
  static const int filt[9] = {1, 2, 1, 2, 4, 2, 1, 2, 1};
  for (int r = 1; r <= G; ++r)
    for (int c = 1; c <= G; ++c) {
      int32_t seen[9];
      int nseen = 0, sum = 0;
      for (int dr = -1; dr <= 1; ++dr)
        for (int dc = -1; dc <= 1; ++dc) {
          const int32_t l = lab[(r + dr) * P + c + dc];
          sum += ind[(r + dr) * P + c + dc] * filt[(dr + 1) * 3 + dc + 1];
          if (l == 0) continue;
          int dup = 0;
          for (int q = 0; q < nseen; ++q) dup |= seen[q] == l;
          if (!dup) seen[nseen++] = l;
        }
      scored[(r - 1) * G + c - 1] = sum * nseen; /* np.sum(window * filter * diversity) */
    }
  int nd = 0;
  for (int a = 0; a < G * G; ++a) {
    int dup = 0;
    for (int b = 0; b < a && !dup; ++b) dup = scored[b] == scored[a];
    nd += !dup;
  }
  *diversity = nd;
  /* count_detours: for every TARGET cell and every PATH cell with label >= 2, the wires (by get_wire_num, empty cells
   * skipped, the cell's own wire excluded unless count_current_wire) that occur both above and below, plus those
   * that occur both left and right */
  int det = 0;
  for (int x = 0; x < G; ++x)
    for (int y = 0; y < G; ++y) {
      const int32_t v = board[x * G + y];
      if (v < 2 || v % 3 == 2) continue;
      const int cur = stat_wire_num(v);
      for (int pass = 0; pass < 2; ++pass) {
        uint64_t before = 0, after = 0; /* wire nums -1 .. 62 as bits 0 .. 63 */
        for (int t = 0; t < G; ++t) {
          const int32_t u = pass == 0 ? board[t * G + y] : board[x * G + t];
          const int pos = pass == 0 ? x : y;
          if (t == pos || u == 0) continue;
          const int w = stat_wire_num(u);
          if (!count_current_wire && w == cur) continue;
          if (t < pos) before |= 1ull << (w + 1);
          else after |= 1ull << (w + 1);
        }
        det += __builtin_popcountll(before & after);
      }
    }
  *detours = det;
  free(lab);
  free(ind);
  free(present);
}

void orc_board_statistics_batch(int64_t B, int G, const int32_t *boards, int count_current_wire, int32_t *scored,
                                int32_t *detours, int32_t *diversity, int nthreads) {
  int nt = pick_threads(nthreads);
  (void)nt;
#pragma omp parallel for num_threads(nt) schedule(static)
  for (int64_t b = 0; b < B; ++b)
    orc_board_statistics(G, &boards[b * G * G], count_current_wire, &scored[b * G * G], &detours[b], &diversity[b]);
}

void orc_validate_batch(int64_t B, int G, int N, const int32_t *boards,
                        int32_t *flags, int nthreads) {
  int nt = pick_threads(nthreads);
  (void)nt;
#pragma omp parallel for num_threads(nt) schedule(static)
  for (int64_t b = 0; b < B; ++b) flags[b] = orc_validate_board(G, N, &boards[b * G * G]);
}

/* OUR random policy (include/rbg_b200.h rbg_random_actions): uniform over the
 * legal actions, NOOP included (distribution-equal to jumanji's
 * masked_categorical_random, not bit-equal: that one is a float32 Gumbel
 * draw).  bits = threefry2x32(state.key; step_count, agent).o0;
 * pick = (bits * m) >> 32 over the m legal actions in action order. */
void orc_random_actions_batch(int64_t B, int G, int N, const int32_t *grid,
                              const int32_t *target, const int32_t *position,
                              const int32_t *step_count, const uint32_t *key,
                              int32_t *action, int nthreads) {
  int nt = pick_threads(nthreads);
  (void)nt;
#pragma omp parallel for num_threads(nt) schedule(static)
  for (int64_t b = 0; b < B; ++b) {
    uint8_t mask[5 * ORC_MAX_N];
    orc_connector_action_mask(G, N, &grid[b * G * G], &target[b * 2 * N], &position[b * 2 * N], mask);
    for (int i = 0; i < N; ++i) {
      uint32_t o0, o1;
      orc_threefry2x32(key[2 * b], key[2 * b + 1], (uint32_t)step_count[b], (uint32_t)i, &o0, &o1);
      int m = 0;
      for (int a = 0; a < 5; ++a) m += mask[5 * i + a];
      int pick = (int)(((uint64_t)o0 * (uint64_t)m) >> 32);
      int act = 0;
      for (int a = 0; a < 5; ++a) {
        if (!mask[5 * i + a]) continue;
        if (pick == 0) {
          act = a;
          break;
        }
        pick--;
      }
      action[b * N + i] = act;
    }
  }
}
