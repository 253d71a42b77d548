/*
 * rbg_b200.h -- C-ABI of the B200-native routing-board engine (librbg_b200.so).
 *
 * The drop-in boundary for the ONE hot path of mwolinska/Routing-Board-Generation:
 * ParallelRandomWalk / SeedExtension / Uniform board generation behind the
 * generator plugin `__call__(key) -> State`, and the Jumanji Connector
 * reset / step / action-mask / observation.  The reference is pure Python
 * (JAX); there is no FFI in it today.  Each entry point below names the
 * reference function (file:line under /root/reference) whose jit(vmap(...))
 * it replaces; the leading axis B of every array is that vmap axis.
 * INTEGRATION.md shows the reference-side binding (ctypes + DLPack).
 *
 * Conventions
 *   - plain C: pointers + sizes, no torch / CUDA types in any signature.
 *   - `stream` is a cudaStream_t passed as void* (NULL = default stream).
 *   - unless a function name ends in `_host`, every array pointer is a DEVICE
 *     pointer on the current CUDA device (what a DLPack capsule of a torch or
 *     JAX GPU array carries); `_host` variants take host pointers and do the
 *     H2D / D2H copies themselves.
 *   - dtypes as the reference with x64 disabled: int32 grids / coordinates /
 *     actions, uint32[2] raw threefry keys, float32 rewards, bool masks as
 *     uint8, step_type int8.
 *   - all arrays are C-contiguous, and int32 arrays of the bulk outputs
 *     (grid, obs_grid, solved) must be 16-byte aligned (torch / XLA
 *     allocations are).
 *   - return value: 0 on success, negative RBG_E* otherwise (never throws,
 *     never falls back to a CPU path); rbg_last_error() has the message.
 *   - kernels are launched asynchronously on `stream`; nothing synchronises
 *     except the `_host` variants.
 *   - square grids only (the reference's _adjacent_cells strides by rows but
 *     divmods by cols, parallel_random_walk.py:276,284): 2 <= G <= 40,
 *     1 <= N <= 32, N <= G*G (2N for the uniform generator).
 *
 * Abbreviations for citations:
 *   PRW  routing_board_generation/board_generation_methods/jax_implementation/board_generation/parallel_random_walk.py
 *   SE   .../jax_implementation/board_generation/seed_extension.py
 *   PRWG routing_board_generation/rl_training/online_generators/parallel_random_walk_generator.py
 *   UG   routing_board_generation/rl_training/online_generators/uniform_generator.py
 *   RSG  routing_board_generation/rl_training/online_generators/random_seed_generator.py
 *   SRW  .../jax_implementation/board_generation/sequential_random_walk.py
 *   ST   routing_board_generation/rl_training/setup_train.py
 *   JUM  jumanji==0.2.2 jumanji/environments/routing/connector/ (UPSTREAM, requirements.txt:5)
 */
#ifndef RBG_B200_H
#define RBG_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RBG_VERSION 200

#define RBG_OK 0
#define RBG_EINVAL (-1)   /* bad size / null pointer / unsupported config */
#define RBG_EALIGN (-2)   /* bulk pointer not 16-byte aligned */
#define RBG_ECUDA (-3)    /* CUDA runtime error (see rbg_last_error) */
#define RBG_ENOMEM (-4)

#define RBG_MAX_G 40
#define RBG_MAX_N 32

/* generator kinds: which `Generator.__call__` a State comes from */
#define RBG_GEN_PRW 0     /* ParallelRandomWalkGenerator  PRWG:46-77 */
#define RBG_GEN_UNIFORM 1 /* UniformRandomGenerator       UG:70-109  */
#define RBG_GEN_SEEDEXT 2 /* SeedExtensionGenerator       RSG:28-57  */
#define RBG_GEN_DATASET 3 /* BoardDatasetGeneratorJAX     rl_training/offline_generation/dataset_generator_jax.py:112-141
                             (needs rbg_env_params.dataset_* / the *_dataset entry points) */
#define RBG_GEN_SEQRW 4   /* SequentialRandomWalkGenerator rl_training/online_generators/sequential_random_walk_generator.py:19-62
                             (G >= 3; auto-reset through the reset-list path, like RBG_GEN_SEEDEXT) */

/* jumanji Connector `State` pytree (JUM types.py; field order as printed in
 * package_evaluation/profiling_generators.ipynb cell 4), struct-of-arrays with
 * the vmap axis leading. */
typedef struct rbg_state {
  int32_t *grid;       /* [B,G,G] */
  int32_t *step_count; /* [B]     */
  int32_t *agent_id;   /* [B,N]   */
  int32_t *start;      /* [B,N,2] */
  int32_t *target;     /* [B,N,2] */
  int32_t *position;   /* [B,N,2] */
  uint32_t *key;       /* [B,2]   */
} rbg_state;

/* jumanji `TimeStep[Observation]` + extras (JUM env.py step/reset). */
typedef struct rbg_timestep {
  int32_t *obs_grid;          /* [B,N,G,G] observation.grid        */
  uint8_t *action_mask;       /* [B,N,5]   observation.action_mask */
  int32_t *obs_step_count;    /* [B]       observation.step_count  */
  float *reward;              /* [B,N] */
  float *discount;            /* [B,N] */
  int8_t *step_type;          /* [B]  0 FIRST, 1 MID, 2 LAST */
  int32_t *num_connections;   /* [B]  extras */
  float *ratio_connections;   /* [B]  extras */
  int32_t *total_path_length; /* [B]  extras */
} rbg_timestep;

/* Connector constructor arguments (JUM env.py __init__; ST:158). */
typedef struct rbg_env_params {
  int32_t time_limit;     /* 50   */
  float timestep_reward;  /* -0.03 (DenseRewardFn) */
  float connected_reward; /* 0.1  */
  int32_t autoreset_kind; /* <0: plain Connector.step; else VmapAutoResetWrapper
                             (ST:166) resetting with that RBG_GEN_* generator */
  /* RBG_GEN_DATASET only (ST:119-133,158: Connector(generator=BoardDatasetGeneratorJAX(...))):
   * the K pre-generated boards' pins as generate_n_boards stores them, DEVICE int32[K,2,N] */
  const int32_t *dataset_heads;
  const int32_t *dataset_targets;
  int64_t dataset_K;
} rbg_env_params;

int rbg_version(void);
const char *rbg_last_error(void);
/* sm major*10+minor of the current device, SM count; returns RBG_ECUDA if no device */
int rbg_device_info(int *sm_arch, int *sm_count);

/* rows [offset, offset+count) of jax.random.split(key, B)  (the reference's key
 * convention: dataset_generator_jax.py:76, ST:397-399; each GPU derives its own
 * slice).  key is a HOST uint32[2]; out is a device uint32[count,2]. */
int rbg_split_keys(const uint32_t key[2], int64_t B, int64_t offset,
                   int64_t count, uint32_t *out, void *stream);

/* ParallelRandomWalkBoard(G,G,N).generate_board(key)   PRW:60-90
 * keys[B,2] -> heads[B,2,N], targets[B,2,N], solved[B,G,G].
 * stats (may be NULL): int32[B,2] = (while-loop trips, collided moves). */
int rbg_prw_generate(const uint32_t *keys, int64_t B, int G, int N,
                     int32_t *heads, int32_t *targets, int32_t *solved,
                     int32_t *stats, void *stream);

/* Generator.__call__(key) -> State for kind in RBG_GEN_*  (PRWG:46-77,
 * UG:70-109, RSG:28-57).  keys[B,2] -> *out. */
int rbg_generator_state(int kind, const uint32_t *keys, int64_t B, int G, int N,
                        const rbg_state *out, void *stream);

/* BoardDatasetGeneratorJAX.__call__(key) -> State
 * (rl_training/offline_generation/dataset_generator_jax.py:112-141): `key, _ = split(key)`,
 * `which = randint(key, (), 0, K)`, State from the K pre-generated boards' pins
 * heads[K,2,N] / targets[K,2,N] (the layout generate_n_boards stores, :58-110). */
int rbg_dataset_state(const uint32_t *keys, int64_t B, int G, int N,
                      const int32_t *heads, const int32_t *targets, int64_t K,
                      const rbg_state *out, void *stream);

/* Connector(generator=BoardDatasetGeneratorJAX(...)).reset(key)  (ST:119-133,158,400) =
 * rbg_dataset_state + rbg_connector_observe */
int rbg_connector_reset_dataset(const uint32_t *keys, int64_t B, int G, int N,
                                const int32_t *heads, const int32_t *targets, int64_t K,
                                const rbg_state *state, const rbg_timestep *ts, void *stream);

/* jax.vmap(lambda k: jax.random.split(k, num))(keys): keys[B,2] -> out[B,num,2].  The per-env key
 * derivations around the env (`key, _ = split(state.key)` of VmapAutoResetWrapper._auto_reset;
 * load_and_test_agents.ipynb cell 10) for callers that reset with their own Generator. */
int rbg_split_each(const uint32_t *keys, int64_t B, int num, uint32_t *out, void *stream);

/* SeedExtensionBoard(G,G,N).return_solved_board(key, randomness, two_sided,
 * extension_iterations, extension_steps)   SE:149-227.
 * extension_steps < 0 means unlimited (the reference default 1e23). */
int rbg_seedext_solved(const uint32_t *keys, int64_t B, int G, int N,
                       float randomness, int two_sided, int iterations,
                       int64_t extension_steps, int32_t *solved, void *stream);
/* SeedExtensionBoard.generate_starts_ends   SE:257-304 -> starts[B,2,N], ends[B,2,N] */
int rbg_seedext_starts_ends(const uint32_t *keys, int64_t B, int G, int N,
                            float randomness, int two_sided, int iterations,
                            int64_t extension_steps, int32_t *starts,
                            int32_t *ends, void *stream);

/* SequentialRandomWalkBoard(G,G,N).generate(key)   SRW:324-392 (SRW = .../jax_implementation/board_generation/
 * sequential_random_walk.py): wires placed one after the other, each a self-avoiding walk from a random empty cell;
 * up to 2G attempts from the same key with a shrinking maximum walk length; a zero board when every attempt fails.
 * board: int32[B,G,G], or with as_float32 != 0 float32[B,G,G] (the reference returns the codes in jnp.zeros'
 * default dtype).  stats (may be NULL): int32[B,2] = (attempt that succeeded, 0 = none; steps of that attempt).
 * The reference draws every cell with jax.random.choice(p in {0,1}, replace=False) = a float32 Gumbel top-k; the
 * result is reproduced exactly for any strictly monotone float32 log (DESIGN.md §8 f4).  The class is not
 * instantiable in the reference as shipped (abstract methods, abstract_board.py:47-53); this is its method bodies.
 * 3 <= G. */
int rbg_seqrw_generate(const uint32_t *keys, int64_t B, int G, int N, void *board, int as_float32, int32_t *stats,
                       void *stream);
/* SequentialRandomWalkBoard.generate_starts_ends   SRW:394-431 -> starts[B,2,N], ends[B,2,N]
 * (first POSITION / TARGET cell of every wire; (0,0) on a zero board) */
int rbg_seqrw_starts_ends(const uint32_t *keys, int64_t B, int G, int N, int32_t *starts, int32_t *ends,
                          void *stream);

/* The observation half of Connector.reset on an existing State (the recipe
 * at demos/board_generator_demo.py:83-96): action mask, per-agent
 * observation, extras, restart() reward 0 / discount 1 / step_type FIRST. */
int rbg_connector_observe(const rbg_state *state, int64_t B, int G, int N,
                          const rbg_timestep *ts, void *stream);

/* Connector(generator).reset(key)  (JUM env.py reset; ST:400) = generator + observe */
int rbg_connector_reset(int kind, const uint32_t *keys, int64_t B, int G, int N,
                        const rbg_state *state, const rbg_timestep *ts,
                        void *stream);

/* bytes of device scratch rbg_connector_step needs when autoreset is on.  The
 * workspace belongs to ONE env batch for as long as that batch is stepped: besides
 * the reset lists it caches, per env, the next episode's start / target pins, which
 * the library generates ahead of time on the caller's stream (the reset key of
 * an episode is known when the episode starts).  16-byte aligned, need not be
 * cleared.  Call rbg_workspace_release before freeing it, and before handing it to
 * another env batch (the library re-initialises it by itself when the shape or the
 * generator kind changes, or after a SeedExtension batch has used it; a batch of the
 * same shape and kind would merely start with cache misses). */
int64_t rbg_step_workspace_bytes(int64_t B, int G, int N);
/* waits for the work queued on `workspace` (on the stream it was last used on) and forgets it */
int rbg_workspace_release(void *workspace);

/* Connector.step(state, action) (JUM env.py step), or with
 * params->autoreset_kind >= 0 VmapAutoResetWrapper(Connector).step (ST:166).
 * in and out may alias (in-place update).  action int32[B,N].
 * workspace: device scratch of rbg_step_workspace_bytes (may be NULL when
 * autoreset is off). */
int rbg_connector_step(const rbg_state *in, const rbg_state *out,
                       const int32_t *action, int64_t B, int G, int N,
                       const rbg_env_params *params, const rbg_timestep *ts,
                       void *workspace, void *stream);

/* Random policy over the legal actions, NOOP included (distribution-equal to
 * jumanji's make_random_policy_connector, ST:246; NOT a bit-parity surface:
 * upstream draws a float32 Gumbel).  bits = threefry2x32(state.key;
 * step_count, agent).o0; pick = (bits * m) >> 32 among the m legal actions. */
int rbg_random_actions(const rbg_state *state, int64_t B, int G, int N,
                       int32_t *action, void *stream);

/* rbg_random_actions + rbg_connector_step in one launch sequence
 * (the agent=random benchmark loop, benchmark_on_random_agent.py:59-102).
 * action_out may be NULL. */
int rbg_connector_step_random(const rbg_state *in, const rbg_state *out,
                              int32_t *action_out, int64_t B, int G, int N,
                              const rbg_env_params *params,
                              const rbg_timestep *ts, void *workspace,
                              void *stream);

/* T consecutive rbg_connector_step_random calls in one call: the rollout of the
 * reference's training / benchmark loop (`n_steps` scan, agent_training/configs/
 * env/connector.yaml:27; benchmark_on_random_agent.py:59-102) with generation,
 * reset and stepping fused into one launch sequence.  `state` is updated in place;
 * every field of `ts` (and action_out, may be NULL) points to arrays with an extra
 * LEADING axis T: obs_grid[T,B,N,G,G], reward[T,B,N], step_type[T,B] ... */
int rbg_connector_rollout_random(const rbg_state *state, int32_t *action_out,
                                 int64_t T, int64_t B, int G, int N,
                                 const rbg_env_params *params,
                                 const rbg_timestep *ts, void *workspace,
                                 void *stream);

/* per-episode metrics of rbg_connector_episodes_random and rbg_connector_eval_step (names as BenchmarkData / PickleLogger) */
typedef struct rbg_episode_metrics {
  float   *episode_return;     /* [B,N] per agent, summed in step order (float32, round-to-nearest) */
  int32_t *episode_length;     /* [B]   steps taken until the first LAST step */
  int32_t *num_connections;    /* [B]   extras of that terminal TimeStep */
  float   *ratio_connections;  /* [B]  */
  int32_t *total_path_length;  /* [B]  */
} rbg_episode_metrics;

/* Run every env of `start` under the random policy (rbg_random_actions' draw) until its first LAST step;
 * Connector(time_limit, DenseRewardFn) semantics from params, params->autoreset_kind must be < 0.
 * `start` is read only.  final_state (may be NULL): the State after each env's terminal step.
 * The random-agent evaluation of a board generator (the reference's benchmarks / evaluators reduce each episode
 * to these five numbers): one launch, no per-step output, and no workspace (the library takes 256 bytes of
 * stream-ordered scratch for the call). */
int rbg_connector_episodes_random(const rbg_state *start, int64_t B, int G, int N,
                                  const rbg_env_params *params, const rbg_episode_metrics *out,
                                  const rbg_state *final_state, void *stream);

/* One plain Connector.step (params->autoreset_kind must be < 0) of the envs whose live[b] != 0, with `action` int32[B,N]
 * given: the step of a policy evaluation, one call per policy call.  For a live env the State is stepped in place and
 * TimeStep row b is written as rbg_connector_step writes it; the record `acc` accumulates episode_return (float32,
 * added in step order) and episode_length, and on LAST takes the TimeStep's extras, live[b] is cleared and the device
 * int32 *live_count is decremented.  An env with live[b] == 0 is not read (but for its live byte) nor written: not its
 * State, TimeStep row, record or action.  The caller starts with `acc` zeroed, live 1 and *live_count = B; from a
 * reset State every env is done after at most time_limit calls. */
int rbg_connector_eval_step(const rbg_state *state, const int32_t *action, uint8_t *live, int32_t *live_count,
                            int64_t B, int G, int N, const rbg_env_params *params, const rbg_timestep *ts,
                            const rbg_episode_metrics *acc, void *stream);

/* Board validity: the reference's NumPy rules (numpy_implementation/utils/
 * post_processor_utils_numpy.py:34-155 = UP, numpy_implementation/utils/board_processor.py:111-162,
 * 391-487 = BP).  flags int32[B], 0 = valid by every rule:
 *     1  EncodingOutOfRangeError: a code < 0 or > 3N (verify_encodings_range BP:406-416); as in
 *        is_valid_board (BP:391-404) nothing else is evaluated then
 *     2  MissingHeadTailError: some wire has no POSITION or no TARGET code (BP:419-431, UP:72-85)
 *     4  InvalidWireStructureError: verify_wire_validity is False (UP:88-121, BP:433-454)
 *     8  a wire's (first) head and target are not connected through the wire's own cells
 *    16  zero-length wire: a lone TARGET (a ParallelRandomWalk quirk; the reference reports 2 | 4)
 *    32  a wire has several heads or targets (the DuplicateHeadsTailsError the reference means to
 *        raise but cannot: its counts run over np.setdiff1d = unique values)
 *    64  PathNotFoundError: BoardProcessor.get_path_from_head_and_target (BP:111-162) finds no path
 *        through the wire's own cells and EMPTY cells
 *   128  rule 2 or 4 is broken by something other than a zero-length wire
 * A generated board is sound when (flags & (1 | 8 | 32 | 64 | 128)) == 0. */
int rbg_validate(const int32_t *boards, int64_t B, int G, int N, int32_t *flags,
                 void *stream);

/* Board statistics of solved boards: EvaluateEmptyBoard (benchmarking/benchmarks/empty_board_evaluation.py:31-155),
 * the deterministic part of what run_benchmark_on_generated_board collects per board.
 *   scored[B,G,G]  score_from_neighbours (:56-88): per cell, the 3x3 window of assess_board's scores (empty -2, head /
 *                  target 3, route 2; zero padding) weighted [[1,2,1],[2,4,2],[1,2,1]], times the number of distinct
 *                  wire labels in the window (labels by _change_heads_to_wire_ids :90-97).  May be NULL.
 *   detours[B]     count_detours(count_current_wire) (:99-137)
 *   diversity[B]   heatmap_score_diversity = len(np.unique(scored_board)) (:155)
 * Codes outside [0, 96] make detours = diversity = -1 for that board.  Not reproduced: BoardProcessor's wire lengths /
 * bends, which come from shortest paths chosen by an unseeded random.shuffle (board_processor.py:111-162). */
int rbg_board_statistics(const int32_t *boards, int64_t B, int G, int count_current_wire,
                         int32_t *scored, int32_t *detours, int32_t *diversity, void *stream);

/* ---- host-buffer variants: same semantics, HOST pointers, copies inside,
 * synchronous.  device < 0 = current device. ------------------------------ */
int rbg_prw_generate_host(const uint32_t *keys, int64_t B, int G, int N,
                          int32_t *heads, int32_t *targets, int32_t *solved,
                          int device);
int rbg_connector_reset_host(int kind, const uint32_t *keys, int64_t B, int G,
                             int N, const rbg_state *state,
                             const rbg_timestep *ts, int device);
int rbg_connector_step_host(const rbg_state *in, const rbg_state *out,
                            const int32_t *action, int64_t B, int G, int N,
                            const rbg_env_params *params,
                            const rbg_timestep *ts, int device);
/* Env-pool style step: `state` holds DEVICE pointers and is updated in place (the State is
 * opaque env state, as it is between two `env.step` calls in the reference's loop), `action`
 * int32[B,N] comes from and every field of `ts` goes to HOST memory (pinned recommended).
 * `state` must have been produced on the device's default stream (or a stream that synchronises with it); the call
 * orders itself behind that stream with an event and waits for its own copy streams at exit.
 * Transport: the observation (96 % of a TimeStep's bytes; codes <= 3 * RBG_MAX_N) crosses the bus as one byte per
 * cell (half a byte when N <= 5: codes <= 15) into a pinned staging buffer of the library and is widened to ts->obs_grid's int32 by a pool of host threads
 * (all cores of the affinity mask / LOCAL_WORLD_SIZE, or RBG_HOST_THREADS), slice by slice while later slices are
 * in flight; ts->obs_grid need not be pinned. */
int rbg_connector_step_host_io(const rbg_state *state, const int32_t *action,
                               int64_t B, int G, int N,
                               const rbg_env_params *params,
                               const rbg_timestep *ts, int device);
/* The host half of that transport on its own: n byte codes in HOST memory -> int32 in HOST memory on the library's
 * thread pool (synchronous).  For consumers that keep observations as bytes and widen on demand, and for bench.py:
 * its rate is the ceiling of what rbg_connector_step_host_io can deliver on a host (no GPU work, no bus). */
int rbg_host_widen(const uint8_t *src, int32_t *dst, int64_t n);
/* the same for the nibble transport (observation codes <= 15, i.e. at most 5 agents: two cells per byte, low nibble
 * first); n = number of int32 outputs, even */
int rbg_host_widen4(const uint8_t *src, int32_t *dst, int64_t n);
/* Bytes the _host_io calls moved over the bus since the last reset (counted where the copies are enqueued) and the
 * number of host threads that widen the observation; any pointer may be NULL. */
int rbg_host_transfer_stats(int64_t *h2d_bytes, int64_t *d2h_bytes, int *host_threads, int reset);
/* pinned host allocation helpers for the _host variants (optional) */
void *rbg_host_alloc(int64_t bytes);
void rbg_host_free(void *p);

/* counters for bench.py's gpu_launches claim: number of kernels this library
 * launched since the last reset */
int64_t rbg_launch_count(int reset);

/* Per-kernel device timing for bench.py's roofline figures.  While enabled,
 * every kernel launch is bracketed by a pair of CUDA events recorded on the
 * launching stream.  rbg_kernel_time synchronises on the recorded events,
 * returns the number of launches of `kernel` (RBG_K_*) and their summed device
 * time since the last call, and clears that kernel's record.  Consecutive fused
 * rollout launches, and a per-step env kernel with the cache refill of the step
 * before it, normally overlap on the stream; while timing is enabled they run one kernel at
 * a time, so that a pair of events times one kernel. */
#define RBG_K_PRW 0        /* prw_kernel: ParallelRandomWalk / Uniform generator */
#define RBG_K_ENV 1        /* env_warp_kernel: Connector step / observe */
#define RBG_K_RANDACT 2    /* random_actions_kernel */
#define RBG_K_SPLIT 3      /* split_keys_kernel */
#define RBG_K_VALIDATE 4   /* validate_kernel */
#define RBG_K_SEEDEXT 5    /* seedext_kernel */
#define RBG_K_ROLLOUT 6    /* rollout_persist_kernel (rollout_warp_kernel for the dataset generator): T fused steps */
#define RBG_K_SEQRW 7      /* seqrw_walk_kernel + its finish kernel */
#define RBG_K_EPISODES 8   /* episode_warp_kernel: random-agent episodes to their first LAST step */
#define RBG_K_EVAL_STEP 9  /* eval_step_kernel: one policy-evaluation step of the live envs */
#define RBG_K_COUNT 10
int rbg_kernel_timing(int enable);
int rbg_kernel_time(int kernel, int64_t *launches, double *total_ms);

#ifdef __cplusplus
}
#endif
#endif /* RBG_B200_H */
