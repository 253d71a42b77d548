// rbg_host.h -- host-side declarations shared by the kernel translation units
// and the C-ABI (c_api.cu).  Internal; the public surface is include/rbg_b200.h.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/rbg_b200.h"
#include "rbg_device.cuh"

namespace rbg {

// error plumbing (c_api.cu)
int set_error(int code, const char *fmt, ...);
int set_cuda_error(cudaError_t e, const char *what);
int check_launch(const char *what);
// properties of the current device (cached per device): SM count, shared memory per SM in bytes
int device_sm_count();
size_t device_smem_per_sm();
// Brackets one kernel launch: counts it (rbg_launch_count) and, while
// rbg_kernel_timing is on, records a CUDA event pair on `stream` around it.
bool kernel_timing_on();  // rbg_kernel_timing(1) is in effect
struct LaunchScope {
  int id;
  cudaStream_t stream;
  void *rec;
  LaunchScope(int kernel_id, cudaStream_t s);
  ~LaunchScope();
};

// ---- generator kernel (prw_kernel.cu) -----------------------------------
enum : int { PRW_MODE_BOARD = 0, PRW_MODE_STATE = 1, PRW_MODE_UNIFORM = 2 };

struct PrwParams {
  const uint32_t *keys;  // [B,2]; with `list`: state.key of all envs
  long long B;
  int G, N;
  int mode;         // PRW_MODE_*
  int extra_split;  // leading key = split(key)[0] applications
  int debug;        // bit0: force the exact selection fallback
  int observe;      // write observation + action mask of the fresh state
  int32_t *heads, *targets, *solved, *stats;
  rbg_state st;
  rbg_timestep ts;
  const int32_t *list;        // optional env list (auto-reset)
  const int32_t *list_count;  // device count of list entries
  int32_t *list_ticket;       // optional: CTAs-done ticket; the last CTA zeroes list_count and the ticket
  // auto-reset cache refill: keys[] is indexed by list slot (not env id) and the
  // result goes to the env's cache entry instead of State / TimeStep
  int keys_compact, to_cache;
  int trigger_dependents;  // griddepcontrol.launch_dependents at the start: the next kernel of the stream, if it was launched
                           // with programmatic stream serialization, need not wait for this one (per-step cache refill)
  unsigned long long *cache_tag;  // [B]   state.key this entry succeeds (k0 | k1 << 32)
  uint2 *cache_key;               // [B]   State.key of the cached episode
  uint32_t *cache_pins;           // [B,N] start_r<<24 | start_c<<16 | target_r<<8 | target_c
  // filled by launch_prw
  int W, S, SBp, cells, M, cap, Np, nsel;
  uint32_t thresh;
  FastDiv divG;
};

int launch_prw(PrwParams p, int64_t max_boards, cudaStream_t stream);
// two short-list launches in one (prw_pair_kernel): `a` then launch_dependents then `b`
int launch_prw_pair(PrwParams a, PrwParams b, int64_t max_boards, cudaStream_t stream);

// ---- connector kernel (connector_kernel.cu) -----------------------------
enum : int { ENV_MODE_STEP = 0, ENV_MODE_OBSERVE = 1 };

struct EnvParams {
  rbg_state in, out;
  rbg_timestep ts;
  const int32_t *action;  // [B,N] (STEP)
  int32_t *action_out;    // optional (random policy)
  long long B;
  int G, N;
  int mode;           // ENV_MODE_*
  int random_policy;  // sample actions in-kernel
  rbg_env_params env;
  int32_t *list;        // auto-reset list (device), may be NULL
  int32_t *list_count;  // device counter
  // speculative auto-reset (c_api.cu "AutoReset"): envs whose next episode is
  // already in the cache swap it in here; every finished env is queued for refill
  const unsigned long long *cache_tag;
  const uint2 *cache_key;
  const uint32_t *cache_pins;
  int32_t *refill_list;    // [B]
  int32_t *refill_count;   // [1]
  uint32_t *refill_keys;   // [B,2] State.key of the episode that just started
  // filled by launch_env
  int cells, E, Np;  // E envs per CTA, Np lanes per env
  int so[2];         // shared memory: [0] bytes of the observation table, [1] bytes of one warp's grid slice
  FastDiv divN, divG, divC4, divCells;
};

// pdl: launch with programmatic stream serialization (the kernel may begin while a preceding kernel that has said
// launch_dependents is still running; any other predecessor completes first)
int launch_env(EnvParams p, cudaStream_t stream, bool pdl = false);
// T random-policy steps in one launch, auto-reset from the board dataset of p.env; ts fields stacked [T,B,...]
int launch_rollout(EnvParams p, int T, int32_t *action_out, cudaStream_t stream);
// T random-policy steps with ParallelRandomWalk / Uniform auto-reset (kind) as a persistent kernel whose CTAs carry
// their own generator warps; needs the cache
// `counter`: 8 zeroed ints (two sets, recycled by the kernel); group_done / group_pending: zeroed int[groups];
// epoch: 1, 2, ... per launch on those arrays; overlap: chain to the previous launch of the stream (PDL)
int launch_rollout_persist(EnvParams p, int kind, int T, int32_t *action_out, int32_t *counter, int32_t *group_done, int32_t *group_pending,
                           int epoch, bool overlap, uint64_t *cache_tag_w, uint2 *cache_key_w, uint32_t *cache_pins_w, cudaStream_t stream);
int launch_random_actions(const rbg_state &st, int64_t B, int G, int N,
                          int32_t *action, cudaStream_t stream);
// every env of `in` to its first LAST step under the random policy (episode_warp_kernel); fin may be NULL
int launch_episodes(const rbg_state &in, const rbg_state *fin, const rbg_episode_metrics &out, int64_t B, int G, int N,
                    const rbg_env_params &env, cudaStream_t stream);
// one Connector.step of the envs whose live byte is set, their episode records accumulated in place (eval_step_kernel)
int launch_eval_step(const rbg_state &st, const int32_t *action, uint8_t *live, int32_t *live_count, int64_t B, int G, int N,
                     const rbg_env_params &env, const rbg_timestep &ts, const rbg_episode_metrics &acc, cudaStream_t stream);

// ---- misc kernels (misc_kernels.cu) --------------------------------------
int launch_split_keys(uint32_t k0, uint32_t k1, int64_t B, int64_t offset,
                      int64_t count, uint32_t *out, cudaStream_t stream);
int launch_split_each(const uint32_t *keys, int64_t B, int num, uint32_t *out, cudaStream_t stream);
int launch_dataset_state(const uint32_t *keys, int64_t B, int G, int N, const int32_t *heads, const int32_t *targets, int64_t K,
                         const rbg_state &st, cudaStream_t stream);
int launch_board_stats(const int32_t *boards, int64_t B, int G, int count_current_wire, int32_t *scored, int32_t *detours, int32_t *diversity,
                       cudaStream_t stream);
int launch_validate(const int32_t *boards, int64_t B, int G, int N,
                    int32_t *flags, cudaStream_t stream);
// int32 codes (< 256) -> bytes, for the host transport of the observation
int launch_narrow_codes(const int32_t *src, uint8_t *dst, int64_t n, cudaStream_t stream, int bits = 8);  // bits = 4: two codes < 16 per byte

// ---- host thread pool (host_pool.cpp): widens byte codes back to int32 in host memory ----
int host_pool_threads();                                          // workers in use (the pool is created on first use)
int host_pool_max_threads();                                      // workers that exist
bool host_pool_fixed();                                           // RBG_HOST_THREADS is set: no tuning
void host_pool_set_threads(int n);                                // workers that take pieces from now on
void host_pool_widen(const uint8_t *src, int32_t *dst, size_t n); // enqueue; split over the workers
void host_pool_widen4(const uint8_t *src, int32_t *dst, size_t n); // the same for two codes per byte (low nibble first), n even
void host_pool_wait();                                            // until every enqueued piece is done

// ---- seed extension (seedext_kernel.cu) ---------------------------------
struct SeedExtParams {
  const uint32_t *keys;
  long long B;
  int G, N;
  float randomness;
  int two_sided, iterations;
  long long ext_steps;  // < 0 unlimited
  int extra_split;
  int mode;  // 0 solved board, 1 starts/ends, 2 State
  int32_t *solved, *starts, *ends;
  rbg_state st;
  rbg_timestep ts;
  int observe;
  const int32_t *list;
  const int32_t *list_count;
  int solved_f32;  // mode 0: the codes as float32 (SequentialRandomWalkBoard.generate returns jnp.zeros' default dtype)
};
int launch_seedext(SeedExtParams p, int64_t max_boards, cudaStream_t stream);
void keep_pool_cached();  // cudaMallocAsync's default pool keeps its memory across synchronisations (scratch of the generators)
// se_finish_kernel on its own: boards[max_boards, CB] bytes (row-major G*G codes, CB = cells rounded up to 16) and
// gkey[max_boards, 2] (State.key) -> the outputs of p.mode (0 board, 1 first POSITION / TARGET cell per wire, 2 State
// (+ observation)); slot m of the scratch is board p.list[m] when p.list is set
int launch_board_finish(const SeedExtParams &p, const uint8_t *boards, const uint32_t *gkey, int CB, int64_t max_boards, int kernel_id,
                        cudaStream_t stream);

// ---- sequential random walk (seqrw_kernel.cu) ----------------------------
struct SeqRwParams {
  const uint32_t *keys;
  long long B;
  int G, N;
  int extra_split;
  int mode;         // 0 board, 1 starts/ends, 2 State
  int float_board;  // mode 0: float32 codes
  int32_t *board, *starts, *ends;
  int32_t *stats;  // optional [B,2]: attempt that succeeded (0 = none), its steps
  rbg_state st;
  rbg_timestep ts;
  int observe;
  const int32_t *list;
  const int32_t *list_count;
};
int launch_seqrw(SeqRwParams p, int64_t max_boards, cudaStream_t stream);

}  // namespace rbg
