// rbg_device.cuh -- device-side building blocks shared by all kernels.
//
// threefry2x32 exactly as jax==0.4.8 (jax/_src/prng.py, Random123 20 rounds,
// jax_threefry_partitionable=False), the jax.random derivations used on the
// hot path (split halves, uniform, randint for power-of-two spans), cell
// encodings (reference seed_extension.py:39-44) and small helpers.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/rbg_b200.h"

namespace rbg {

enum : int { EMPTY = 0, PATH = 1, POSITION = 2, TARGET = 3 };
enum : int { NOOP = 0, UP = 1, RIGHT = 2, DOWN = 3, LEFT = 4 };

constexpr uint32_t FULL = 0xffffffffu;

__device__ __forceinline__ uint32_t rotl(uint32_t x, int r) {
  return __funnelshift_l(x, x, r);
}

// Plain additions: moving them to the FMA pipe as IMADs measured slower on B200 (ParallelRandomWalk 10x10/5
// 267 M vs 283 M boards/s, SeedExtension 14x14/7 7.26 M vs 7.68 M boards/s; DESIGN.md §7).  The
// add -> rotate -> xor chain is bound by dependent-issue latency, not by ALU-pipe throughput, and a
// cross-pipe dependency costs one extra cycle per round.
#define RBG_TF_ADD(a, b) ((a) + (b))

#define RBG_TF_ROUND(r)    \
  x0 = RBG_TF_ADD(x0, x1); \
  x1 = rotl(x1, r);        \
  x1 ^= x0;

// One threefry2x32 block: key (k0,k1), counter (x0,x1) -> (o0,o1).
__device__ __forceinline__ void tf_block(uint32_t k0, uint32_t k1, uint32_t x0,
                                         uint32_t x1, uint32_t &o0,
                                         uint32_t &o1) {
  const uint32_t ks2 = k0 ^ k1 ^ 0x1BD11BDAu;
  x0 = RBG_TF_ADD(x0, k0);
  x1 = RBG_TF_ADD(x1, k1);
  RBG_TF_ROUND(13) RBG_TF_ROUND(15) RBG_TF_ROUND(26) RBG_TF_ROUND(6)
  x0 = RBG_TF_ADD(x0, k1);
  x1 = RBG_TF_ADD(x1, ks2 + 1u);
  RBG_TF_ROUND(17) RBG_TF_ROUND(29) RBG_TF_ROUND(16) RBG_TF_ROUND(24)
  x0 = RBG_TF_ADD(x0, ks2);
  x1 = RBG_TF_ADD(x1, k0 + 2u);
  RBG_TF_ROUND(13) RBG_TF_ROUND(15) RBG_TF_ROUND(26) RBG_TF_ROUND(6)
  x0 = RBG_TF_ADD(x0, k0);
  x1 = RBG_TF_ADD(x1, k1 + 3u);
  RBG_TF_ROUND(17) RBG_TF_ROUND(29) RBG_TF_ROUND(16) RBG_TF_ROUND(24)
  x0 = RBG_TF_ADD(x0, k1);
  x1 = RBG_TF_ADD(x1, ks2 + 4u);
  RBG_TF_ROUND(13) RBG_TF_ROUND(15) RBG_TF_ROUND(26) RBG_TF_ROUND(6)
  x0 = RBG_TF_ADD(x0, ks2);
  x1 = RBG_TF_ADD(x1, k0 + 5u);
  o0 = x0;
  o1 = x1;
}

// split(key) = [(o0(0,2), o0(1,3)), (o1(0,2), o1(1,3))]; both halves, one thread.
__device__ __forceinline__ void split2(uint32_t k0, uint32_t k1, uint32_t &a0,
                                       uint32_t &a1, uint32_t &b0,
                                       uint32_t &b1) {
  uint32_t p0, p1, q0, q1;
  tf_block(k0, k1, 0u, 2u, p0, p1);
  tf_block(k0, k1, 1u, 3u, q0, q1);
  a0 = p0;
  a1 = q0;
  b0 = p1;
  b1 = q1;
}

// random_bits(key, 32, ()) = block(key; 0, 0).o0
__device__ __forceinline__ uint32_t bits_scalar(uint32_t k0, uint32_t k1) {
  uint32_t o0, o1;
  tf_block(k0, k1, 0u, 0u, o0, o1);
  return o0;
}

// jax.random.uniform float32 from 32 random bits
__device__ __forceinline__ float bits_to_uniform(uint32_t bits) {
  return __fsub_rn(__uint_as_float((bits >> 9) | 0x3F800000u), 1.0f);
}

// randint(key, (), 0, span) for span a power of two <= 2^16: the multiplier
// (2^16 % span)^2 % span is 0, so only the low draw of the second split half
// matters: random_bits(split(key)[1]) & (span-1).
__device__ __forceinline__ uint32_t randint_pow2(uint32_t k0, uint32_t k1,
                                                 uint32_t span) {
  uint32_t a0, a1, b0, b1;
  split2(k0, k1, a0, a1, b0, b1);
  return bits_scalar(b0, b1) & (span - 1u);
}

// BoardDatasetGeneratorJAX.__call__ (rl_training/offline_generation/dataset_generator_jax.py:112-141):
// `key, _ = split(key)` -> State.key (nk0, nk1); `which = randint(key, (), 0, K)` with jax's two-draw
// formula (SURVEY A.9): k1, k2 = split(key); ((bits(k1) % K) * ((2^16 % K)^2 % K) + bits(k2) % K) % K
// in uint32 wrap-around arithmetic.
__device__ __forceinline__ uint32_t dataset_pick(uint32_t k0, uint32_t k1, uint32_t K,
                                                 uint32_t &nk0, uint32_t &nk1) {
  uint32_t b0, b1, h0, h1, l0, l1;
  split2(k0, k1, nk0, nk1, b0, b1);
  split2(nk0, nk1, h0, h1, l0, l1);
  const uint32_t hi = bits_scalar(h0, h1), lo = bits_scalar(l0, l1);
  uint32_t mult = 65536u % K;
  mult = (uint32_t)(((unsigned long long)mult * mult) % K);
  return ((hi % K) * mult + (lo % K)) % K;
}

// "Same destination -> only the highest agent id moves" (parallel_random_walk.py:104-145, jumanji
// Connector._step_agents) inside a group of W lanes that starts at lane `base`, lane = agent: a mover
// loses iff a HIGHER agent of its group moves to the same cell.  N shuffles; __match_any_sync, which
// this replaces, serialises over the distinct values of the warp (one per non-moving lane as well) and was
// the largest single stall of the latency-bound walk (profiles/r01d_prw_bulk_source_top.txt,
// profiles/r02a_persist_source_top.txt).  `val` must be unique per lane for non-movers.
__device__ __forceinline__ bool wins_collision(uint32_t val, bool moves, int a, int base, int N) {
  bool lose = false;
  for (int i = 1; i < N; ++i) {  // agent 0 never beats anyone
    const uint32_t o = __shfl_sync(FULL, val, base + i);
    lose |= (i > a) && (o == val);
  }
  return moves && !lose;
}

// global-memory flag with release / acquire semantics at GPU scope (cheaper than __threadfence pairs)
__device__ __forceinline__ void st_release_u64(unsigned long long *p, unsigned long long v) {
  asm volatile("st.release.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned long long ld_acquire_u64(const unsigned long long *p) {
  unsigned long long v;
  asm volatile("ld.acquire.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}

__device__ __forceinline__ void st_release_s32(int *p, int v) {
  asm volatile("st.release.gpu.global.s32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ int ld_acquire_s32(const int *p) {
  int v;
  asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}

// exact n / d for n*d < 2^32 (host checks the range), d >= 1
struct FastDiv {
  uint32_t mul;
  uint32_t d;
  __host__ static FastDiv make(uint32_t d) {
    FastDiv f;
    f.d = d;
    f.mul = d <= 1 ? 0u : (uint32_t)((((uint64_t)1 << 32) + d - 1) / d);
    return f;
  }
  __device__ __forceinline__ uint32_t div(uint32_t n) const {
    return d <= 1 ? n : __umulhi(n, mul);
  }
  __device__ __forceinline__ void divmod(uint32_t n, uint32_t &q,
                                         uint32_t &r) const {
    q = div(n);
    r = n - q * d;
  }
};

__device__ __forceinline__ int4 bytes_to_int4(uint32_t w) {
  return make_int4((int)(w & 0xffu), (int)((w >> 8) & 0xffu),
                   (int)((w >> 16) & 0xffu), (int)(w >> 24));
}

// Connector per-agent observation value (JUM env.py _obs_from_grid): own
// codes become 1,2,3, other agents are shifted cyclically.
__device__ __forceinline__ int obs_value(int v, int a3, int n3) {
  int t = v - a3;
  t += (t < 1) ? n3 : 0;
  return v == 0 ? 0 : t;
}

// true when v in {3a+1, 3a+2, 3a+3}; base = 3a+1
__device__ __forceinline__ bool own_wire(uint32_t v, uint32_t base) {
  return (v - base) < 3u;
}

}  // namespace rbg
