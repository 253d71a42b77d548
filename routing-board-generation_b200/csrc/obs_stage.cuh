// obs_stage.cuh -- the per-agent observation views of a warp's envs, built in shared memory and
// written to global memory by bulk asynchronous copies (cp.async.bulk, SASS UBLKCP.G.S).
//
// observation.grid[e, a] is the env's grid with the wire codes rotated so that agent a sees
// itself as agent 0 (jumanji==0.2.2 Connector._obs_from_grid; UPSTREAM).  A warp owns K
// consecutive envs, so its part of observation.grid is ONE contiguous range of
// K * N * G * G int32: it is staged in that layout and leaves as a few large copies that
// the LSU queue never sees (DESIGN.md "K2b" explains why that matters).  Used by the
// per-step kernel and the fused rollout kernel (connector_kernel.cu).
#pragma once

#include "rbg_device.cuh"

namespace rbg {

// The fused rollout kernel uses ONE stride for every N (codes 0..96), so that the per-agent
// table rows sit at compile-time offsets from the four cell addresses of a packed word.
constexpr int OBS_RS = 100;

// four cells (one packed word) -> the same four cells in every agent's view: per agent four
// table bytes and one 128-bit store, nothing else (views are c4 int4 apart).
__device__ __forceinline__ void emit_views(const uint8_t *lut, uint32_t w, int N, int4 *o, int c4) {
  const uint8_t *l0 = lut + (w & 0xffu), *l1 = lut + ((w >> 8) & 0xffu), *l2 = lut + ((w >> 16) & 0xffu), *l3 = lut + (w >> 24);
  int x = N;
  for (; x >= 4; x -= 4) {
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      *o = make_int4(l0[u * OBS_RS], l1[u * OBS_RS], l2[u * OBS_RS], l3[u * OBS_RS]);
      o += c4;
    }
    l0 += 4 * OBS_RS;
    l1 += 4 * OBS_RS;
    l2 += 4 * OBS_RS;
    l3 += 4 * OBS_RS;
  }
  if (x & 2) {
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      *o = make_int4(l0[u * OBS_RS], l1[u * OBS_RS], l2[u * OBS_RS], l3[u * OBS_RS]);
      o += c4;
    }
    l0 += 2 * OBS_RS;
    l1 += 2 * OBS_RS;
    l2 += 2 * OBS_RS;
    l3 += 2 * OBS_RS;
  }
  if (x & 1) *o = make_int4(l0[0], l1[0], l2[0], l3[0]);
}


// Shared-memory accesses by 32-bit shared address: the staged observation loop keeps its three
// base addresses (packed grid words, table, staging) in registers instead of letting the
// compiler rebuild them from threadIdx in every iteration.
__device__ __forceinline__ uint32_t lds_u32(uint32_t a) {
  uint32_t v;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(a));
  return v;
}
template <int OFF>
__device__ __forceinline__ uint32_t lds_u8(uint32_t a) {
  uint32_t v;
  asm volatile("ld.shared.u8 %0, [%1+%2];" : "=r"(v) : "r"(a), "n"(OFF));
  return v;
}
__device__ __forceinline__ void sts_v4(uint32_t a, uint32_t x, uint32_t y, uint32_t z, uint32_t w) {
  asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"(a), "r"(x), "r"(y), "r"(z), "r"(w) : "memory");
}
__device__ __forceinline__ uint32_t opaque(uint32_t v) {  // the compiler may not re-derive v
  asm volatile("" : "+r"(v));
  return v;
}
template <int U>
__device__ __forceinline__ void stage_view(uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t o) {
  sts_v4(o, lds_u8<U * OBS_RS>(a0), lds_u8<U * OBS_RS>(a1), lds_u8<U * OBS_RS>(a2), lds_u8<U * OBS_RS>(a3));
}
// four cells (packed word w) -> the same four cells of nv consecutive agents' views, staged at
// shared address o with views vs bytes apart; lut_s = shared address of the first agent's table row
__device__ __forceinline__ void stage_views(uint32_t lut_s, uint32_t w, int nv, uint32_t o, uint32_t vs) {
  uint32_t a0 = lut_s + (w & 0xffu), a1 = lut_s + ((w >> 8) & 0xffu), a2 = lut_s + ((w >> 16) & 0xffu), a3 = lut_s + (w >> 24);
  int x = nv;
  for (; x >= 4; x -= 4) {
    stage_view<0>(a0, a1, a2, a3, o);
    stage_view<1>(a0, a1, a2, a3, o + vs);
    stage_view<2>(a0, a1, a2, a3, o + 2 * vs);
    stage_view<3>(a0, a1, a2, a3, o + 3 * vs);
    a0 += 4 * OBS_RS;
    a1 += 4 * OBS_RS;
    a2 += 4 * OBS_RS;
    a3 += 4 * OBS_RS;
    o += 4 * vs;
  }
  if (x & 2) {
    stage_view<0>(a0, a1, a2, a3, o);
    stage_view<1>(a0, a1, a2, a3, o + vs);
    a0 += 2 * OBS_RS;
    a1 += 2 * OBS_RS;
    a2 += 2 * OBS_RS;
    a3 += 2 * OBS_RS;
    o += 2 * vs;
  }
  if (x & 1) stage_view<0>(a0, a1, a2, a3, o);
}

// the same with the agent count known at compile time: straight-line code
template <int NV>
__device__ __forceinline__ void stage_views_fixed(uint32_t lut_s, uint32_t w, uint32_t o, uint32_t vs) {
  const uint32_t a0 = lut_s + (w & 0xffu), a1 = lut_s + ((w >> 8) & 0xffu), a2 = lut_s + ((w >> 16) & 0xffu), a3 = lut_s + (w >> 24);
  stage_view<0>(a0, a1, a2, a3, o);
  if (NV > 1) stage_view<1>(a0, a1, a2, a3, o += vs);
  if (NV > 2) stage_view<2>(a0, a1, a2, a3, o += vs);
  if (NV > 3) stage_view<3>(a0, a1, a2, a3, o += vs);
  if (NV > 4) stage_view<4>(a0, a1, a2, a3, o += vs);
  if (NV > 5) stage_view<5>(a0, a1, a2, a3, o += vs);
  if (NV > 6) stage_view<6>(a0, a1, a2, a3, o += vs);
  if (NV > 7) stage_view<7>(a0, a1, a2, a3, o += vs);
}

// Bulk asynchronous copy shared -> global (the TMA unit moves the bytes, the LSU queue does not
// see them).  Issued by one lane; the buffer may be rewritten once its group has been READ.
__device__ __forceinline__ void bulk_store(void *gdst, uint32_t ssrc, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gdst), "r"(ssrc), "r"(bytes) : "memory");
  asm volatile("cp.async.bulk.commit_group;" ::: "memory");
}
template <int PENDING>
__device__ __forceinline__ void bulk_wait_read() {
  asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(PENDING) : "memory");
}


// How a warp's observation range is cut into staged chunks (host side, launch_env / launch_rollout):
// the whole range if it is at most `whole` bytes (one buffer; the caller guarantees that enough
// time passes before it is refilled or waits), else two alternating buffers of about `target`
// bytes holding a whole number of envs, or of views of one env.
struct ObsStagePlan {
  int bytes;  // per buffer
  int nbuf;   // 1 or 2; 0 = do not stage, store directly (a chunk would be a single view)
  int ce;     // envs per chunk (cv == N)
  int cv;     // views per chunk (ce == 1) or N
};
inline ObsStagePlan obs_stage_plan(int K, int N, int cells, size_t target, size_t whole) {
  ObsStagePlan pl;
  const size_t view = (size_t)cells * 4, envb = view * N;
  pl.nbuf = 1;
  pl.ce = 1;
  pl.cv = N;
  if ((size_t)K * envb <= whole) {
    pl.ce = K;
    pl.bytes = (int)(K * envb);
  } else if (envb <= target) {
    pl.nbuf = 2;
    pl.ce = (int)(target / envb) < K ? (int)(target / envb) : K;
    pl.bytes = (int)(pl.ce * envb);
  } else {
    pl.nbuf = 2;
    pl.cv = view >= target ? 1 : (int)(target / view);
    if (pl.cv > N) pl.cv = N;
    pl.bytes = (int)(pl.cv * view);
    if (pl.cv < 2 && N > 1) {
      pl.nbuf = 0;
      pl.bytes = 0;
    }
  }
  return pl;
}

// Per-warp state of the staged writer.  Word q = m * c4 + rem of the warp's packed grids (4 cells
// each) goes to int4 slot m * N * c4 + rem of the warp's first env's first view.
struct ObsStager {
  uint32_t stage_s, lut_s, wq_s, view_b;  // shared addresses: staging, table, this lane's first word; bytes per view
  int stage_bytes, nbuf, ce, cv;
  int rem0, off0, q_rem, q_off, q_wrap;
  int buf;

  __device__ __forceinline__ void init(const uint8_t *stage, const uint8_t *lut, const uint32_t *wg32, int N, int c4, const FastDiv &divC4,
                                       int lane, int stage_bytes_, int nbuf_, int ce_, int cv_) {
    stage_s = opaque((uint32_t)__cvta_generic_to_shared(stage));
    lut_s = opaque((uint32_t)__cvta_generic_to_shared(lut));
    wq_s = opaque((uint32_t)__cvta_generic_to_shared(wg32) + 4u * (uint32_t)lane);
    view_b = (uint32_t)c4 * 16u;
    stage_bytes = stage_bytes_;
    nbuf = nbuf_;
    ce = ce_;
    cv = cv_;
    const int m0 = (int)divC4.div((uint32_t)lane), qm = (int)divC4.div(32u);
    rem0 = lane - m0 * c4;
    off0 = m0 * N * c4 + rem0;
    q_rem = 32 - qm * c4;
    q_off = qm * N * c4 + q_rem;
    q_wrap = (N - 1) * c4;
    buf = 0;
  }

  // the words of one chunk -> its staging buffer; NV = views per word when known at compile time, else 0
  template <int NV>
  __device__ __forceinline__ void fill(uint32_t row, uint32_t wq, uint32_t sb, int nw, int nv, int c4, int lane) const {
    uint32_t o = sb + 16u * (uint32_t)off0;
    int rem = rem0;
    for (int q = lane; q < nw; q += 32) {
      const uint32_t w = lds_u32(wq);
      if (NV > 0)
        stage_views_fixed<(NV > 0 ? NV : 1)>(row, w, o, view_b);
      else
        stage_views(row, w, nv, o, view_b);
      wq += 128u;
      rem += q_rem;  // word q + 32: same env or the next one(s)
      o += 16u * (uint32_t)q_off;
      if (rem >= c4) {
        rem -= c4;
        o += 16u * (uint32_t)q_wrap;
      }
    }
  }

  // all 32 lanes: stage and send the views of the warp's kc envs to odst (int4 units, 16-byte aligned)
  __device__ __forceinline__ void emit(int kc, int N, int c4, int lane, int4 *odst) {
    for (int m0 = 0; m0 < kc; m0 += ce) {
      const int nenv = min(ce, kc - m0), nw = nenv * c4;
      for (int x0 = 0; x0 < N; x0 += cv) {
        const int nv = min(cv, N - x0);
        if (lane == 0) {  // the buffer about to be filled has been read
          if (nbuf == 1)
            bulk_wait_read<0>();
          else
            bulk_wait_read<1>();
        }
        __syncwarp();
        const uint32_t sb = stage_s + (uint32_t)(buf * stage_bytes);
        const uint32_t row = lut_s + (uint32_t)(x0 * OBS_RS);
        const uint32_t wq = wq_s + 4u * (uint32_t)(m0 * c4);
        switch (nv) {  // warp-uniform; the agent count of the common cases is a compile-time constant
          case 2: fill<2>(row, wq, sb, nw, 2, c4, lane); break;
          case 3: fill<3>(row, wq, sb, nw, 3, c4, lane); break;
          case 4: fill<4>(row, wq, sb, nw, 4, c4, lane); break;
          case 5: fill<5>(row, wq, sb, nw, 5, c4, lane); break;
          case 6: fill<6>(row, wq, sb, nw, 6, c4, lane); break;
          case 7: fill<7>(row, wq, sb, nw, 7, c4, lane); break;
          case 8: fill<8>(row, wq, sb, nw, 8, c4, lane); break;
          default: fill<0>(row, wq, sb, nw, nv, c4, lane);
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        __syncwarp();
        if (lane == 0) bulk_store(odst + (size_t)(m0 * N + x0) * c4, sb, (uint32_t)(((nenv - 1) * N + nv) * c4) * 16u);
        buf ^= nbuf - 1;
      }
    }
  }

  // the same views by direct 128-bit stores: for boards whose views are so large that a staged chunk
  // would hold a single view (32x32: 4 KB), where re-reading the packed words once per view costs
  // more than the bulk copies save (measured: 32x32/16 82.6 M env-steps/s direct, 69 M staged;
  // 20x20/10 with two views per chunk 356 M staged, 321 M direct)
  __device__ __forceinline__ void emit_direct(const uint8_t *lut, const uint32_t *wg32, int kc, int N, int c4, int lane, int4 *odst) const {
    int rem = rem0, off = off0;
    for (int q = lane; q < kc * c4; q += 32) {
      emit_views(lut, wg32[q], N, odst + off, c4);
      rem += q_rem;
      off += q_off;
      if (rem >= c4) {
        rem -= c4;
        off += q_wrap;
      }
    }
  }

  // shared memory must outlive the copies: before the staging is reused for anything else, and before exit
  __device__ __forceinline__ void drain(int lane) {
    if (lane == 0) bulk_wait_read<0>();
    __syncwarp();
  }
};

}  // namespace rbg
