// Learner-state copy of population-based training (Jaderberg et al., 2017): the "exploit" step copies the learner state of
// one agent over another's, the "explore" step rewrites some of the destination's hyper-parameters. Both are one launch of
// pbt_copy_kernel for a list of (source, destination) pairs.
//
// The learner state is two spans of an agent's arena block (build_layout, sacx_engine.cuh):
//   span 0  [scal_off, P0 + 3 blk): the scalar block, then the online parameters, Adam m and v (block.params / .m / .v)
//   span 1  [T0, T0 + align4(n_critic)): the target critics (block.targets)
// The gradient block (P0 + 3 blk, between the two spans), the batch, activation and delta buffers are per-update scratch and
// are not copied. A packed state is the two spans back to back; an endpoint is either an agent's arena block or a slot of a
// packed buffer, so one kernel serves the local copy (arena -> arena), the pack (arena -> buffer) and the unpack (buffer ->
// arena).
//
// When the destination is an arena block, the words of the scalar block that belong to the destination stay (scal_word_kept):
// the update counter and the RNG keys (the destination keeps drawing its own (seed, agent, counter) streams, so no triple is
// drawn twice), the metrics, the non-finite flag and the data-parallel shares (they report the destination's own last update).
// A pair's hyper-parameter record is written after the copy by the CTA that copied the scalar block.
#pragma once
#include <stddef.h>

#include "../../include/sacx.h"
#include "sacx_types.cuh"

namespace sacx {

static_assert(sizeof(AgentScalars) % 16 == 0, "the scalar block is copied in 16-byte words");
constexpr int SCAL_WORDS = (int)(sizeof(AgentScalars) / 4);

__host__ __device__ constexpr bool scal_word_kept(int w) {
  return (w >= (int)(offsetof(AgentScalars, updates) / 4) && w < (int)(offsetof(AgentScalars, alpha_lr) / 4)) ||
         (w >= (int)(offsetof(AgentScalars, metrics) / 4) && w < (int)(offsetof(AgentScalars, lr) / 4)) ||
         w >= (int)(offsetof(AgentScalars, rng_agent) / 4);
}

struct PbtPair {
  int src, dst;            // agent (arena endpoint) or slot (buffer endpoint)
  sacx_pbt_record rec;     // rec.set == 0: no record
};

struct PbtEnd {
  float* base;
  i64 stride;              // floats between consecutive agents / slots
  i64 off0, off1;          // float offsets of span 0 and span 1 inside an agent block / slot
};

constexpr int PBT_THREADS = 256;
constexpr int PBT_UNROLL = 4;                                   // 16-byte words in flight per thread
constexpr int PBT_CHUNK = PBT_THREADS * PBT_UNROLL;             // 16-byte words per CTA (16 KB)

// grid (ceil((n0 + n1) / PBT_CHUNK), min(n_pairs, 65535)); n0 / n1 are the spans' lengths in 16-byte words
__global__ void __launch_bounds__(PBT_THREADS) pbt_copy_kernel(PbtEnd src, PbtEnd dst, i64 n0, i64 n1, int dst_arena,
                                                              const PbtPair* __restrict__ pairs, int n_pairs) {
  const i64 n4 = n0 + n1;
  const i64 base = (i64)blockIdx.x * PBT_CHUNK + threadIdx.x;
  for (int p = blockIdx.y; p < n_pairs; p += gridDim.y) {
    const int ps = pairs[p].src, pd = pairs[p].dst;
    const float* s = src.base + (i64)ps * src.stride;
    float* d = dst.base + (i64)pd * dst.stride;
    float4 v[PBT_UNROLL];
#pragma unroll
    for (int u = 0; u < PBT_UNROLL; ++u) {
      const i64 i = base + (i64)u * PBT_THREADS;
      if (i < n4) {
        const float* sp = i < n0 ? s + src.off0 + 4 * i : s + src.off1 + 4 * (i - n0);
        v[u] = __ldg(reinterpret_cast<const float4*>(sp));
      }
    }
#pragma unroll
    for (int u = 0; u < PBT_UNROLL; ++u) {
      const i64 i = base + (i64)u * PBT_THREADS;
      if (i < n4) {
        float* dp = i < n0 ? d + dst.off0 + 4 * i : d + dst.off1 + 4 * (i - n0);
        float4 w = v[u];
        if (dst_arena && i < SCAL_WORDS / 4) {
          const float4 keep = *reinterpret_cast<const float4*>(dp);
          const int w0 = 4 * (int)i;
          if (scal_word_kept(w0)) w.x = keep.x;
          if (scal_word_kept(w0 + 1)) w.y = keep.y;
          if (scal_word_kept(w0 + 2)) w.z = keep.z;
          if (scal_word_kept(w0 + 3)) w.w = keep.w;
        }
        *reinterpret_cast<float4*>(dp) = w;
      }
    }
    if (dst_arena && blockIdx.x == 0 && pairs[p].rec.set) {   // uniform per CTA
      __syncthreads();                                         // the scalar block of this pair is copied (CTA 0, threads 0-13)
      if (threadIdx.x == 0) {
        const sacx_pbt_record r = pairs[p].rec;
        AgentScalars* sc = reinterpret_cast<AgentScalars*>(d + dst.off0);
        if (r.set & SACX_PBT_ALPHA) { sc->log_alpha = r.log_alpha; sc->alpha = r.alpha; sc->alpha_f32 = r.alpha_f32; }
        if (r.set & SACX_PBT_ALPHA_LR) sc->alpha_lr = r.alpha_lr;
        if (r.set & SACX_PBT_ACTOR_LR) sc->lr[0] = r.actor_lr;
        if (r.set & SACX_PBT_CRITIC_LR) { sc->lr[1] = r.critic_lr; sc->lr[2] = r.critic_lr; }
        if (r.set & SACX_PBT_TAU) { sc->tau = r.tau; sc->one_minus_tau = r.one_minus_tau; }
        if (r.set & SACX_PBT_GAMMA) sc->gamma = r.gamma;
      }
    }
  }
}

}  // namespace sacx
