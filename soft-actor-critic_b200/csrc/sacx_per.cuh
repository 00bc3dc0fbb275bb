// Prioritized experience replay (Schaul et al., 2016) over the device ring: a sum/min tree of fan-out 32 over the ring's
// slots, the stratified proportional sampler, the importance weights and the priority write-back. One cooperative kernel
// (per_refresh_kernel) does all tree work of one call in a fixed phase order separated by grid barriers:
//   1. write-back keys: priority p = (delta + eps)^alpha of every written row; p_max <- max(p_max, p); per slot the highest row
//      index claims the slot (64-bit atomicMax of (epoch << 32 | row): which row wins does not depend on scheduling);
//   2. leaves: the winning rows store p; slots pushed since the tree last looked at the ring header get p_max (lazily: every
//      producer -- host staging flush, push_n_dev, the DonkeyVae assembler -- only advances RingMeta.pushes); more than one
//      ring's worth of pushes, or a push counter that went backwards (ring image loaded), resets every leaf;
//   3. one level per barrier: every touched internal node is recomputed from its 32 children in a fixed order (xor butterfly).
//      No atomicAdd deltas: a node is a pure function of its children, so replicas, bursts and a rebuilt tree are bit-identical;
//   4. sampling: one warp per row walks root -> leaf, 32 children (one 128-byte read) per level; a slot with p = 0 is never
//      taken (oracle/per_numpy.py walk_f32 restates the walk bit for bit).
// Leaves are the priorities themselves ([cap] floats, 0 = empty slot); level l >= 1 holds (sum, min) of groups of 32 nodes of
// level l - 1 as two arrays; an empty leaf counts as (0, +inf) in the min.
#pragma once
#include <cooperative_groups.h>
#include <stdint.h>

#include "sacx_math.cuh"
#include "sacx_types.cuh"

namespace sacx {

constexpr int PER_FANOUT = 32;
constexpr int PER_MAX_LEVELS = 8;          // 32^7 > any int64 ring that fits a device

struct PerState {                          // device-resident, one per tree
  i64 seen;                                // ring pushes the leaves reflect
  i64 sample_oldest;                       // oldest slot at the most recent sample: logical index -> slot of a later write-back
  unsigned pmax_bits;                      // p_max as float bits (positive floats order like their bits)
  unsigned pad;
};

struct PerArgs {
  float* leaf;                             // [cap]
  float* sum[PER_MAX_LEVELS + 1];          // [1..depth]
  float* mn[PER_MAX_LEVELS + 1];
  unsigned* mark[PER_MAX_LEVELS + 1];      // claim marks of the incremental propagation (value = epoch of the last claim)
  i64 nodes[PER_MAX_LEVELS + 1];           // nodes[0] = cap, nodes[depth] = 1
  int depth;
  unsigned epoch;                          // distinct per launch (claims, write-back keys)
  unsigned long long* win;                 // [cap] write-back winner keys
  PerState* st;
  const RingMeta* hdr;                     // the ring block's header: device push counter
  i64 cap;
  int rebuild;                             // recompute every internal node (after the leaves were loaded)
  // write-back: rows [0, wb_n); slot from wb_idx (logical, against st->sample_oldest) or wb_slots; delta given or from q1/q2/y
  int wb_n;
  const i64* wb_idx;
  const i64* wb_slots;
  const float* wb_delta;
  const float *wb_q1, *wb_q2, *wb_y;
  float alpha, eps;
  // sampling: rows [0, B)
  int B;
  const float* u_ext;                      // [B] uniforms in [0, 1), or null -> Philox
  unsigned long long seed, counter;
  unsigned agent;
  float beta;
  const AgentScalars* scal;                // non-null: seed / agent / counter / beta schedule come from the agent's scalars
  double beta0;
  i64 beta_steps;
  i64* out_idx;                            // [B] logical indices ((slot - oldest) mod cap, the idx_ext format)
  float* out_w;                            // [B] importance weights
  i64* out_slots;                          // [B] slots (deferred write-back of an agent update)
};

// U[0, 1) for row k of update `counter`: its own Philox stream (word 3 tag 0x7E, never used by the normal / index / rollout streams)
__device__ __forceinline__ float per_uniform(unsigned long long seed, unsigned long long counter, uint32_t k, uint32_t agent) {
  uint32_t o[4];
  philox4x32_10((uint32_t)counter, (uint32_t)(counter >> 32), k, 0x7E000000u, (uint32_t)seed ^ (agent * 0x9E3779B9u),
                (uint32_t)(seed >> 32) ^ 0x5AC5AC5Au, o);
  return (float)(o[0] >> 8) * 5.9604644775390625e-8f;       // 24 bits: exactly representable, < 1
}

__device__ __forceinline__ i64 per_wb_slot(const PerArgs& a, int k, i64 len) {
  if (a.wb_idx) {
    const i64 j = a.wb_idx[k];
    if (j < 0 || j >= len) return -1;                         // out-of-range positions are ignored
    i64 s = a.st->sample_oldest + j;
    return s >= a.cap ? s - a.cap : s;
  }
  return a.wb_slots[k];
}

__device__ __forceinline__ float per_wb_priority(const PerArgs& a, int k) {
  float d;
  if (a.wb_delta) d = fabsf(a.wb_delta[k]);
  else {
    const float y = a.wb_y[k];
    d = 0.5f * (fabsf(a.wb_q1[k] - y) + fabsf(a.wb_q2[k] - y));
  }
  return powf(d + a.eps, a.alpha);
}

// (sum, min) of node `node` of level l from its 32 children; lane 0 stores. The butterfly order is part of the format: a host
// recomputation (tests) and every replica follow it.
__device__ __forceinline__ void per_node(const PerArgs& a, int l, i64 node, int lane) {
  const i64 c = node * PER_FANOUT + lane, nc = a.nodes[l - 1];
  float s = 0.f, m = INFINITY;
  if (c < nc) {
    if (l == 1) { s = a.leaf[c]; m = s > 0.f ? s : INFINITY; }
    else { s = a.sum[l - 1][c]; m = a.mn[l - 1][c]; }
  }
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) {
    s += __shfl_xor_sync(0xffffffffu, s, off);
    m = fminf(m, __shfl_xor_sync(0xffffffffu, m, off));
  }
  if (lane == 0) { a.sum[l][node] = s; a.mn[l][node] = m; }
}

__global__ void __launch_bounds__(256) per_refresh_kernel(PerArgs a) {
  namespace cg = cooperative_groups;
  cg::grid_group g = cg::this_grid();
  const int lane = threadIdx.x & 31;
  const i64 gt = (i64)blockIdx.x * blockDim.x + threadIdx.x, nt = (i64)gridDim.x * blockDim.x;
  const i64 gw = gt >> 5, nw = nt >> 5;
  const i64 cap = a.cap;
  const i64 pushes = *(volatile const i64*)&a.hdr->pushes, seen = *(volatile const i64*)&a.st->seen;
  const i64 len = pushes < cap ? pushes : cap;
  const i64 n_new = pushes - seen;
  const bool reset = n_new < 0 || n_new >= cap;
  const i64 seen_slot = reset ? 0 : seen % cap;
  auto is_new = [&](i64 s) { i64 d = s - seen_slot; if (d < 0) d += cap; return d < n_new; };

  // (every condition that skips a phase below is the same in all threads: the grid barriers stay matched)
  // 1. write-back keys and p_max
  if (a.wb_n > 0) {
    for (i64 k = gt; k < a.wb_n; k += nt) {
      const i64 s = per_wb_slot(a, (int)k, len);
      if (s < 0) continue;
      const float p = per_wb_priority(a, (int)k);
      if (p == p) atomicMax(&a.st->pmax_bits, __float_as_uint(p));
      atomicMax(&a.win[s], ((unsigned long long)a.epoch << 32) | (unsigned long long)k);
    }
    g.sync();
  }
  // 2. leaves
  const float pmax = __uint_as_float(*(volatile unsigned*)&a.st->pmax_bits);
  if (!reset)
    for (i64 k = gt; k < a.wb_n; k += nt) {
      const i64 s = per_wb_slot(a, (int)k, len);
      if (s < 0 || is_new(s) || a.win[s] != (((unsigned long long)a.epoch << 32) | (unsigned long long)k)) continue;
      a.leaf[s] = per_wb_priority(a, (int)k);
    }
  if (reset) {
    for (i64 s = gt; s < cap; s += nt) a.leaf[s] = s < len ? pmax : 0.f;
  } else {
    for (i64 i = gt; i < n_new; i += nt) { i64 s = seen_slot + i; if (s >= cap) s -= cap; a.leaf[s] = pmax; }
  }
  const bool full = reset || a.rebuild;
  const i64 items = a.wb_n + (full ? 0 : n_new);
  if (full || items > 0) g.sync();
  // 3. internal levels
  for (int l = 1; l <= a.depth && (full || items > 0); ++l) {
    const int shift = 5 * l;
    if (full) {
      for (i64 node = gw; node < a.nodes[l]; node += nw) per_node(a, l, node, lane);
    } else {
      for (i64 it = gw; it < items; it += nw) {
        i64 s;
        if (it < a.wb_n) { s = per_wb_slot(a, (int)it, len); if (s < 0) continue; }
        else { s = seen_slot + (it - a.wb_n); if (s >= cap) s -= cap; }
        const i64 node = s >> shift;
        unsigned claimed = 0;
        if (lane == 0) claimed = atomicExch(&a.mark[l][node], a.epoch) != a.epoch;
        if (__shfl_sync(0xffffffffu, claimed, 0)) per_node(a, l, node, lane);
      }
    }
    g.sync();
  }
  // every thread read st->seen before its first barrier (and without a barrier in this launch nothing was pushed: the store
  // below does not change it)
  if (gt == 0) a.st->seen = pushes;
  // 4. sampling
  if (a.B <= 0) return;
  unsigned long long seed = a.seed, counter = a.counter;
  unsigned agent = a.agent;
  float beta = a.beta;
  if (a.scal) {
    seed = a.scal->rng_seed; agent = a.scal->rng_agent;
    const i64 t = a.scal->updates;
    counter = (unsigned long long)t;
    beta = a.beta_steps > 0 ? (float)fmin(1.0, a.beta0 + (1.0 - a.beta0) * (double)t / (double)a.beta_steps) : (float)a.beta0;
  }
  const float total = a.sum[a.depth][0], pmin = a.mn[a.depth][0];
  const i64 oldest = pushes > cap ? pushes % cap : 0;
  for (i64 k = gw; k < a.B; k += nw) {
    const float U = a.u_ext ? a.u_ext[k] : per_uniform(seed, counter, (uint32_t)k, agent);
    float u = ((float)k + U) / (float)a.B * total;
    i64 node = 0;
    for (int l = a.depth; l >= 1; --l) {
      const i64 c = node * PER_FANOUT + lane;
      const float v = c < a.nodes[l - 1] ? (l == 1 ? a.leaf[c] : a.sum[l - 1][c]) : 0.f;
      float sc = v;
#pragma unroll
      for (int off = 1; off < 32; off <<= 1) {
        const float t = __shfl_up_sync(0xffffffffu, sc, off);
        if (lane >= off) sc += t;
      }
      // first child with p > 0 whose prefix sum exceeds u. Without `v > 0` rounding could take an empty slot (p = 0, weight
      // inf): an empty child's scanned sum can round above its left neighbour's (a draw at the end of a partly filled ring),
      // and u - before below can round below 0 (a draw at the start of a child whose first slots are empty)
      const unsigned hit = __ballot_sync(0xffffffffu, v > 0.f && sc > u);
      int f;
      if (hit) f = __ffs(hit) - 1;
      else {                                                  // u within rounding of the node's sum: last child with p > 0
        const unsigned nz = __ballot_sync(0xffffffffu, v > 0.f);
        f = nz ? 31 - __clz(nz) : 0;
      }
      const float before = __shfl_sync(0xffffffffu, sc - v, f), vf = __shfl_sync(0xffffffffu, v, f);
      u = hit ? u - before : vf;
      node = node * PER_FANOUT + f;
    }
    if (lane == 0) {
      const float p = a.leaf[node];
      i64 j = node - oldest;
      if (j < 0) j += cap;
      a.out_idx[k] = j;
      a.out_w[k] = powf(p / pmin, -beta);
      if (a.out_slots) a.out_slots[k] = node;
    }
  }
  if (gt == 0) a.st->sample_oldest = oldest;
}

}  // namespace sacx
