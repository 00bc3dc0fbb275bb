// Elementwise math of the SAC update: the seven activations of the reference's _ACTIVATIONS table
// (sac/models.py:104-112) with the derivative forms torch's backward uses, torch's softplus, the per-row formulas of
// the losses and their gradients that every kernel path calls, and the counter-based RNGs of the throughput mode
// (Philox4x32-10 normals, keyed Feistel index bijection).
#pragma once
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

#include "../../include/sacx.h"

namespace sacx {

#define SELU_ALPHA 1.6732632423543772848170429916717f
#define SELU_SCALE 1.0507009873554804934193349852946f

__device__ __noinline__ float act_fwd_general(int act, float z) {
  switch (act) {
    case SACX_ACT_RELU: return fmaxf(z, 0.f);
    case SACX_ACT_TANH: return tanhf(z);
    case SACX_ACT_ELU: return z > 0.f ? z : expm1f(z);
    case SACX_ACT_LEAKY_RELU: return z > 0.f ? z : 0.01f * z;
    case SACX_ACT_GELU: return 0.5f * z * (1.f + erff(z * 0.70710678118654752440f));
    case SACX_ACT_SELU: return z > 0.f ? SELU_SCALE * z : (SELU_SCALE * SELU_ALPHA) * expm1f(z);
    default: return z;
  }
}

// ReLU / identity (every shipped config) stay inline; the transcendental activations are one out-of-line call
__device__ __forceinline__ float act_fwd(int act, float z) {
  if (act == SACX_ACT_RELU) return fmaxf(z, 0.f);
  if (act == SACX_ACT_IDENTITY) return z;
  return act_fwd_general(act, z);
}

// activations whose derivative is evaluated from the pre-activation z (the others use the output h)
__host__ __device__ __forceinline__ bool act_needs_z(int act) {
  return act == SACX_ACT_ELU || act == SACX_ACT_GELU || act == SACX_ACT_SELU;
}

// d act / d z given aux = z (elu, gelu, selu) or aux = h (relu, tanh, leaky_relu, identity)
__device__ __noinline__ float act_dz_general(int act, float aux) {
  switch (act) {
    case SACX_ACT_RELU: return aux > 0.f ? 1.f : 0.f;
    case SACX_ACT_TANH: return 1.f - aux * aux;
    case SACX_ACT_ELU: return aux > 0.f ? 1.f : expf(aux);
    case SACX_ACT_LEAKY_RELU: return aux > 0.f ? 1.f : 0.01f;
    case SACX_ACT_GELU: {
      float cdf = 0.5f * (1.f + erff(aux * 0.70710678118654752440f));
      float pdf = expf(-0.5f * aux * aux) * 0.39894228040143267794f;
      return cdf + aux * pdf;
    }
    case SACX_ACT_SELU: return aux > 0.f ? SELU_SCALE : (SELU_SCALE * SELU_ALPHA) * expf(aux);
    default: return 1.f;
  }
}

__device__ __forceinline__ float act_dz(int act, float aux) {
  if (act == SACX_ACT_RELU) return aux > 0.f ? 1.f : 0.f;
  if (act == SACX_ACT_IDENTITY) return 1.f;
  return act_dz_general(act, aux);
}

// derivative when both z and h are at hand (output layers)
__device__ __forceinline__ float act_dz2(int act, float z, float h) { return act_dz(act, act_needs_z(act) ? z : h); }

// F.softplus(beta=1, threshold=20)
__device__ __forceinline__ float softplus20(float x) { return x > 20.f ? x : log1pf(expf(x)); }

// ---------------------------------------------------------------- per-row SAC formulas
// Each per-row formula of the update, stated once for the tile row ops, the tensor-core tails, the row-parallel kernel and
// act_kernel; loads, stores and the work split stay with the callers. Fixed operation order: equal inputs, equal bits on every path.

// tanh-squashed Gaussian rsample and its log-prob for one action dimension (models.py:79-87). The caller scales tz by
// action_scale and stores se = sd * e; in_clamp is the mask of the log_std clamp's gradient, bad flags a non-finite head.
struct SacSample { float tz, sd, lp; bool in_clamp, bad; };
__device__ __forceinline__ SacSample sac_rsample(float mu, float ls_raw, float e, float lo, float hi) {
  const float sd = expf(fminf(fmaxf(ls_raw, lo), hi));
  const float z = mu + e * sd;                       // Normal.rsample: loc + eps * scale
  const float dzm = z - mu;
  // Normal.log_prob: -(z-mu)^2 / (2 var) - log(std) - log(sqrt(2 pi))
  float lp = -(dzm * dzm) / (2.f * (sd * sd)) - logf(sd) - 0.91893853320467274178f;
  // tanh Jacobian, softplus form: 2 (log 2 - z - softplus(-2 z))   (F7: no -log(action_scale))
  lp -= 2.f * (0.69314718055994530942f - z - softplus20(-2.f * z));
  return {tanhf(z), sd, lp, ls_raw >= lo && ls_raw <= hi, !(isfinite(mu) && isfinite(sd))};
}

// soft Bellman target y = r + gamma (1 - d) (min(Q1t, Q2t) - alpha logpi')      (agent.py:208-210)
__device__ __forceinline__ float sac_target(float r, float d, float gamma, float alpha, float tq1, float tq2, float lp2) {
  return r + (gamma * (1.f - d)) * (fminf(tq1, tq2) - alpha * lp2);
}

// one critic's row of the weighted mse (agent.py:213-236, DESIGN §8): q = act(z), loss w diff^2, and d loss / d z =
// 2 w diff / B through the output activation. w is the importance weight of prioritized replay, 1.f (exact) without it.
struct SacCriticRow { float q, dout, loss; };
__device__ __forceinline__ SacCriticRow sac_critic_row(int act_out, float z, float y, float w, int B_global) {
  const float q = act_fwd(act_out, z), dq = act_dz2(act_out, z, q), diff = q - y;
  return {q, (2.f * (w * diff) / (float)B_global) * dq, w * (diff * diff)};
}

// torch.min backward of the policy loss (agent.py:238-260): gradient to the smaller critic, ties split 1/2 - 1/2, through
// each critic's output activation
struct SacRoute { float c1, c2; };
__device__ __forceinline__ SacRoute sac_actor_route(int act_out, float z1, float q1, float z2, float q2, int B_global) {
  const float w1 = q1 < q2 ? 1.f : (q1 == q2 ? 0.5f : 0.f);
  const float g1 = -w1 / (float)B_global, g2 = -(1.f - w1) / (float)B_global;
  return {g1 * act_dz2(act_out, z1, q1), g2 * act_dz2(act_out, z2, q2)};
}
__device__ __forceinline__ float sac_policy_loss_row(float alpha, float lp, float q1, float q2) { return alpha * lp - fminf(q1, q2); }

// closed-form head backward (SURVEY a8), da = dQ/da of both critics, ab = alpha / B: dL/dz = ab 2 tanh z + da c (1 - tanh^2 z),
// dL/dmu = dL/dz, dL/dlogstd_raw = (sigma eps dL/dz - ab) mask; then through the head's activation (zm, zl: pre-activations)
struct SacHeadGrad { float dmu, dls; };
__device__ __forceinline__ SacHeadGrad sac_head_bwd(int act_out, float tz, float se, float mk, float da, float ab,
                                                    float action_scale, float zm, float zl) {
  const float dz = ab * (2.f * tz) + da * (action_scale * (1.f - tz * tz));
  float dmu = dz, dls = (se * dz - ab) * mk;
  if (act_out != SACX_ACT_IDENTITY) {
    dmu *= act_dz2(act_out, zm, act_fwd(act_out, zm));
    dls *= act_dz2(act_out, zl, act_fwd(act_out, zl));
  }
  return {dmu, dls};
}

// delta of a hidden layer: s act'(h), or c w act'(h) behind an output layer of width 1; h is the saved activation. act by
// reference, so a caller's op.act is read per element: by value, nvcc merges a float4's four act_dz tests into one branch
// and copies the products into both sides (+28 FMUL per tile kernel)
__device__ __forceinline__ float sac_dact(float s, float h, const int& act) { return s * act_dz(act, h); }
__device__ __forceinline__ float4 sac_dact(float4 s, float4 h, const int& act) {
  return make_float4(s.x * act_dz(act, h.x), s.y * act_dz(act, h.y), s.z * act_dz(act, h.z), s.w * act_dz(act, h.w));
}
__device__ __forceinline__ float sac_delta(float c, float w, float h, const int& act) { return c * w * act_dz(act, h); }
__device__ __forceinline__ float4 sac_delta(float c, float4 w, float4 h, const int& act) {
  return make_float4(c * w.x * act_dz(act, h.x), c * w.y * act_dz(act, h.y), c * w.z * act_dz(act, h.z), c * w.w * act_dz(act, h.w));
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// ---------------------------------------------------------------- optimiser arithmetic (a10, a11)
__device__ __forceinline__ void adam_update(float g, float& p, float& m, float& v, float step_size, float bc2_sqrt) {
  // torch _single_tensor_adam: m.lerp_(g, 1-b1); v.mul_(b2).addcmul_(g, g, 1-b2);
  // denom = sqrt(v)/sqrt(bc2) + eps; p.addcdiv_(m, denom, -lr/bc1)
  m = m + 0.1f * (g - m);
  v = v * 0.999f + 0.001f * g * g;
  const float denom = sqrtf(v) / bc2_sqrt + 1e-8f;
  p = p - step_size * (m / denom);
}

__device__ __forceinline__ float polyak_mix(float tau, float omt, float p, float t) {
  // tau * p + (1 - tau) * t with separately rounded products (agent.py:288-291), no FMA contraction
  return __fadd_rn(__fmul_rn(tau, p), __fmul_rn(omt, t));
}

// ---------------------------------------------------------------- Philox4x32-10
__device__ __forceinline__ void philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0,
                                              uint32_t k1, uint32_t out[4]) {
  const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    uint32_t hi0 = __umulhi(M0, c0), lo0 = M0 * c0;
    uint32_t hi1 = __umulhi(M1, c2), lo1 = M1 * c2;
    uint32_t n0 = hi1 ^ c1 ^ k0, n1 = lo1, n2 = hi0 ^ c3 ^ k1, n3 = lo0;
    c0 = n0; c1 = n1; c2 = n2; c3 = n3;
    k0 += W0; k1 += W1;
  }
  out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

// N(0,1) for element (update, which, global row, j): Box-Muller on two Philox words
__device__ __noinline__ float philox_normal(unsigned long long seed, unsigned long long update, int which,
                                               uint32_t row, uint32_t j, uint32_t agent) {
  uint32_t o[4];
  philox4x32_10((uint32_t)update, (uint32_t)(update >> 32), row, ((uint32_t)which << 24) | j,
                (uint32_t)seed ^ (agent * 0x9E3779B9u), (uint32_t)(seed >> 32) ^ 0x5AC5AC5Au, o);
  float u1 = ((float)o[0] + 1.0f) * 2.3283064365386963e-10f;   // (0, 1]
  float u2 = (float)o[1] * 2.3283064365386963e-10f;
  u1 = fminf(fmaxf(u1, 1e-30f), 1.0f);
  return sqrtf(-2.0f * logf(u1)) * cospif(2.0f * u2);
}

// ---------------------------------------------------------------- keyed bijection on [0, n)
// Balanced Feistel network over 2*half bits with cycle walking: position i in [0, n) -> a distinct
// element of [0, n).  Evaluating it at i = 0..B-1 yields B distinct logical indices (sampling without
// replacement, as random.sample does) with no inter-thread communication.
__device__ __forceinline__ uint32_t mix32(uint32_t x) {
  x ^= x >> 16; x *= 0x85EBCA6Bu; x ^= x >> 13; x *= 0xC2B2AE35u; x ^= x >> 16;
  return x;
}

// the bijection's round keys: one Philox block per (update counter, agent, seed) -- the same for every row of an update
__device__ __forceinline__ void feistel_key(unsigned long long seed, unsigned long long counter, uint32_t agent, uint32_t (&key)[4]) {
  philox4x32_10((uint32_t)counter, (uint32_t)(counter >> 32), 0x1D8E4E27u, agent, (uint32_t)seed, (uint32_t)(seed >> 32), key);
}
__device__ __forceinline__ unsigned long long feistel_apply(unsigned long long i, unsigned long long n, const uint32_t (&key)[4]) {
  if (n <= 1) return 0;
  int bits = 64 - __clzll((long long)(n - 1));
  int half = (bits + 1) >> 1;
  if (half < 1) half = 1;
  const uint32_t mask = (half >= 32) ? 0xFFFFFFFFu : ((1u << half) - 1u);
  unsigned long long x = i;
  do {
    uint32_t L = (uint32_t)(x >> half) & mask, R = (uint32_t)x & mask;
#pragma unroll
    for (int r = 0; r < 6; ++r) {
      uint32_t f = mix32(R ^ key[r & 3] ^ (0x9E3779B9u * (uint32_t)(r + 1))) & mask;
      uint32_t nl = R;
      R = L ^ f;
      L = nl;
    }
    x = ((unsigned long long)L << half) | R;
  } while (x >= n);
  return x;
}
__device__ __noinline__ unsigned long long feistel_index(unsigned long long i, unsigned long long n,
                                                            unsigned long long seed, unsigned long long counter,
                                                            uint32_t agent) {
  uint32_t key[4];
  feistel_key(seed, counter, agent, key);
  return feistel_apply(i, n, key);
}

}  // namespace sacx
