// Row work folded into the GEMM tiles (single-agent latency path).
//
// In the unfused plan the narrow output layers and the elementwise SAC arithmetic behind them are separate
// "row" phases: 32 CTAs busy, 10-16K cycles each, plus a grid barrier. Here they disappear into their neighbours:
//   * PART  -- the GEMM tile that PRODUCES the last hidden activations (or the critics' layer-0 delta) also emits,
//              from its epilogue, the tile's share of the head dot products: part[tn][m][j] = sum over the tile's
//              columns of val[m][col] * Wp(j, col). Summing the tn shares in a fixed order is deterministic.
//   * GEN   -- the dA GEMM tile that CONSUMES delta of the last hidden layer builds that operand itself: a short
//              prologue turns the shares into per-row scalars (Q, target y, dQ routing, head backward), and the
//              activations it would have needed anyway are transformed in shared memory, chunk by chunk, by the
//              thread that copied them: delta[r][k] = coef[r] * W_L[k] * act'(h[r][k]).
//   * OP_DW_HEAD -- gradient + Adam (+Polyak) of the critics' output layer, from the same per-row scalars.
// Per-row side outputs (y, Q, log-pi, loss rows, dhead) are written by the tn == 0 tiles only.
#pragma once
#include "sacx_math.cuh"
#include "sacx_types.cuh"

namespace sacx {

enum GenKind : int { GEN_NONE = 0, GEN_CRITIC = 3, GEN_ACTORQ = 4, GEN_PIBWD = 5 };
constexpr int XSM_FLOATS = 8192;        // extra shared memory for the fused paths
constexpr int XS_WP = 0;                // [nh][32] slice of the partial-product weights (nh <= 32)
constexpr int XS_COEF = 1024;           // [64] per-row coefficient
constexpr int XS_DHEAD = 1088;          // [32][16] head gradient rows (2A <= 16)
constexpr int XS_WL = 1600;             // W_L[K] or Wpi_L[2A][K]  (<= 6592 floats)
constexpr int XS_WL_CAP = XSM_FLOATS - XS_WL;

struct FusedCtx {
  float* base;
  const AgentScalars* scal;
  const Hyper* hp;
  float* xsm;
  const float* w_ext;             // RunArgs::w_ext
};

__device__ __forceinline__ float sum_parts(const float* __restrict__ p, int n_part, i64 stride) {
  float s = 0.f;
  for (int j = 0; j < n_part; ++j) s += __ldcg(p + j * stride);
  return s;
}
// the same sum with the shares spread over the 8 lanes that own a row (one L2 round trip instead of n_part);
// summation order is fixed (lane-strided partial sums, then a butterfly), hence deterministic
__device__ __forceinline__ float sum_parts8(const float* __restrict__ p, int n_part, i64 stride, int j8, bool ok) {
  float s = 0.f;
  if (ok) for (int j = j8; j < n_part; j += 8) s += __ldcg(p + j * stride);
  s += __shfl_xor_sync(0xffffffffu, s, 1);
  s += __shfl_xor_sync(0xffffffffu, s, 2);
  s += __shfl_xor_sync(0xffffffffu, s, 4);
  return s;
}

// GEN_CRITIC slots: o[2..3]=target-critic shares [tn][B]  o[4..5]=target output biases  o[6]=r o[7]=d o[8]=logpi' o[9]=y out
//   o[10..11]=tq out  o[12]=this critic's shares  o[13]=its output bias  o[14]=q out  o[15]=dout out (ld 4)  o[16]=lossrow out
//   o[17]=W_L of this critic   i[2]=number of shares  i[3]=critic index
struct CriticRow { float y, tq1, tq2, q, dout, diff, w; };
// all 8 lanes of the row call this (shuffles inside); every lane returns the full result
__device__ __forceinline__ CriticRow critic_row_scalars(const Op& op, const FusedCtx& c, int m, int j8, bool ok) {
  const Hyper& hp = *c.hp;
  const float* base = c.base;
  const int np = op.i[2];
  const i64 B = hp.B;
  // independent loads first (one round trip), then the reductions
  const float bt1 = __ldcg(base + op.o[4]), bt2 = __ldcg(base + op.o[5]), bq = __ldcg(base + op.o[13]);
  const float alpha = __ldcg(&c.scal->alpha_f32);
  const float rew = ok ? __ldcg(base + op.o[6] + m) : 0.f, done = ok ? __ldcg(base + op.o[7] + m) : 0.f;
  const float lp2 = ok ? __ldcg(base + op.o[8] + m) : 0.f;
  const float s1 = sum_parts8(base + op.o[2] + m, np, B, j8, ok);
  const float s2 = sum_parts8(base + op.o[3] + m, np, B, j8, ok);
  const float sq = sum_parts8(base + op.o[12] + m, np, B, j8, ok);
  CriticRow r;
  r.tq1 = act_fwd(op.act_out, s1 + bt1);
  r.tq2 = act_fwd(op.act_out, s2 + bt2);
  // y = r + gamma (1 - d) (min(Q1t, Q2t) - alpha logpi')      (agent.py:208-210)
  r.y = rew + (__ldcg(&c.scal->gamma) * (1.f - done)) * (fminf(r.tq1, r.tq2) - alpha * lp2);
  const float z = sq + bq;
  r.q = act_fwd(op.act_out, z);
  r.diff = r.q - r.y;
  r.w = (c.w_ext && ok) ? __ldcg(c.w_ext + m) : 1.f;       // importance weight (prioritized replay); 1 multiplies exactly
  r.dout = (2.f * (r.w * r.diff) / (float)hp.B_global) * act_dz2(op.act_out, z, r.q);     // d mse / d q through the output activation
  return r;
}

// prologue of a generating tile (32 rows x 8 lanes = 256 threads): per-row scalars -> xsm, W_L -> xsm; side outputs
// by the tn == 0 tiles
__device__ __forceinline__ void gen_prologue(const Op& op, const FusedCtx& c, int m0, int tn, int BM) {
  const int tid = threadIdx.x;
  float* xs = c.xsm;
  float* base = c.base;
  const Hyper& hp = *c.hp;
  const int K = op.K;
  const int r = tid >> 3, j8 = tid & 7, m = m0 + r;
  const bool ok = m < hp.B;
  if (op.mode == GEN_CRITIC || op.mode == GEN_ACTORQ) {
    for (int k = tid; k < K; k += 256) xs[XS_WL + k] = __ldcg(base + op.o[17] + k);
    float coef = 0.f;
    if (op.mode == GEN_CRITIC) {
      const CriticRow cr = critic_row_scalars(op, c, m, j8, ok);
      coef = ok ? cr.dout : 0.f;
      if (tn == 0 && ok && j8 == 0) {
        if (op.i[3] == 0) { base[op.o[9] + m] = cr.y; base[op.o[10] + m] = cr.tq1; base[op.o[11] + m] = cr.tq2; }
        base[op.o[14] + m] = cr.q;
        base[op.o[15] + (i64)m * 4] = cr.dout;
        base[op.o[16] + m] = cr.w * (cr.diff * cr.diff);
      }
    } else {
      // GEN_ACTORQ: o[2..3]=shares of Q1,Q2(s, a~pi)  o[4..5]=output biases  o[8]=logpi  o[10..11]=q out  o[16]=policy loss rows
      const int np = op.i[2];
      const float b1 = __ldcg(base + op.o[4]), b2 = __ldcg(base + op.o[5]);
      const float alpha = __ldcg(&c.scal->alpha_f32);
      const float lp = ok ? __ldcg(base + op.o[8] + m) : 0.f;
      const float z1 = sum_parts8(base + op.o[2] + m, np, hp.B, j8, ok) + b1;
      const float z2 = sum_parts8(base + op.o[3] + m, np, hp.B, j8, ok) + b2;
      const float q1 = act_fwd(op.act_out, z1), q2 = act_fwd(op.act_out, z2);
      // torch.min backward: gradient to the smaller input, ties split 1/2 - 1/2
      const float w1 = q1 < q2 ? 1.f : (q1 == q2 ? 0.5f : 0.f);
      const bool first = (op.i[3] == 0);
      coef = ok ? (first ? -w1 : -(1.f - w1)) / (float)hp.B_global * (first ? act_dz2(op.act_out, z1, q1) : act_dz2(op.act_out, z2, q2)) : 0.f;
      if (tn == 0 && first && ok && j8 == 0) {
        base[op.o[10] + m] = q1;
        base[op.o[11] + m] = q2;
        base[op.o[16] + m] = alpha * lp - fminf(q1, q2);
      }
    }
    if (j8 == 0) xs[XS_COEF + r] = coef;
  } else if (op.mode == GEN_PIBWD) {
    // o[2..3]=dQ/da shares of the two critics [tn][B][A]  o[4]=tanh z  o[5]=sigma eps  o[6]=clamp mask  o[7]=head pre-activations
    // o[8]=dhead out [B][2A]  o[17]=Wpi_L [2A][K]
    const int A = hp.act, np = op.i[2];
    for (int k = tid * 4; k < 2 * A * K; k += 1024)
      *reinterpret_cast<float4*>(xs + XS_WL + k) = __ldcg(reinterpret_cast<const float4*>(base + op.o[17] + k));
    const float alpha = __ldcg(&c.scal->alpha_f32), ab = alpha / (float)hp.B_global;
    const i64 sj = (i64)hp.B * A;
    // lane j8 < A also owns action dimension j8 of its row (A <= 8)
    const bool own = ok && j8 < A;
    const float tz = own ? __ldcg(base + op.o[4] + (i64)m * A + j8) : 0.f, se = own ? __ldcg(base + op.o[5] + (i64)m * A + j8) : 0.f;
    const float mk = own ? __ldcg(base + op.o[6] + (i64)m * A + j8) : 0.f;
    float zm = 0.f, zl = 0.f;
    if (own && op.act_out != SACX_ACT_IDENTITY) {
      zm = __ldcg(base + op.o[7] + (i64)m * 2 * A + j8);
      zl = __ldcg(base + op.o[7] + (i64)m * 2 * A + A + j8);
    }
    float da_mine = 0.f;
    for (int j = 0; j < A; ++j) {      // every dimension's sum is computed by all 8 lanes together
      const float d = sum_parts8(base + op.o[2] + (i64)m * A + j, np, sj, j8, ok) + sum_parts8(base + op.o[3] + (i64)m * A + j, np, sj, j8, ok);
      if (j == j8) da_mine = d;
    }
    if (j8 < A) {
      // dL/dz = (alpha/B) 2 tanh z + dL/da c (1 - tanh^2 z); dL/dmu = dL/dz; dL/dlogstd_raw = (sigma eps dL/dz - alpha/B) mask
      const float dz = ab * (2.f * tz) + da_mine * (hp.action_scale * (1.f - tz * tz));
      float dmu = ok ? dz : 0.f, dls = ok ? (se * dz - ab) * mk : 0.f;
      if (own && op.act_out != SACX_ACT_IDENTITY) {
        dmu *= act_dz2(op.act_out, zm, act_fwd(op.act_out, zm));
        dls *= act_dz2(op.act_out, zl, act_fwd(op.act_out, zl));
      }
      if (tn == 0 && ok) {
        base[op.o[8] + (i64)m * 2 * A + j8] = dmu;
        base[op.o[8] + (i64)m * 2 * A + A + j8] = dls;
      }
      xs[XS_DHEAD + r * 16 + j8] = dmu;
      xs[XS_DHEAD + r * 16 + A + j8] = dls;
    }
  }
}

// in-place transform of one float4 of the landed A stage: v = saved activations -> delta
__device__ __forceinline__ float4 gen_transform(const Op& op, const FusedCtx& c, float4 v, int row, int gk, bool valid) {
  if (!valid) return make_float4(0.f, 0.f, 0.f, 0.f);
  const float* xs = c.xsm;
  if (op.mode == GEN_PIBWD) {
    const int A2 = 2 * c.hp->act, K = op.K;
    float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int j = 0; j < A2; ++j) {
      const float g = xs[XS_DHEAD + row * 16 + j];
      const float4 w = *reinterpret_cast<const float4*>(xs + XS_WL + j * K + gk);
      s.x = fmaf(g, w.x, s.x); s.y = fmaf(g, w.y, s.y); s.z = fmaf(g, w.z, s.z); s.w = fmaf(g, w.w, s.w);
    }
    return make_float4(s.x * act_dz(op.act, v.x), s.y * act_dz(op.act, v.y), s.z * act_dz(op.act, v.z), s.w * act_dz(op.act, v.w));
  }
  const float co = xs[XS_COEF + row];
  const float4 w = *reinterpret_cast<const float4*>(xs + XS_WL + gk);
  return make_float4(co * w.x * act_dz(op.act, v.x), co * w.y * act_dz(op.act, v.y), co * w.z * act_dz(op.act, v.z),
                     co * w.w * act_dz(op.act, v.w));
}

// PART: i[4]=1, i[5]=nh, i[6]=stride over j, i[7]=stride over n, o[0]=Wp base, o[1]=out [tn][M][nh]
__device__ __forceinline__ void part_stage(const Op& op, const FusedCtx& c, int n0, int BN) {
  const int nh = op.i[5];
  for (int idx = threadIdx.x; idx < nh * BN; idx += 256) {
    const int j = idx / BN, n = n0 + idx % BN;
    c.xsm[XS_WP + idx] = (n < op.N) ? __ldcg(c.base + op.o[0] + (i64)j * op.i[6] + (i64)n * op.i[7]) : 0.f;
  }
}
// val = the four values this thread just stored for (m, n0+c4 .. +3); the 8 lanes of a row reduce with shuffles
__device__ __forceinline__ void part_emit(const Op& op, const FusedCtx& c, float4 val, int m, int c4, int tn, int BN) {
  const int nh = op.i[5];
  const float* wp = c.xsm + XS_WP;
  for (int j = 0; j < nh; ++j) {
    const float4 w = *reinterpret_cast<const float4*>(wp + j * BN + c4);
    float p = val.x * w.x + val.y * w.y + val.z * w.z + val.w * w.w;
    p += __shfl_xor_sync(0xffffffffu, p, 1);
    p += __shfl_xor_sync(0xffffffffu, p, 2);
    p += __shfl_xor_sync(0xffffffffu, p, 4);
    if ((threadIdx.x & 7) == 0 && m < op.M) c.base[op.o[1] + ((i64)tn * op.M + m) * nh + j] = p;
  }
}

// ---------------------------------------------------------------- OP_DW_HEAD
// Gradient and optimiser step of a critic's output layer: dW_L[k] = sum_b dout[b] h[b][k], db_L = sum_b dout[b].
// Same slots as GEN_CRITIC plus o[18]=last hidden activations, i[0]=ld, i[1]=K; parameter block fields p/pm/pv/pt/pg (+bias).
// One tile = 32 columns k; dout [B] (row stride 4) was written by the generating dA tiles of the previous phase.
__device__ __noinline__ void tile_dw_head(const Op& op, const FusedCtx& c, int tile, float* __restrict__ sm) {
  const Hyper& hp = *c.hp;
  float* base = c.base;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int B = hp.B, K = op.i[1], ld = op.i[0];
  float* dout_s = sm;                     // [B] (B <= capacity checked on the host)
  float* red = sm + ((B + 31) & ~31);     // [8][33]
  for (int b = tid; b < B; b += 256) dout_s[b] = __ldcg(base + op.o[15] + (i64)b * 4);     // written by the generating tiles one phase earlier
  __syncthreads();
  const int k = tile * 32 + lane;
  float acc = 0.f, bsum = 0.f;
  const float* h = base + op.o[18];
  for (int b = warp; b < B; b += 8) {
    const float d = dout_s[b];
    if (k < K) acc = fmaf(d, __ldcg(h + (i64)b * ld + k), acc);
    bsum += d;
  }
  red[warp * 33 + lane] = acc;
  if (lane == 0) red[warp * 33 + 32] = bsum;
  __syncthreads();
  if (warp == 0) {
    float g = 0.f, gb = 0.f;
#pragma unroll
    for (int w = 0; w < 8; ++w) { g += red[w * 33 + lane]; gb += red[w * 33 + 32]; }
    const float ss = __ldcg(&c.scal->adam_step_size[op.opt]), bc = __ldcg(&c.scal->adam_bc2_sqrt[op.opt]);
    const float tau = __ldcg(&c.scal->tau), omt = __ldcg(&c.scal->one_minus_tau);
    if (k < K) {
      if (op.flags & DW_STORE_GRAD) base[op.pg + k] = g;
      if (op.flags & DW_ADAM) {
        float p = __ldcg(base + op.p + k), mm = __ldcg(base + op.pm + k), vv = __ldcg(base + op.pv + k);
        adam_update(g, p, mm, vv, ss, bc);
        base[op.p + k] = p; base[op.pm + k] = mm; base[op.pv + k] = vv;
        if (op.flags & DW_POLYAK) base[op.pt + k] = polyak_mix(tau, omt, p, __ldcg(base + op.pt + k));
      }
    }
    if (tile == 0 && lane == 0) {
      if (op.flags & DW_STORE_GRAD) base[op.pbg] = gb;
      if (op.flags & DW_ADAM) {
        float p = __ldcg(base + op.pb), mm = __ldcg(base + op.pbm), vv = __ldcg(base + op.pbv);
        adam_update(gb, p, mm, vv, ss, bc);
        base[op.pb] = p; base[op.pbm] = mm; base[op.pbv] = vv;
        if (op.flags & DW_POLYAK) base[op.pbt] = polyak_mix(tau, omt, p, __ldcg(base + op.pbt));
      }
    }
  }
  __syncthreads();
}

}  // namespace sacx
