// Row-wise operations of the SAC update: one warp owns one batch row, one CTA tile = 8 rows. These are the
// narrow output layers (policy head N=2A, critic head N=1) and everything the reference computes right
// after them: the tanh-squashed Gaussian rsample/log_prob (sac/models.py:79-87), the soft Bellman target
// (sac/agent.py:207-210), the critic/actor loss gradients and the closed-form head backward (SURVEY
// section 8 a5/a8), the temperature step (agent.py:263-280).
//
// Latency structure (what the profile asked for): the small weight matrices a tile needs are staged once
// per CTA into shared memory with cp.async while every warp's own row (last hidden activations, saved
// activations) travels into registers, so a tile pays ONE L2 round trip; all dot products then read
// shared memory / registers and reduce with warp shuffles.
#pragma once
#include "sacx_gemm.cuh"
#include "sacx_math.cuh"
#include "sacx_types.cuh"

namespace sacx {

constexpr int ROWS_PER_TILE = 8;     // 256 threads = 8 warps = 8 rows
constexpr int ROW_MAXK = 256;        // widest last-hidden layer handled by the register-resident path
constexpr int ROW_KREG = ROW_MAXK / 128;

struct RowCtx {
  float* base;
  AgentScalars* scal;
  const RunArgs* args;
  int agent, step;
  float* wsm;          // per-warp shared scratch, 4*SACX_MAX_ACT floats
  float* tsm;          // CTA-wide shared staging area (aliases the GEMM ring), tsm_floats floats
  int tsm_floats;
  unsigned long long* t;   // optional timestamps (profiling aid)
  int pf_rows = 0;         // light kernel: row distance to the tile this CTA runs two iterations from now (L2 prefetch), 0 = off
  int fresh = 1;           // 0: this CTA's previous tile belonged to the same op and agent -> the staged weights in tsm are still valid
  // OP_GATHER, cached per thread across the rows it gathers for one (agent, update): the sampler's round keys, the ring's push
  // count and the slot of the oldest survivor -- one Philox block, one header read and one 64-bit modulo per update, not per row
  // (kept in the warp's shared scratch, not in registers: [0] agent [1] step [2..5] keys [6..7] pushes [8..9] oldest slot)
  uint32_t* gcache = nullptr;
};
constexpr int GCACHE_WORDS = 12;
#ifdef SACX_DEBUG_HOOKS
#define SACX_RSTAMP(i) do { if (c.t && threadIdx.x == 0) c.t[i] = clock64(); } while (0)
#else
#define SACX_RSTAMP(i) do { } while (0)
#endif

// ---- staging helpers -------------------------------------------------------------------------------
// copy n floats global -> shared by the whole CTA (cp.async when 16B-aligned, scalar otherwise)
__device__ __noinline__ void stage_vec(float* dst, const float* src, int n) {
  if (((n & 3) == 0) && ((((uintptr_t)src) & 15) == 0) && ((((uintptr_t)dst) & 15) == 0)) {
    for (int i = threadIdx.x * 4; i < n; i += 1024) cp_async16(dst + i, src + i, 16);
  } else {
    for (int i = threadIdx.x; i < n; i += 256) dst[i] = __ldcg(src + i);
  }
}
__device__ __forceinline__ void stage_finish() {
  cp_async_commit();
  cp_async_wait<0>();
  __syncthreads();
}

// a row of K floats (K <= ROW_MAXK, row 16B-aligned, K % 4 == 0) in registers: lane owns float4 chunks lane + 32*i
struct RowReg {
  float4 v[ROW_KREG];
};
__device__ __forceinline__ bool row_fast(int K, const float* p) { return K <= ROW_MAXK && (K & 3) == 0 && ((((uintptr_t)p) & 15) == 0); }
__device__ __forceinline__ void row_load(RowReg& r, const float* __restrict__ p, int K, int lane) {
#pragma unroll
  for (int i = 0; i < ROW_KREG; ++i) {
    const int k = (lane + 32 * i) * 4;
    r.v[i] = (k < K) ? __ldcg(reinterpret_cast<const float4*>(p + k)) : make_float4(0.f, 0.f, 0.f, 0.f);
  }
}
// pull a future row (K floats) into L2: the large-batch row kernels are bound by HBM latency x bytes in flight
__device__ __forceinline__ void row_prefetch(const float* p, int K, int lane) {
  if (lane * 32 < K) asm volatile("prefetch.global.L2 [%0];" ::"l"(p + lane * 32));
}
// dot(row in registers, w in shared memory)
__device__ __forceinline__ float row_dot_partial(const RowReg& r, const float* __restrict__ w, int K, int lane) {
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < ROW_KREG; ++i) {
    const int k = (lane + 32 * i) * 4;
    if (k < K) {
      const float4 b = *reinterpret_cast<const float4*>(w + k);
      s = fmaf(r.v[i].x, b.x, s); s = fmaf(r.v[i].y, b.y, s); s = fmaf(r.v[i].z, b.z, s); s = fmaf(r.v[i].w, b.w, s);
    }
  }
  return s;
}
// generic fallback: both operands wherever they live
__device__ __noinline__ float warp_dot_any(const float* __restrict__ h, const float* __restrict__ w, int K, int lane) {
  float s = 0.f;
  for (int k = lane; k < K; k += 32) s = fmaf(__ldcg(h + k), w[k], s);
  return s;
}

// ---------------------------------------------------------------- OP_GATHER
// o[0]=X_sa o[1]=X_s2 o[2]=X_pi o[3]=r o[4]=d o[5]=idx(i64)  i[0]=ldx
__device__ __forceinline__ void op_gather(const Op& op, RowCtx& c, int row, int lane) {
  const RunArgs& a = *c.args;
  const Hyper& hp = a.hp;
  if (row >= hp.B) return;
  const float* ring = a.ring + (i64)c.agent * a.ring_stride;
  const i64 cap = a.ring_capacity;
  uint32_t* gc = c.gcache;
  if ((int)gc[0] != c.agent || (int)gc[1] != c.step) {       // first row of this (agent, update) on this warp
    __syncwarp();
    if (lane == 0) {
      const i64 pushes = reinterpret_cast<const RingMeta*>(ring)->pushes;
      const i64 oldest_slot = pushes > cap ? (pushes - cap) % cap : 0;
      uint32_t key[4] = {0u, 0u, 0u, 0u};
      if (!a.idx_ext)
        feistel_key(__ldcg(&c.scal->rng_seed), (unsigned long long)__ldcg(&c.scal->updates), __ldcg(&c.scal->rng_agent), key);
      gc[2] = key[0]; gc[3] = key[1]; gc[4] = key[2]; gc[5] = key[3];
      gc[6] = (uint32_t)pushes; gc[7] = (uint32_t)((unsigned long long)pushes >> 32);
      gc[8] = (uint32_t)oldest_slot; gc[9] = (uint32_t)((unsigned long long)oldest_slot >> 32);
      gc[0] = (uint32_t)c.agent; gc[1] = (uint32_t)c.step;
    }
    __syncwarp();
  }
  const i64 g_pushes = (i64)(((unsigned long long)gc[7] << 32) | gc[6]), g_oldest_slot = (i64)(((unsigned long long)gc[9] << 32) | gc[8]);
  const i64 n = g_pushes < cap ? g_pushes : cap;
  i64 j;
  if (a.idx_ext) {
    j = a.idx_ext[((i64)c.step * a.n_agents + c.agent) * hp.B + row];
  } else {
    // throughput mode: position (global row) of a keyed bijection on [0, n) -> distinct indices
    const uint32_t key[4] = {gc[2], gc[3], gc[4], gc[5]};
    j = (i64)feistel_apply((unsigned long long)(hp.row0_global + row), (unsigned long long)n, key);
  }
  i64 slot = g_oldest_slot + j;                                // both < capacity: a conditional subtraction replaces the modulo
  if (slot >= cap) slot -= cap;
  float* base = c.base;
  const int O = hp.obs, A = hp.act, ldx = op.i[0];
  if (lane == 0) reinterpret_cast<i64*>(base + op.o[5])[row] = j;
  const float* rec = ring + slot * a.ring_rs;            // packed record [s | s2 | a | r | d]
  const float* rs = rec + a.ring_s;
  const float* rs2 = rec + a.ring_s2;
  float* xsa = base + op.o[0] + (i64)row * ldx;
  float* xs2 = base + op.o[1] + (i64)row * ldx;
  float* xpi = base + op.o[2] + (i64)row * ldx;
  for (int k = lane; k < O; k += 32) {
    const float v = __ldcs(rs + k);
    xsa[k] = v;
    xpi[k] = v;
    xs2[k] = __ldcs(rs2 + k);
  }
  const float* ra = rec + a.ring_a;
  for (int k = lane; k < A; k += 32) xsa[O + k] = __ldcs(ra + k);
  if (lane == 0) {
    base[op.o[3] + row] = __ldcs(rec + a.ring_r);
    base[op.o[4] + row] = __ldcs(rec + a.ring_d);
  }
}

// ---------------------------------------------------------------- OP_PI_HEAD
// o[0]=h(last hidden) o[1]=W_L o[2]=b_L o[3]=X(dest, action at col obs+j) o[4]=lp o[5]=eps buf
// o[6]=tz o[7]=se o[8]=mask o[9]=headz (each -1 when not saved)   i[0]=ldh i[1]=K i[2]=ldx   mode: 1 target / 2 actor
template <int V>
__device__ __noinline__ void tile_pi_head(const Op& op, const RowCtx& c, int tile) {
  SACX_RSTAMP(0);
  const RunArgs& a = *c.args;
  const Hyper& hp = a.hp;
  float* base = c.base;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int row = tile * ROWS_PER_TILE + warp;
  const int A = hp.act, K = op.i[1];
  const bool in = row < hp.B;
  const float* h = base + op.o[0] + (i64)row * op.i[0];
  const float* Wg = base + op.o[1];
  const bool staged = (2 * A * K + 2 * A) <= c.tsm_floats;
  const bool fast = staged && row_fast(K, h) && row_fast(K, Wg);
  float* Ws = c.tsm;
  float* bs = c.tsm + 2 * A * K;
  RowReg hr;
  const float* eps_ext = (op.mode == 1) ? a.eps1_ext : a.eps2_ext;
  float e_pre = 0.f;
  if (in && lane < A) {
    if (eps_ext) e_pre = eps_ext[(((i64)c.step * a.n_agents + c.agent) * hp.B + row) * A + lane];
    else e_pre = philox_normal(__ldcg(&c.scal->rng_seed), (unsigned long long)__ldcg(&c.scal->updates), op.mode, (uint32_t)(hp.row0_global + row),
                               (uint32_t)lane, __ldcg(&c.scal->rng_agent));
  }
  if (staged) {
    if (c.fresh) {
      stage_vec(Ws, Wg, 2 * A * K);
      for (int i = threadIdx.x; i < 2 * A; i += 256) bs[i] = __ldcg(base + op.o[2] + i);
    }
    if (fast && in) row_load(hr, h, K, lane);
    if (V == 1 && c.pf_rows && row + c.pf_rows < hp.B) row_prefetch(h + (i64)c.pf_rows * op.i[0], K, lane);
    if (c.fresh) stage_finish();
  }
  SACX_RSTAMP(1); SACX_RSTAMP(2); SACX_RSTAMP(3);
  if (!in) { SACX_RSTAMP(4); return; }
  const float* W = staged ? Ws : Wg;
  float* hs = c.wsm;                      // head post-activation [2A], then pre-activation [2A]
  for (int j = 0; j < 2 * A; ++j) {
    const float part = fast ? row_dot_partial(hr, W + (i64)j * K, K, lane) : warp_dot_any(h, W + (i64)j * K, K, lane);
    const float z = warp_sum(part) + (staged ? bs[j] : __ldcg(base + op.o[2] + j));
    if (lane == 0) {
      hs[j] = act_fwd(op.act_out, z);
      hs[2 * SACX_MAX_ACT + j] = z;
    }
  }
  __syncwarp();
  float lp_part = 0.f;
  bool bad = false;
  for (int j = lane; j < A; j += 32) {
    const float e = e_pre;
    base[op.o[5] + (i64)row * A + j] = e;
    const SacSample s = sac_rsample(hs[j], hs[A + j], e, hp.log_std_min, hp.log_std_max);
    base[op.o[3] + (i64)row * op.i[2] + hp.obs + j] = s.tz * hp.action_scale;
    lp_part += s.lp;
    bad |= s.bad;
    if (op.o[6] >= 0) {
      base[op.o[6] + (i64)row * A + j] = s.tz;
      base[op.o[7] + (i64)row * A + j] = s.sd * e;
      base[op.o[8] + (i64)row * A + j] = s.in_clamp ? 1.f : 0.f;
    }
  }
  if (op.o[9] >= 0)
    for (int j = lane; j < 2 * A; j += 32) base[op.o[9] + (i64)row * 2 * A + j] = hs[2 * SACX_MAX_ACT + j];
  const float lp = warp_sum(lp_part);
  if (lane == 0) base[op.o[4] + row] = lp;
  if (bad) atomicOr(&c.scal->nonfinite, 1);
  __syncwarp();
  SACX_RSTAMP(4);
}

// ---------------------------------------------------------------- OP_PI_TAIL (large batch, tensor-core path)
// The policy's output layer is a skinny GEMM (N = 2A) that the tensor-core kernel runs like any other layer; what is left of
// OP_PI_HEAD is per-row scalar work, so ONE THREAD owns a row (256 rows per tile) instead of one warp: ~30x fewer warp
// instructions per row than the shuffle-reduced head. Same sac_rsample as tile_pi_head.
// o[0]=z (head pre-activations [B][i[3]]) o[3]=X(dest) o[4]=lp o[5]=eps buf o[6]=tz o[7]=se o[8]=mask o[9]=compact z copy (-1: not saved)
// i[2]=ldx i[3]=row stride of z   mode 1/2
constexpr int TAIL_ROWS = 256;
__device__ __forceinline__ void tile_pi_tail(const Op& op, const RowCtx& c, int tile) {
  const RunArgs& a = *c.args;
  const Hyper& hp = a.hp;
  float* base = c.base;
  const int row = tile * TAIL_ROWS + threadIdx.x, A = hp.act;
  if (row >= hp.B) return;
  const float* z = base + op.o[0] + (i64)row * op.i[3];
  const float* eps_ext = (op.mode == 1) ? a.eps1_ext : a.eps2_ext;
  const unsigned long long upd = eps_ext ? 0ull : (unsigned long long)__ldcg(&c.scal->updates);
  const unsigned long long rng_seed = eps_ext ? 0ull : __ldcg(&c.scal->rng_seed);
  const uint32_t rng_agent = eps_ext ? 0u : __ldcg(&c.scal->rng_agent);
  float lp = 0.f;
  bool bad = false;
  for (int j = 0; j < A; ++j) {
    const float zm = __ldcg(z + j), zl = __ldcg(z + A + j);
    if (op.o[9] >= 0) { base[op.o[9] + (i64)row * 2 * A + j] = zm; base[op.o[9] + (i64)row * 2 * A + A + j] = zl; }
    const float mu = act_fwd(op.act_out, zm), ls_raw = act_fwd(op.act_out, zl);
    const float e = eps_ext ? eps_ext[(((i64)c.step * a.n_agents + c.agent) * hp.B + row) * A + j]
                            : philox_normal(rng_seed, upd, op.mode, (uint32_t)(hp.row0_global + row), (uint32_t)j, rng_agent);
    base[op.o[5] + (i64)row * A + j] = e;
    const SacSample s = sac_rsample(mu, ls_raw, e, hp.log_std_min, hp.log_std_max);
    base[op.o[3] + (i64)row * op.i[2] + hp.obs + j] = s.tz * hp.action_scale;
    lp += s.lp;
    bad |= s.bad;
    if (op.o[6] >= 0) {
      base[op.o[6] + (i64)row * A + j] = s.tz;
      base[op.o[7] + (i64)row * A + j] = s.sd * e;
      base[op.o[8] + (i64)row * A + j] = s.in_clamp ? 1.f : 0.f;
    }
  }
  base[op.o[4] + row] = lp;
  if (bad) atomicOr(&c.scal->nonfinite, 1);
}

// ---------------------------------------------------------------- OP_Q_TAIL / OP_DELTA (large batch, tensor-core path)
// The critics' output layer (N = 1) rides on the last hidden layer's GEMM: its epilogue thread owns a whole row and projects
// it onto W_L (sacx_tc.cuh: TcOp.proj_*), leaving z = h . W_L + b in the q buffers. What remains of OP_Q_ROW / OP_ACTOR_Q is
// scalar work per row (OP_Q_TAIL, one thread per row) and one element-wise pass that needs h again (OP_DELTA).
// mode bits: 1 target y (agent.py:195-211), 2 critic loss gradient (agent.py:213-236), 4 actor routing (agent.py:238-260).
// o[0..1]=tq (z in, value out) o[2..3]=q (z in, value out) o[4..5]=qa (z in, value out) o[6]=r o[7]=d o[8]=lp2 o[9]=y
// o[10..11]=dout/coef (row stride 4) o[12..13]=lossrow o[14]=lp o[15]=plossrow
__device__ __forceinline__ void tile_q_tail(const Op& op, const RowCtx& c, int tile) {
  const Hyper& hp = c.args->hp;
  float* base = c.base;
  const int row = tile * TAIL_ROWS + threadIdx.x;
  if (row >= hp.B) return;
  const float alpha = __ldcg(&c.scal->alpha_f32);
  float y = 0.f;
  if (op.mode & 1) {
    const float t0 = act_fwd(op.act_out, __ldcg(base + op.o[0] + row)), t1 = act_fwd(op.act_out, __ldcg(base + op.o[1] + row));
    const float r = __ldcg(base + op.o[6] + row), d = __ldcg(base + op.o[7] + row), lp2 = __ldcg(base + op.o[8] + row);
    y = sac_target(r, d, __ldcg(&c.scal->gamma), alpha, t0, t1, lp2);
    base[op.o[0] + row] = t0; base[op.o[1] + row] = t1; base[op.o[9] + row] = y;
  }
  if (op.mode & 2) {
    if (!(op.mode & 1)) y = c.args->y_ext ? c.args->y_ext[row] : __ldcg(base + op.o[9] + row);
    const float w = c.args->w_ext ? __ldcg(c.args->w_ext + row) : 1.f;     // importance weight; 1 multiplies exactly
#pragma unroll
    for (int cc = 0; cc < 2; ++cc) {
      const SacCriticRow cr = sac_critic_row(op.act_out, __ldcg(base + op.o[2 + cc] + row), y, w, hp.B_global);
      base[op.o[2 + cc] + row] = cr.q;
      base[op.o[10 + cc] + (i64)row * 4] = cr.dout;
      base[op.o[12 + cc] + row] = cr.loss;
    }
  }
  if (op.mode & 4) {
    const float z0 = __ldcg(base + op.o[4] + row), z1 = __ldcg(base + op.o[5] + row);
    const float q0 = act_fwd(op.act_out, z0), q1 = act_fwd(op.act_out, z1);
    const SacRoute g = sac_actor_route(op.act_out, z0, q0, z1, q1, hp.B_global);
    base[op.o[4] + row] = q0; base[op.o[5] + row] = q1;
    base[op.o[10] + (i64)row * 4] = g.c1;
    base[op.o[11] + (i64)row * 4] = g.c2;
    base[op.o[15] + row] = sac_policy_loss_row(alpha, __ldcg(base + op.o[14] + row), q0, q1);
  }
}

// o[0..1]=coef (row stride 4) o[2..3]=W_L o[4..5]=aux (saved activation, ld i[0]) o[6..7]=delta out (ld i[0])  i[1]=H  i[2]=tiles per critic
// tile = 16 rows of one critic; thread = one float4 of a row, 256 / (H / 4) rows per pass
constexpr int DELTA_ROWS = 16;
__device__ __forceinline__ void tile_delta(const Op& op, const RowCtx& c, int tile) {
  const Hyper& hp = c.args->hp;
  float* base = c.base;
  const int cc = tile / op.i[2], rb = (tile % op.i[2]) * DELTA_ROWS;
  const int H = op.i[1], ld = op.i[0], cpr = H >> 2;
  if ((int)threadIdx.x >= (256 / cpr) * cpr) return;
  const int k = (threadIdx.x % cpr) << 2, r0 = threadIdx.x / cpr, rstep = 256 / cpr;
  const float4 w = __ldg(reinterpret_cast<const float4*>(base + op.o[2 + cc] + k));
  // a thread's rows (r0, r0 + rstep, ...: at most DELTA_ROWS / 4 = 4 at width 256, more for narrow layers) are loaded TOGETHER
  // before the first is used: the pass is a pure stream, and one dependent DRAM round trip per row left it latency-bound
  // (413 us for the two critics of a 1024-agent population, 2.6 TB/s)
  constexpr int U = 4;
  for (int rbase = r0; rbase < DELTA_ROWS; rbase += U * rstep) {
    float co[U];
    float4 h[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int r = rbase + u * rstep, row = rb + r;
      const bool ok = r < DELTA_ROWS && row < hp.B;
      co[u] = ok ? __ldcg(base + op.o[cc] + (i64)row * 4) : 0.f;
      h[u] = ok ? __ldcs(reinterpret_cast<const float4*>(base + op.o[4 + cc] + (i64)row * ld + k)) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const int r = rbase + u * rstep, row = rb + r;
      if (r < DELTA_ROWS && row < hp.B)
        *reinterpret_cast<float4*>(base + op.o[6 + cc] + (i64)row * ld + k) = sac_delta(co[u], w, h[u], op.act);
    }
  }
}

// ---------------------------------------------------------------- OP_Q_ROW: target y (mode & 1) and / or critic delta (mode & 2)
// target: o[0..1]=hqt(last hidden) o[2..3]=Wt_L o[4..5]=bt_L o[6]=r o[7]=d o[8]=lp2 o[9]=y o[10..11]=tq
// critic: o[12..13]=hq(last hidden) o[14..15]=aux(z or h) o[16..17]=W_L o[18..19]=b_L o[20..21]=q out o[22..23]=dout
//         o[24..25]=delta(last hidden) o[26..27]=lossrow          i[0]=ldh i[1]=K      (y read from o[9] or y_ext)
template <int V>
__device__ __noinline__ void tile_q_row(const Op& op, const RowCtx& c, int tile) {
  SACX_RSTAMP(0);
  const Hyper& hp = c.args->hp;
  float* base = c.base;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int row = tile * ROWS_PER_TILE + warp;
  const bool in = row < hp.B;
  const int K = op.i[1], ld = op.i[0];
  const bool do_t = op.mode & 1, do_c = op.mode & 2;
  const bool staged = 4 * K <= c.tsm_floats;
  float* Ws = c.tsm;                          // [4][K]: target W x2, online W x2
  const float* hp_t[2] = {base + (do_t ? op.o[0] : 0) + (i64)row * ld, base + (do_t ? op.o[1] : 0) + (i64)row * ld};
  const float* hp_c[2] = {base + (do_c ? op.o[12] : 0) + (i64)row * ld, base + (do_c ? op.o[13] : 0) + (i64)row * ld};
  const float* ax_c[2] = {base + (do_c ? op.o[14] : 0) + (i64)row * ld, base + (do_c ? op.o[15] : 0) + (i64)row * ld};
  const bool fast = staged && row_fast(K, base + (do_t ? op.o[0] : op.o[12]) + (i64)row * ld) && ((ld & 3) == 0);
  const bool aux_is_h = do_c && (op.o[14] == op.o[12]);
  RowReg ht[2], hc[2], ac[2];
  // scalars of this row travel together with the staged weights (no dependent L2 round trip after the barrier)
  float bt[2] = {0.f, 0.f}, bc_[2] = {0.f, 0.f}, alpha = 0.f, r_ = 0.f, d_ = 0.f, lp2_ = 0.f, y_in = 0.f, w_in = 1.f;
  if (in) {
    if (do_t) {
      bt[0] = __ldcg(base + op.o[4]); bt[1] = __ldcg(base + op.o[5]);
      alpha = __ldcg(&c.scal->alpha_f32);
      r_ = __ldcg(base + op.o[6] + row); d_ = __ldcg(base + op.o[7] + row); lp2_ = __ldcg(base + op.o[8] + row);
    }
    if (do_c) {
      bc_[0] = __ldcg(base + op.o[18]); bc_[1] = __ldcg(base + op.o[19]);
      if (c.args->y_ext) y_in = c.args->y_ext[row];
      else if (!do_t) y_in = __ldcg(base + op.o[9] + row);
      if (c.args->w_ext) w_in = __ldcg(c.args->w_ext + row);
    }
  }
  if (staged) {
    if (c.fresh) {
      if (do_t) { stage_vec(Ws, base + op.o[2], K); stage_vec(Ws + K, base + op.o[3], K); }
      if (do_c) { stage_vec(Ws + 2 * K, base + op.o[16], K); stage_vec(Ws + 3 * K, base + op.o[17], K); }
    }
    if (fast && in) {
      if (do_t) { row_load(ht[0], hp_t[0], K, lane); row_load(ht[1], hp_t[1], K, lane); }
      if (V == 1 && c.pf_rows && row + c.pf_rows < hp.B) {
        const i64 pf = (i64)c.pf_rows * ld;
        if (do_t) { row_prefetch(hp_t[0] + pf, K, lane); row_prefetch(hp_t[1] + pf, K, lane); }
        if (do_c) {
          row_prefetch(hp_c[0] + pf, K, lane); row_prefetch(hp_c[1] + pf, K, lane);
          if (!aux_is_h) { row_prefetch(ax_c[0] + pf, K, lane); row_prefetch(ax_c[1] + pf, K, lane); }
        }
      }
      if (do_c) {
        row_load(hc[0], hp_c[0], K, lane); row_load(hc[1], hp_c[1], K, lane);
        if (!aux_is_h) { row_load(ac[0], ax_c[0], K, lane); row_load(ac[1], ax_c[1], K, lane); }
        else { ac[0] = hc[0]; ac[1] = hc[1]; }
      }
    }
    if (c.fresh) stage_finish();
  }
  SACX_RSTAMP(1); SACX_RSTAMP(2); SACX_RSTAMP(3);
  if (!in) { SACX_RSTAMP(4); return; }
  float y = 0.f;
  if (do_t) {
    float tq[2];
#pragma unroll
    for (int n = 0; n < 2; ++n) {
      const float* W = staged ? Ws + n * K : base + op.o[2 + n];
      const float part = fast ? row_dot_partial(ht[n], W, K, lane) : warp_dot_any(hp_t[n], W, K, lane);
      tq[n] = act_fwd(op.act_out, warp_sum(part) + bt[n]);
    }
    y = sac_target(r_, d_, __ldcg(&c.scal->gamma), alpha, tq[0], tq[1], lp2_);
    if (lane == 0) {
      base[op.o[9] + row] = y;
      base[op.o[10] + row] = tq[0];
      base[op.o[11] + row] = tq[1];
    }
  }
  if (do_c) {
    if (c.args->y_ext || !do_t) y = y_in;
#pragma unroll
    for (int n = 0; n < 2; ++n) {
      const float* W = staged ? Ws + (2 + n) * K : base + op.o[16 + n];
      const float part = fast ? row_dot_partial(hc[n], W, K, lane) : warp_dot_any(hp_c[n], W, K, lane);
      const SacCriticRow cr = sac_critic_row(op.act_out, warp_sum(part) + bc_[n], y, w_in, hp.B_global);
      const float dout = cr.dout;
      if (lane == 0) {
        base[op.o[20 + n] + row] = cr.q;
        base[op.o[22 + n] + (i64)row * 4] = dout;
        base[op.o[26 + n] + row] = cr.loss;
      }
      float* dl = base + op.o[24 + n] + (i64)row * ld;
      if (fast) {
        const RowReg& ar = ac[n];
#pragma unroll
        for (int i = 0; i < ROW_KREG; ++i) {
          const int k = (lane + 32 * i) * 4;
          if (k < K) *reinterpret_cast<float4*>(dl + k) = sac_delta(dout, *reinterpret_cast<const float4*>(W + k), ar.v[i], op.act);
        }
      } else {
        for (int k = lane; k < K; k += 32) dl[k] = sac_delta(dout, W[k], __ldcg(ax_c[n] + k), op.act);
      }
    }
  }
  SACX_RSTAMP(4);
}

// ---------------------------------------------------------------- OP_ACTOR_Q
// o[0..1]=hq(last hidden) o[2..3]=aux o[4..5]=W_L o[6..7]=b_L o[8]=lp o[9..10]=q out o[13..14]=delta o[15]=plossrow
template <int V>
__device__ __noinline__ void tile_actor_q(const Op& op, const RowCtx& c, int tile) {
  SACX_RSTAMP(0);
  const Hyper& hp = c.args->hp;
  float* base = c.base;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int row = tile * ROWS_PER_TILE + warp;
  const bool in = row < hp.B;
  const int K = op.i[1], ld = op.i[0];
  const bool staged = 2 * K <= c.tsm_floats;
  float* Ws = c.tsm;
  const float* hq[2] = {base + op.o[0] + (i64)row * ld, base + op.o[1] + (i64)row * ld};
  const float* ax[2] = {base + op.o[2] + (i64)row * ld, base + op.o[3] + (i64)row * ld};
  const bool fast = staged && row_fast(K, hq[0]) && ((ld & 3) == 0);
  const bool aux_is_h = op.o[2] == op.o[0];
  RowReg hr[2], ar[2];
  float bq[2] = {0.f, 0.f}, alpha = 0.f, lp_ = 0.f;
  if (in) {
    bq[0] = __ldcg(base + op.o[6]); bq[1] = __ldcg(base + op.o[7]);
    alpha = __ldcg(&c.scal->alpha_f32);
    lp_ = __ldcg(base + op.o[8] + row);
  }
  if (staged) {
    if (c.fresh) {
      stage_vec(Ws, base + op.o[4], K);
      stage_vec(Ws + K, base + op.o[5], K);
    }
    if (fast && in) {
      row_load(hr[0], hq[0], K, lane); row_load(hr[1], hq[1], K, lane);
      if (V == 1 && c.pf_rows && row + c.pf_rows < hp.B) {
        const i64 pf = (i64)c.pf_rows * ld;
        row_prefetch(hq[0] + pf, K, lane); row_prefetch(hq[1] + pf, K, lane);
        if (!aux_is_h) { row_prefetch(ax[0] + pf, K, lane); row_prefetch(ax[1] + pf, K, lane); }
      }
      if (!aux_is_h) { row_load(ar[0], ax[0], K, lane); row_load(ar[1], ax[1], K, lane); }
      else { ar[0] = hr[0]; ar[1] = hr[1]; }
    }
    if (c.fresh) stage_finish();
  }
  SACX_RSTAMP(1); SACX_RSTAMP(2); SACX_RSTAMP(3);
  if (!in) { SACX_RSTAMP(4); return; }
  float q[2], z[2];
#pragma unroll
  for (int n = 0; n < 2; ++n) {
    const float* W = staged ? Ws + n * K : base + op.o[4 + n];
    const float part = fast ? row_dot_partial(hr[n], W, K, lane) : warp_dot_any(hq[n], W, K, lane);
    z[n] = warp_sum(part) + bq[n];
    q[n] = act_fwd(op.act_out, z[n]);
  }
  const SacRoute g = sac_actor_route(op.act_out, z[0], q[0], z[1], q[1], hp.B_global);
  if (lane == 0) {
    base[op.o[9] + row] = q[0];
    base[op.o[10] + row] = q[1];
    base[op.o[15] + row] = sac_policy_loss_row(alpha, lp_, q[0], q[1]);
  }
#pragma unroll
  for (int n = 0; n < 2; ++n) {
    const float dout = n ? g.c2 : g.c1;
    const float* W = staged ? Ws + n * K : base + op.o[4 + n];
    float* dl = base + op.o[13 + n] + (i64)row * ld;
    if (fast) {
      const RowReg& a2 = ar[n];
#pragma unroll
      for (int i = 0; i < ROW_KREG; ++i) {
        const int k = (lane + 32 * i) * 4;
        if (k < K) *reinterpret_cast<float4*>(dl + k) = sac_delta(dout, *reinterpret_cast<const float4*>(W + k), a2.v[i], op.act);
      }
    } else {
      for (int k = lane; k < K; k += 32) dl[k] = sac_delta(dout, W[k], __ldcg(ax[n] + k), op.act);
    }
  }
  SACX_RSTAMP(4);
}

// ---------------------------------------------------------------- OP_ACTOR_BWD
// o[0..1]=delta0 of critics [B,H0q] o[2..3]=W_0 of critics [H0q, obs+act]
// o[4]=tz o[5]=se o[6]=mask o[7]=headz o[8]=dhead out o[9]=Wpi_L o[11]=aux pi(last hidden) o[12]=delta pi(last hidden)
// i[0]=ld delta0  i[1]=H0q  i[2]=ldW0 (=obs+act)  i[3]=ld pi hidden  i[4]=Kpi
template <int V>
__device__ __noinline__ void tile_actor_bwd(const Op& op, const RowCtx& c, int tile) {
  SACX_RSTAMP(0);
  const Hyper& hp = c.args->hp;
  float* base = c.base;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int row = tile * ROWS_PER_TILE + warp;
  const bool in = row < hp.B;
  const int A = hp.act, O = hp.obs, H0 = op.i[1], Kp = op.i[4];
  const bool staged = (2 * A * H0 + 2 * A * Kp) <= c.tsm_floats;
  float* Wa = c.tsm;                        // [2][A][H0]: action columns of the critics' first layers
  float* Wp = c.tsm + 2 * A * H0;           // [2A][Kp]: policy output layer
  const float* d0[2] = {base + op.o[0] + (i64)row * op.i[0], base + op.o[1] + (i64)row * op.i[0]};
  const float* auxp = base + op.o[11] + (i64)row * op.i[3];
  const bool fast = staged && row_fast(H0, d0[0]) && ((op.i[0] & 3) == 0) && row_fast(Kp, auxp) && ((op.i[3] & 3) == 0) &&
                    row_fast(Kp, Wp) && row_fast(H0, Wa);
  RowReg dr[2], ap;
  float alpha = 0.f, tz_ = 0.f, se_ = 0.f, mk_ = 0.f, zm_ = 0.f, zl_ = 0.f;       // lane j < A owns action dim j (A <= 32)
  if (in) {
    alpha = __ldcg(&c.scal->alpha_f32);
    if (lane < A) {
      tz_ = __ldcg(base + op.o[4] + (i64)row * A + lane);
      se_ = __ldcg(base + op.o[5] + (i64)row * A + lane);
      mk_ = __ldcg(base + op.o[6] + (i64)row * A + lane);
      if (op.act_out != SACX_ACT_IDENTITY) {
        zm_ = __ldcg(base + op.o[7] + (i64)row * 2 * A + lane);
        zl_ = __ldcg(base + op.o[7] + (i64)row * 2 * A + A + lane);
      }
    }
  }
  if (staged) {
    if (c.fresh) {
      for (int i = threadIdx.x; i < 2 * A * H0; i += 256) {
        const int n = i / (A * H0), j = (i / H0) % A, k = i % H0;
        Wa[i] = __ldcg(base + op.o[2 + n] + (i64)k * op.i[2] + O + j);
      }
      stage_vec(Wp, base + op.o[9], 2 * A * Kp);
    }
    if (fast && in) { row_load(dr[0], d0[0], H0, lane); row_load(dr[1], d0[1], H0, lane); row_load(ap, auxp, Kp, lane); }
    if (V == 1 && c.pf_rows && row + c.pf_rows < hp.B) {
      row_prefetch(d0[0] + (i64)c.pf_rows * op.i[0], H0, lane); row_prefetch(d0[1] + (i64)c.pf_rows * op.i[0], H0, lane);
      row_prefetch(auxp + (i64)c.pf_rows * op.i[3], Kp, lane);
    }
    if (c.fresh) stage_finish();
  }
  SACX_RSTAMP(1); SACX_RSTAMP(2); SACX_RSTAMP(3);
  if (!in) { SACX_RSTAMP(4); return; }
  float* da = c.wsm;                          // [A] dQ/da, then dhead [2A]
  float* dh = c.wsm + SACX_MAX_ACT;
  // d(-minQ)/d a_j = sum_c sum_h delta0_c[h] * W0_c[h, obs + j]
  for (int j = 0; j < A; ++j) {
    float s = 0.f;
#pragma unroll
    for (int n = 0; n < 2; ++n) {
      if (fast) s += row_dot_partial(dr[n], Wa + (n * A + j) * H0, H0, lane);
      else if (staged) s += warp_dot_any(d0[n], Wa + (n * A + j) * H0, H0, lane);
      else {
        const float* W0 = base + op.o[2 + n] + O + j;
        for (int k = lane; k < H0; k += 32) s = fmaf(__ldcg(d0[n] + k), __ldcg(W0 + (i64)k * op.i[2]), s);
      }
    }
    s = warp_sum(s);
    if (lane == 0) da[j] = s;
  }
  __syncwarp();
  const float ab = alpha / (float)hp.B_global;
  for (int j = lane; j < A; j += 32) {
    const SacHeadGrad g = sac_head_bwd(op.act_out, tz_, se_, mk_, da[j], ab, hp.action_scale, zm_, zl_);
    dh[j] = g.dmu;
    dh[A + j] = g.dls;
    base[op.o[8] + (i64)row * 2 * A + j] = g.dmu;
    base[op.o[8] + (i64)row * 2 * A + A + j] = g.dls;
  }
  __syncwarp();
  // delta of the policy's last hidden layer: (dhead . Wpi_L) * act'(.)
  float* dl = base + op.o[12] + (i64)row * op.i[3];
  if (fast) {
#pragma unroll
    for (int i = 0; i < ROW_KREG; ++i) {
      const int k = (lane + 32 * i) * 4;
      if (k < Kp) {
        float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
        for (int j = 0; j < 2 * A; ++j) {
          const float4 w = *reinterpret_cast<const float4*>(Wp + j * Kp + k);
          const float g = dh[j];
          s.x = fmaf(g, w.x, s.x); s.y = fmaf(g, w.y, s.y); s.z = fmaf(g, w.z, s.z); s.w = fmaf(g, w.w, s.w);
        }
        *reinterpret_cast<float4*>(dl + k) = sac_dact(s, ap.v[i], op.act);
      }
    }
  } else {
    const float* W = staged ? Wp : base + op.o[9];
    for (int k = lane; k < Kp; k += 32) {
      float s = 0.f;
      for (int j = 0; j < 2 * A; ++j) s = fmaf(dh[j], staged ? W[j * Kp + k] : __ldcg(W + (i64)j * Kp + k), s);
      dl[k] = sac_dact(s, __ldcg(auxp + k), op.act);
    }
  }
  __syncwarp();
  SACX_RSTAMP(4);
}

// ---------------------------------------------------------------- OP_PROLOGUE (one thread)
// mode = bitmask of optimisers (1 << OptId) whose step advances in this update
// beta^t for Adam's bias corrections (torch: `1 - beta ** step` in Python doubles). exp(t ln beta) instead of pow(): the fp64 pow
// was ~1.5 K cycles a call on this GPU, six calls per update on ONE thread that the rest of its 8-CTA group -- and at the phase
// barrier everyone -- waited for (10 K cycles in front of phase A; tools/phase_profile.py, tag 101 -> 1000). The product
// t ln(beta) carries |t ln beta| x 1.1e-16 <= 5e-15 of relative error into the result (beta^t < 4e-18 past |t ln beta| = 40 is
// dropped: 1 - beta^t rounds to 1.0 either way), far below what the float32 step size / the 1e-12 temperature check resolve.
__device__ __forceinline__ double adam_beta_pow(double ln_beta, i64 t) {
  const double x = (double)t * ln_beta;
  return x < -40.0 ? 0.0 : exp(x);
}
constexpr double LN_BETA1 = -0.10536051565782628;       // ln 0.9
constexpr double LN_BETA2 = -0.0010005003335835335;     // ln 0.999

// Adam step counters and bias-correction scalars of optimiser `o` (one lane each: the callers pass lanes 0-2)
__device__ __forceinline__ void op_prologue(const Op& op, const RowCtx& c, int o) {
  AgentScalars* s = c.scal;
  const Hyper& hp = c.args->hp;
  if (o >= 3 || !(op.mode & (1 << o))) return;
  const i64 t = s->step[o] + 1;
  s->step[o] = t;
  // python-double bias corrections of torch's _single_tensor_adam
  const double bc1 = 1.0 - adam_beta_pow(LN_BETA1, t);
  const double bc2 = 1.0 - adam_beta_pow(LN_BETA2, t);
  s->adam_step_size[o] = (float)((s->lr[o] > 0.0 ? s->lr[o] : hp.lr[o]) / bc1);      // per-agent learning rate when set
  s->adam_bc2_sqrt[o] = (float)sqrt(bc2);
}

// ---------------------------------------------------------------- OP_FINAL (one warp; CTA = true: the whole CTA, large batch)
// mode bits: 1 critic loss means, 2 policy loss mean, 4 temperature step, 8 count the update, 16/32 see below
// o[0..1]=lossrow o[2]=plossrow o[3]=lp o[4..5]=q o[6]=y
// sum over the callers (a warp, or all 256 threads through `red`), same value in every thread
template <bool CTA>
__device__ __forceinline__ float final_sum(float v, float* red) {
  v = warp_sum(v);
  if (!CTA) return v;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  __syncthreads();
  if (lane == 0) red[warp] = v;
  __syncthreads();
  float t = 0.f;
#pragma unroll
  for (int w = 0; w < 8; ++w) t += red[w];
  return t;
}
// scalar tail of OP_FINAL (one thread): temperature step from the entropy-gap means, update counter
__device__ __forceinline__ void final_tail(const Op& op, const RowCtx& c) {
  const Hyper& hp = c.args->hp;
  float* base = c.base;
  AgentScalars* s = c.scal;
  if (op.mode & (4 | 32)) {
    const float mean_t = (op.mode & 32) ? __ldcg(base + op.o[7]) : s->dp_mean_t;       // 32: the all-reduced shares
    const float mean_lt = (op.mode & 32) ? __ldcg(base + op.o[7] + 1) : s->dp_mean_lt;
    s->metrics[8] = mean_t - hp.target_entropy;
    if (hp.auto_alpha) {
      // alpha_loss = -(log_alpha * (logpi + H).detach()).mean();  d/dlog_alpha = -mean(logpi + H)
      // alpha_lr < 0: temperature frozen -- what the reference does after load_agent, where the optimiser keeps stepping the
      // pre-load tensor (agent.py:549-554); SAC.load_agent(..., reference_temperature_semantics=True) selects it
      if (!(s->alpha_lr < 0.0)) {
        const double g = -(double)mean_t;
        const i64 t = s->step[OPT_ALPHA] + 1;
        s->step[OPT_ALPHA] = t;
        s->alpha_m = s->alpha_m + (1.0 - 0.9) * (g - s->alpha_m);
        s->alpha_v = s->alpha_v * 0.999 + (1.0 - 0.999) * g * g;
        const double bc1 = 1.0 - adam_beta_pow(LN_BETA1, t), bc2 = 1.0 - adam_beta_pow(LN_BETA2, t);
        const double denom = sqrt(s->alpha_v) / sqrt(bc2) + 1e-8;
        const double alr = s->alpha_lr > 0.0 ? s->alpha_lr : hp.alpha_lr;      // per-agent override (Optuna trials as a population)
        s->log_alpha = s->log_alpha - (alr / bc1) * (s->alpha_m / denom);
        s->alpha = exp(s->log_alpha);
        s->alpha_f32 = (float)s->alpha;
      }
      s->metrics[3] = -mean_lt;
    }
    s->metrics[4] = (float)s->alpha;
    s->metrics[5] = (float)s->log_alpha;
  }
  if (op.mode & 8) s->updates += 1;
}
template <bool CTA>
__device__ __forceinline__ void op_final_impl(const Op& op, const RowCtx& c, int lane, float* red) {
  const Hyper& hp = c.args->hp;
  float* base = c.base;
  AgentScalars* s = c.scal;
  const int B = hp.B;
  const float invB = 1.f / (float)hp.B_global;
  constexpr int NT = CTA ? 256 : 32;
  auto mean_of = [&](const float* p) {
    float acc[4] = {0.f, 0.f, 0.f, 0.f};
    if (CTA && (B & 3) == 0 && ((((uintptr_t)p) & 15) == 0)) {
      // large batch: 16-byte loads, four per thread in flight (a 65536-term mean was 60 us of dependent round trips)
      const float4* p4 = reinterpret_cast<const float4*>(p);
      const int n4 = B >> 2;
      float4 a4[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) a4[u] = make_float4(0.f, 0.f, 0.f, 0.f);
      int i = lane;
      for (; i + 3 * NT < n4; i += 4 * NT) {
        const float4 v0 = __ldcg(p4 + i), v1 = __ldcg(p4 + i + NT), v2 = __ldcg(p4 + i + 2 * NT), v3 = __ldcg(p4 + i + 3 * NT);
        a4[0].x += v0.x; a4[0].y += v0.y; a4[0].z += v0.z; a4[0].w += v0.w;
        a4[1].x += v1.x; a4[1].y += v1.y; a4[1].z += v1.z; a4[1].w += v1.w;
        a4[2].x += v2.x; a4[2].y += v2.y; a4[2].z += v2.z; a4[2].w += v2.w;
        a4[3].x += v3.x; a4[3].y += v3.y; a4[3].z += v3.z; a4[3].w += v3.w;
      }
      for (; i < n4; i += NT) { const float4 v = __ldcg(p4 + i); a4[0].x += v.x; a4[0].y += v.y; a4[0].z += v.z; a4[0].w += v.w; }
      const float s = ((a4[0].x + a4[0].y) + (a4[0].z + a4[0].w)) + ((a4[1].x + a4[1].y) + (a4[1].z + a4[1].w)) +
                      ((a4[2].x + a4[2].y) + (a4[2].z + a4[2].w)) + ((a4[3].x + a4[3].y) + (a4[3].z + a4[3].w));
      return final_sum<CTA>(s, red) * invB;
    }
    int b = lane;
    for (; b + 3 * NT < B; b += 4 * NT) {        // four independent loads in flight per thread
      acc[0] += __ldcg(p + b); acc[1] += __ldcg(p + b + NT); acc[2] += __ldcg(p + b + 2 * NT); acc[3] += __ldcg(p + b + 3 * NT);
    }
    for (; b < B; b += NT) acc[0] += __ldcg(p + b);
    return final_sum<CTA>((acc[0] + acc[1]) + (acc[2] + acc[3]), red) * invB;
  };
  if (op.mode & 1) {
    const float l1 = mean_of(base + op.o[0]), l2 = mean_of(base + op.o[1]);
    const float q1 = mean_of(base + op.o[4]), q2 = mean_of(base + op.o[5]);
    const float ym = mean_of(base + op.o[6]);
    if (lane == 0) { s->metrics[0] = l1; s->metrics[1] = l2; s->metrics[6] = q1; s->metrics[7] = q2; s->metrics[9] = ym; }
  }
  if (op.mode & 2) {
    const float pl = mean_of(base + op.o[2]);
    if (lane == 0) s->metrics[2] = pl;
  }
  // temperature (a9): bit 4 = gradient + step (single GPU); bit 16 = this rank's share of the gradient only;
  // bit 32 = step from the (all-reduced) shares in the scalar block
  if (op.mode & (4 | 16)) {
    const float* lp = c.args->lp_ext ? c.args->lp_ext : base + op.o[3];
    float acc = 0.f, accl = 0.f;
    const float la32 = (float)s->log_alpha;
    if (CTA && (B & 3) == 0 && ((((uintptr_t)lp) & 15) == 0)) {
      const float4* p4 = reinterpret_cast<const float4*>(lp);
      for (int i = lane; i < (B >> 2); i += NT) {
        const float4 v = __ldcg(p4 + i);
        const float t0 = v.x + hp.target_entropy, t1 = v.y + hp.target_entropy, t2 = v.z + hp.target_entropy, t3 = v.w + hp.target_entropy;
        acc += (t0 + t1) + (t2 + t3);
        accl += (la32 * t0 + la32 * t1) + (la32 * t2 + la32 * t3);
      }
    } else
    for (int b = lane; b < B; b += NT) {
      const float t = __ldcg(lp + b) + hp.target_entropy;
      acc += t;
      accl += la32 * t;
    }
    const float mean_t = final_sum<CTA>(acc, red) * invB;           // f32 mean, as in the reference
    const float mean_lt = final_sum<CTA>(accl, red) * invB;
    if (lane == 0) {
      s->dp_mean_t = mean_t; s->dp_mean_lt = mean_lt;
      if (op.mode & 16) { base[op.o[7]] = mean_t; base[op.o[7] + 1] = mean_lt; }      // travels with the policy gradients
    }
    if (CTA) __syncthreads();
  }
  if (lane == 0) final_tail(op, c);
}
__device__ __forceinline__ void op_final(const Op& op, const RowCtx& c, int lane) { op_final_impl<false>(op, c, lane, nullptr); }
// Row-parallel kernel (batch <= 512): the whole CTA is called, warp k takes the k-th mean -- each with the summation order of
// op_final_impl<false> (lane-strided, four loads in flight, butterfly) -- and thread 0 finishes. One warp doing the seven means
// one after the other made this tile (17.6 K cycles) the longest of its phase, 6 K past the weight-gradient tiles.
// red: 16 floats of shared memory.
__device__ __forceinline__ void op_final_par(const Op& op, const RowCtx& c, float* red) {
  const Hyper& hp = c.args->hp;
  float* base = c.base;
  AgentScalars* s = c.scal;
  const int B = hp.B, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const float invB = 1.f / (float)hp.B_global;
  auto warp_mean = [&](const float* p) {
    float acc[4] = {0.f, 0.f, 0.f, 0.f};
    int b = lane;
    for (; b + 96 < B; b += 128) {
      acc[0] += __ldcg(p + b); acc[1] += __ldcg(p + b + 32); acc[2] += __ldcg(p + b + 64); acc[3] += __ldcg(p + b + 96);
    }
    for (; b < B; b += 32) acc[0] += __ldcg(p + b);
    return warp_sum((acc[0] + acc[1]) + (acc[2] + acc[3])) * invB;
  };
  float r = 0.f, r2 = 0.f;
  if (op.mode & 1) {
    if (warp == 0) r = warp_mean(base + op.o[0]);
    else if (warp == 1) r = warp_mean(base + op.o[1]);
    else if (warp == 2) r = warp_mean(base + op.o[4]);
    else if (warp == 3) r = warp_mean(base + op.o[5]);
    else if (warp == 4) r = warp_mean(base + op.o[6]);
  }
  if ((op.mode & 2) && warp == 5) r = warp_mean(base + op.o[2]);
  if ((op.mode & (4 | 16)) && warp == 6) {
    const float* lp = c.args->lp_ext ? c.args->lp_ext : base + op.o[3];
    float acc = 0.f, accl = 0.f;
    const float la32 = (float)s->log_alpha;
    for (int b = lane; b < B; b += 32) {
      const float t = __ldcg(lp + b) + hp.target_entropy;
      acc += t;
      accl += la32 * t;
    }
    r = warp_sum(acc) * invB;             // f32 mean, as in the reference
    r2 = warp_sum(accl) * invB;
  }
  if (lane == 0) { red[warp] = r; if (warp == 6) red[8] = r2; }
  __syncthreads();
  if (threadIdx.x == 0) {
    if (op.mode & 1) { s->metrics[0] = red[0]; s->metrics[1] = red[1]; s->metrics[6] = red[2]; s->metrics[7] = red[3]; s->metrics[9] = red[4]; }
    if (op.mode & 2) s->metrics[2] = red[5];
    if (op.mode & (4 | 16)) {
      s->dp_mean_t = red[6]; s->dp_mean_lt = red[8];
      if (op.mode & 16) { base[op.o[7]] = red[6]; base[op.o[7] + 1] = red[8]; }      // travels with the policy gradients
    }
    final_tail(op, c);
  }
}

// ---------------------------------------------------------------- OP_POLYAK / OP_ADAM_FLAT (elementwise tiles)
constexpr int FLAT_TILE = 256 * 8;
// OP_POLYAK: o[0]=online o[1]=target o[2]=count
__device__ __forceinline__ void op_polyak(const Op& op, const RowCtx& c, int tile) {
  float* base = c.base;
  const i64 n = op.o[2];
  const float tau = __ldcg(&c.scal->tau), omt = __ldcg(&c.scal->one_minus_tau);
  for (i64 e = (i64)tile * FLAT_TILE + threadIdx.x; e < n && e < (i64)(tile + 1) * FLAT_TILE; e += 256) {
    const float p = __ldcg(base + op.o[0] + e);
    float* t = base + op.o[1] + e;
    *t = polyak_mix(tau, omt, p, __ldcg(t));
  }
}
// OP_ADAM_FLAT: o[0]=p o[1]=m o[2]=v o[3]=g o[4]=count o[5]=target or -1 (Polyak after the step)
__device__ __forceinline__ void op_adam_flat(const Op& op, const RowCtx& c, int tile) {
  float* base = c.base;
  const i64 n = op.o[4];
  const float ss = __ldcg(&c.scal->adam_step_size[op.opt]), bc = __ldcg(&c.scal->adam_bc2_sqrt[op.opt]);
  const float tau = __ldcg(&c.scal->tau), omt = __ldcg(&c.scal->one_minus_tau);
  for (i64 e = (i64)tile * FLAT_TILE + threadIdx.x; e < n && e < (i64)(tile + 1) * FLAT_TILE; e += 256) {
    float p = __ldcg(base + op.o[0] + e), m = __ldcg(base + op.o[1] + e), v = __ldcg(base + op.o[2] + e);
    adam_update(__ldcg(base + op.o[3] + e), p, m, v, ss, bc);
    base[op.o[0] + e] = p;
    base[op.o[1] + e] = m;
    base[op.o[2] + e] = v;
    if (op.o[5] >= 0) {
      float* t = base + op.o[5] + e;
      *t = polyak_mix(tau, omt, p, __ldcg(t));
    }
  }
}

}  // namespace sacx
