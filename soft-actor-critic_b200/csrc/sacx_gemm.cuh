// FP32 tiled GEMM for the MLP layers of the SAC update, with the layer's elementwise work fused into
// the epilogue (bias+activation forward, activation-derivative backward, Adam(+Polyak) on dW).
//
// One CTA (256 threads) computes a BM x BN output tile; every thread owns an 8x8 register microtile
// (64 FFMA per 4 LDS.128 -- the ratio at which shared-memory bandwidth stops being the limiter) and the
// K range is split over KG thread groups inside the CTA (intra-CTA split-K), reduced through shared
// memory at the end. At batch 256 / hidden 256 a layer is only 256x256x256, so the latency configuration
// uses 32x32 tiles (16 K-groups) to spread one layer over the 148 SMs; the throughput configuration
// (population / large batch) uses 64x64 tiles (4 K-groups).
//
// Operands move global -> shared with cp.async.cg (16 B, L2-only so that data written by other SMs in the
// previous phase is seen) through a 4-stage ring: for K <= 256 the whole tile is in flight at once, so a
// tile pays one L2 round trip instead of one per K block (measured: the register-prefetch version
// serialised ~1.6K cycles of load latency with ~1.4K cycles of math per 64-wide K block). Shared tiles
// keep the global orientation -- [row][k] when K is contiguous in memory (activations, nn.Linear weights
// in the forward pass) and [k][row] otherwise (weights in backward-dA, both operands of dW) -- so no
// transposition is needed on the way in; the fragment loads transpose in registers for free.
// Epilogue operands (bias / saved activation / parameter, Adam moments, target) are prefetched into
// registers when the tile starts, so the epilogue adds no dependent L2 round trip.
//
// Precision: plain FFMA, fp32 accumulate -- the parity contract is rel 1e-4 against the fp32 reference,
// which rules out TF32/BF16 tensor-core inputs for this path (SURVEY 2b note).
#pragma once
#include "sacx_math.cuh"
#include "sacx_types.cuh"

namespace sacx {

constexpr int GEMM_BK = 64;      // K extent of one pipeline stage
constexpr int GEMM_NS = 4;       // stages in the cp.async ring
constexpr int GEMM_LDK = GEMM_BK + 4;

template <int BM_, int BN_>
struct TileCfg {
  static constexpr int BM = BM_, BN = BN_;
  static constexpr int TY = BM / 8, TX = BN / 8;          // thread grid inside one K group
  static constexpr int TPG = TY * TX;                     // threads per K group
  static constexpr int KG = 256 / TPG;                    // K groups
  static constexpr int KPG = GEMM_BK / KG;                // k per group per stage
  static constexpr int A_FLOATS = (BM * GEMM_LDK > GEMM_BK * (BM + 4)) ? BM * GEMM_LDK : GEMM_BK * (BM + 4);
  static constexpr int B_FLOATS = (BN * GEMM_LDK > GEMM_BK * (BN + 4)) ? BN * GEMM_LDK : GEMM_BK * (BN + 4);
  static constexpr int STAGE_FLOATS = A_FLOATS + B_FLOATS;
  static constexpr int RS = BN + 4;                       // reduction row stride (+1 column for bias sums)
  static constexpr int RBLK = BM * RS + 16;              // per-K-group block (+16: the two K groups of a warp hit disjoint banks)
  static constexpr int RED_FLOATS = KG * RBLK;
  static constexpr int PIPE_FLOATS = GEMM_NS * STAGE_FLOATS;
  static constexpr int SMEM_FLOATS = PIPE_FLOATS > RED_FLOATS ? PIPE_FLOATS : RED_FLOATS;   // red aliases the ring
  static constexpr int NV = BM * BN / 4 / 256;            // float4 outputs per thread in the epilogue
  static_assert(KPG % 4 == 0 && KPG >= 4, "each K group consumes whole float4 K blocks");
};

using CfgSmall = TileCfg<32, 32>;     // latency config: many small tiles (single agent)
using CfgLarge = TileCfg<64, 64>;     // throughput config: population / large batch

struct EpiCtx {
  float* base;                  // agent arena base
  const AgentScalars* scal;
  const Hyper* hp;
  unsigned long long* t;        // optional intra-tile timestamps (profiling aid), 8 slots
};
// (intra-tile timestamps for tools/phase_profile.py: debug library only, like the row-parallel kernel's event trace)
#ifdef SACX_DEBUG_HOOKS
#define SACX_TSTAMP(i) do { if (ctx.t && threadIdx.x == 0) ctx.t[i] = clock64(); } while (0)
#else
#define SACX_TSTAMP(i) do { } while (0)
#endif

// ---- cp.async helpers --------------------------------------------------------------------------------
__device__ __forceinline__ void cp_async16(float* smem_dst, const float* gsrc, int src_bytes) {
  const unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(d), "l"(gsrc), "r"(src_bytes) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// One operand tile of a stage: R rows (m or n) x 64 k.
//   kmajor == false: element (row, k) at base[row*ld + k]  -> smem S[row*LDK + k]
//   kmajor == true : element (row, k) at base[k*ld + row]  -> smem S[k*(R+4) + row]
// vec: 16-byte aligned rows -> cp.async with zero fill; otherwise a synchronous scalar path.
template <int R, bool kmajor>
__device__ __forceinline__ void stage_load(float* __restrict__ S, const float* __restrict__ base, int ld,
                                           bool vec, int row0, int rows_total, int k0, int k_total) {
  const int tid = threadIdx.x;
#pragma unroll
  for (int i = 0; i < R / 16; ++i) {
    const int id = tid + i * 256;
    int row, k, avail;
    float* dst;
    const float* src;
    if (!kmajor) {
      row = id >> 4; k = (id & 15) << 2;
      dst = S + row * GEMM_LDK + k;
      src = base + (i64)(row0 + row) * ld + (k0 + k);
      avail = (row0 + row < rows_total) ? (k_total - (k0 + k)) : 0;
    } else {
      k = id / (R / 4); row = (id % (R / 4)) << 2;
      dst = S + k * (R + 4) + row;
      src = base + (i64)(k0 + k) * ld + (row0 + row);
      avail = (k0 + k < k_total) ? (rows_total - (row0 + row)) : 0;
    }
    avail = avail < 0 ? 0 : (avail > 4 ? 4 : avail);
    if (vec) {
      cp_async16(dst, avail > 0 ? src : base, avail * 4);
    } else {
      float4 t = make_float4(0.f, 0.f, 0.f, 0.f);
      if (avail > 0) t.x = __ldcg(src + 0);
      if (avail > 1) t.y = __ldcg(src + 1);
      if (avail > 2) t.z = __ldcg(src + 2);
      if (avail > 3) t.w = __ldcg(src + 3);
      *reinterpret_cast<float4*>(dst) = t;
    }
  }
}

// ---- epilogues ---------------------------------------------------------------------------------------
struct EpiPre {            // operands prefetched at tile start (latency config, one float4 per thread)
  float4 a, b, c, d;       // FWD: a=bias | DACT: a=aux | DW: a=p b=m c=v d=target
  float ss, bc, tau, omt;
  bool valid;
};

__device__ __forceinline__ bool epi_vec_ok(const Op& op, int n) {
  if (n + 3 >= op.N) return false;
  if (op.epi == EPI_FWD) return ((op.bias | op.c) & 3) == 0 && (op.ldc & 3) == 0 && (op.zout < 0 || (op.zout & 3) == 0);
  if (op.epi == EPI_DACT) return ((op.aux | op.c) & 3) == 0 && ((op.ldc | op.ld_aux) & 3) == 0;
  return (op.N & 3) == 0 && ((op.p | op.pm | op.pv | op.pg) & 3) == 0 && (op.pt < 0 || (op.pt & 3) == 0);
}

template <int MODE>
__device__ __forceinline__ void epi_prefetch(const Op& op, const EpiCtx& ctx, int m, int n, EpiPre& pre) {
  pre.valid = (m < op.M) && epi_vec_ok(op, n);
  if (!pre.valid) return;
  const float* base = ctx.base;
  if (MODE == 0) {
    pre.a = __ldcg(reinterpret_cast<const float4*>(base + op.bias + n));
  } else if (MODE == 1) {
    pre.a = __ldcg(reinterpret_cast<const float4*>(base + op.aux + (i64)m * op.ld_aux + n));
  } else if (op.flags & DW_ADAM) {
    const i64 e = (i64)m * op.N + n;
    pre.a = __ldcg(reinterpret_cast<const float4*>(base + op.p + e));
    pre.b = __ldcg(reinterpret_cast<const float4*>(base + op.pm + e));
    pre.c = __ldcg(reinterpret_cast<const float4*>(base + op.pv + e));
    if (op.flags & DW_POLYAK) pre.d = __ldcg(reinterpret_cast<const float4*>(base + op.pt + e));
    pre.ss = __ldcg(&ctx.scal->adam_step_size[op.opt]);
    pre.bc = __ldcg(&ctx.scal->adam_bc2_sqrt[op.opt]);
    if (op.flags & DW_POLYAK) { pre.tau = __ldcg(&ctx.scal->tau); pre.omt = __ldcg(&ctx.scal->one_minus_tau); }
  }
}

template <int MODE>
__device__ __forceinline__ void epilogue_row4(const Op& op, const EpiCtx& ctx, int m, int n, float4 acc, EpiPre& pre,
                                              bool have_pre) {
  float* base = ctx.base;
  if (m >= op.M || n >= op.N) return;
  if (!have_pre) epi_prefetch<MODE>(op, ctx, m, n, pre);
  const bool vec = pre.valid;
  float v[4] = {acc.x, acc.y, acc.z, acc.w};
  if (MODE == 0) {
    float* c = base + op.c + (i64)m * op.ldc + n;
    float* z = op.zout >= 0 ? base + op.zout + (i64)m * op.ldc + n : nullptr;
    if (vec) {
      const float4 zz = make_float4(v[0] + pre.a.x, v[1] + pre.a.y, v[2] + pre.a.z, v[3] + pre.a.w);
      if (z) *reinterpret_cast<float4*>(z) = zz;
      *reinterpret_cast<float4*>(c) = make_float4(act_fwd(op.act, zz.x), act_fwd(op.act, zz.y), act_fwd(op.act, zz.z), act_fwd(op.act, zz.w));
    } else {
      const float* bias = base + op.bias + n;
#pragma unroll
      for (int j = 0; j < 4; ++j)
        if (n + j < op.N) {
          const float zz = v[j] + __ldcg(bias + j);
          if (z) z[j] = zz;
          c[j] = act_fwd(op.act, zz);
        }
    }
  } else if (MODE == 1) {
    float* c = base + op.c + (i64)m * op.ldc + n;
    if (vec) {
      *reinterpret_cast<float4*>(c) = make_float4(v[0] * act_dz(op.act, pre.a.x), v[1] * act_dz(op.act, pre.a.y),
                                                  v[2] * act_dz(op.act, pre.a.z), v[3] * act_dz(op.act, pre.a.w));
    } else {
      const float* aux = base + op.aux + (i64)m * op.ld_aux + n;
#pragma unroll
      for (int j = 0; j < 4; ++j)
        if (n + j < op.N) c[j] = v[j] * act_dz(op.act, __ldcg(aux + j));
    }
  } else {  // EPI_DW: (m, n) = (out neuron, in feature); parameter leading dim = N (= K_in)
    const i64 e = (i64)m * op.N + n;
    if (op.flags & DW_ATOMIC) {
#pragma unroll
      for (int j = 0; j < 4; ++j)
        if (n + j < op.N) atomicAdd(base + op.pg + e + j, v[j]);
    } else if (vec) {
      if (op.flags & DW_STORE_GRAD) *reinterpret_cast<float4*>(base + op.pg + e) = acc;
      if (op.flags & DW_ADAM) {
        float p[4] = {pre.a.x, pre.a.y, pre.a.z, pre.a.w}, mm[4] = {pre.b.x, pre.b.y, pre.b.z, pre.b.w},
              vv[4] = {pre.c.x, pre.c.y, pre.c.z, pre.c.w}, t[4] = {pre.d.x, pre.d.y, pre.d.z, pre.d.w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          adam_update(v[j], p[j], mm[j], vv[j], pre.ss, pre.bc);
          if (op.flags & DW_POLYAK) t[j] = polyak_mix(pre.tau, pre.omt, p[j], t[j]);
        }
        *reinterpret_cast<float4*>(base + op.p + e) = make_float4(p[0], p[1], p[2], p[3]);
        *reinterpret_cast<float4*>(base + op.pm + e) = make_float4(mm[0], mm[1], mm[2], mm[3]);
        *reinterpret_cast<float4*>(base + op.pv + e) = make_float4(vv[0], vv[1], vv[2], vv[3]);
        if (op.flags & DW_POLYAK) *reinterpret_cast<float4*>(base + op.pt + e) = make_float4(t[0], t[1], t[2], t[3]);
      }
    } else {
      const float ss = __ldcg(&ctx.scal->adam_step_size[op.opt]), bc = __ldcg(&ctx.scal->adam_bc2_sqrt[op.opt]);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        if (n + j < op.N) {
          const float g = v[j];
          if (op.flags & DW_STORE_GRAD) base[op.pg + e + j] = g;
          if (op.flags & DW_ADAM) {
            float p = __ldcg(base + op.p + e + j), mm = __ldcg(base + op.pm + e + j), vv = __ldcg(base + op.pv + e + j);
            adam_update(g, p, mm, vv, ss, bc);
            base[op.p + e + j] = p;
            base[op.pm + e + j] = mm;
            base[op.pv + e + j] = vv;
            if (op.flags & DW_POLYAK) {
              float* t = base + op.pt + e + j;
              *t = polyak_mix(__ldcg(&ctx.scal->tau), __ldcg(&ctx.scal->one_minus_tau), p, __ldcg(t));
            }
          }
        }
      }
    }
  }
}

__device__ __forceinline__ void epilogue_bias(const Op& op, const EpiCtx& ctx, int m, float g, const float (&bpre)[8]) {
  if (m >= op.M) return;
  float* base = ctx.base;
  if (op.flags & DW_ATOMIC) { atomicAdd(base + op.pbg + m, g); return; }
  if (op.flags & DW_STORE_GRAD) base[op.pbg + m] = g;
  if (op.flags & DW_ADAM) {
    const float ss = bpre[4], bc = bpre[5];
    float p = bpre[0], mm = bpre[1], vv = bpre[2];
    adam_update(g, p, mm, vv, ss, bc);
    base[op.pb + m] = p;
    base[op.pbm + m] = mm;
    base[op.pbv + m] = vv;
    if (op.flags & DW_POLYAK) base[op.pbt + m] = polyak_mix(bpre[6], bpre[7], p, bpre[3]);
  }
}

// ---- the math -------------------------------------------------------------------------------------------
// Thread (kg, ty, tx) accumulates its 8x8 microtile; one "block" = 4 consecutive k of its K group.
//   row-major operand: rows {ty + TY*i}, fragment = float4 along k     (conflict-free: consecutive rows, LDK=68)
//   k-major operand  : rows {h*BM/2 + 4*ty + ii}, fragment = float4 along the rows
// The A block (8 rows x 4 k) is loaded whole and double-buffered across blocks; B is streamed one float4 at a
// time, so the live fragment registers stay at ~72 next to the 64 accumulators.
template <class C, bool AKM>
__device__ __forceinline__ void load_a_block(const float* __restrict__ As, int kb, int ty, float (&a)[8][4]) {
  if (!AKM) {
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const float4 q = *reinterpret_cast<const float4*>(As + (ty + C::TY * i) * GEMM_LDK + kb);
      a[i][0] = q.x; a[i][1] = q.y; a[i][2] = q.z; a[i][3] = q.w;
    }
  } else {
#pragma unroll
    for (int kk = 0; kk < 4; ++kk)
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const float4 q = *reinterpret_cast<const float4*>(As + (kb + kk) * (C::BM + 4) + h * (C::BM / 2) + 4 * ty);
        a[h * 4 + 0][kk] = q.x; a[h * 4 + 1][kk] = q.y; a[h * 4 + 2][kk] = q.z; a[h * 4 + 3][kk] = q.w;
      }
  }
}

template <class C, bool BKM, bool BSUM>
__device__ __forceinline__ void block_math(const float (&a)[8][4], const float* __restrict__ Bs, int kb, int tx,
                                           float (&acc)[8][8], float (&bsum)[8]) {
  if (!BKM) {
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const float4 q = *reinterpret_cast<const float4*>(Bs + (tx + C::TX * j) * GEMM_LDK + kb);
      const float b[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
      for (int kk = 0; kk < 4; ++kk)
#pragma unroll
        for (int i = 0; i < 8; ++i) acc[i][j] = fmaf(a[i][kk], b[kk], acc[i][j]);
    }
  } else {
#pragma unroll
    for (int kk = 0; kk < 4; ++kk) {
      const float4 q0 = *reinterpret_cast<const float4*>(Bs + (kb + kk) * (C::BN + 4) + 4 * tx);
      const float4 q1 = *reinterpret_cast<const float4*>(Bs + (kb + kk) * (C::BN + 4) + (C::BN / 2) + 4 * tx);
      const float b[8] = {q0.x, q0.y, q0.z, q0.w, q1.x, q1.y, q1.z, q1.w};
#pragma unroll
      for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] = fmaf(a[i][kk], b[j], acc[i][j]);
    }
  }
  if (BSUM) {
#pragma unroll
    for (int kk = 0; kk < 4; ++kk)
#pragma unroll
      for (int i = 0; i < 8; ++i) bsum[i] += a[i][kk];
  }
}

#ifndef SACX_MATH_VARIANT
#define SACX_MATH_VARIANT 1
#endif

template <class C, bool BKM>
__device__ __forceinline__ void load_b_block(const float* __restrict__ Bs, int kb, int tx, float (&b)[8][4]) {
  if (!BKM) {
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const float4 q = *reinterpret_cast<const float4*>(Bs + (tx + C::TX * j) * GEMM_LDK + kb);
      b[j][0] = q.x; b[j][1] = q.y; b[j][2] = q.z; b[j][3] = q.w;
    }
  } else {
#pragma unroll
    for (int kk = 0; kk < 4; ++kk)
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const float4 q = *reinterpret_cast<const float4*>(Bs + (kb + kk) * (C::BN + 4) + h * (C::BN / 2) + 4 * tx);
        b[h * 4 + 0][kk] = q.x; b[h * 4 + 1][kk] = q.y; b[h * 4 + 2][kk] = q.z; b[h * 4 + 3][kk] = q.w;
      }
  }
}

// all blocks of one stage. `more`: the next stage has landed too, so fragments may be prefetched across the boundary
template <class C, bool AKM, bool BKM, bool BSUM>
__device__ __forceinline__ void stage_math(const float* __restrict__ st, const float* __restrict__ st_next, bool more, int kg,
                                           int ty, int tx, float (&a_cur)[8][4], float (&acc)[8][8], float (&bsum)[8]) {
  constexpr int NB = C::KPG / 4;            // blocks per stage
#if SACX_MATH_VARIANT == 0
#pragma unroll
  for (int q = 0; q < NB; ++q) {
    const int kb = kg * C::KPG + q * 4;
    float a_nxt[8][4];
    if (q + 1 < NB) load_a_block<C, AKM>(st, kb + 4, ty, a_nxt);
    else if (more) load_a_block<C, AKM>(st_next, kg * C::KPG, ty, a_nxt);
    block_math<C, BKM, BSUM>(a_cur, st + C::A_FLOATS, kb, tx, acc, bsum);
    if (q + 1 < NB || more) {
#pragma unroll
      for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int kk = 0; kk < 4; ++kk) a_cur[i][kk] = a_nxt[i][kk];
    }
  }
#else
  // whole-block fragments (16 LDS.128) then 256 FFMA; the compiler is free to interleave
#pragma unroll
  for (int q = 0; q < NB; ++q) {
    const int kb = kg * C::KPG + q * 4;
    float a[8][4], b[8][4];
    load_a_block<C, AKM>(st, kb, ty, a);
    load_b_block<C, BKM>(st + C::A_FLOATS, kb, tx, b);
#pragma unroll
    for (int kk = 0; kk < 4; ++kk) {
#pragma unroll
      for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] = fmaf(a[i][kk], b[j][kk], acc[i][j]);
      if (BSUM) {
#pragma unroll
        for (int i = 0; i < 8; ++i) bsum[i] += a[i][kk];
      }
    }
  }
#endif
}

// ---- the tile --------------------------------------------------------------------------------------------
// MODE 0: forward      C = X . W^T      A [m][k] row-major, B [n][k] row-major
// MODE 1: backward dA  C = dY . W       A [m][k] row-major, B [k][n] k-major
// MODE 2: dW           C = dY^T . X     A [k][m] k-major,   B [k][n] k-major   (+ column sums of A = bias gradient)
template <class C, int MODE>
__device__ __noinline__ void gemm_tile_impl(const Op& op, const EpiCtx& ctx, int tile, float* __restrict__ smem) {
  constexpr bool AKM = (MODE == 2), BKM = (MODE >= 1), BSUM = (MODE == 2);
  constexpr int BM = C::BM, BN = C::BN, RS = C::RS, KG = C::KG;
  const int tid = threadIdx.x;
  // dW at large batch: the reduction (batch) range is split over op.i[0] CTAs, partial sums meet in the gradient
  // block with atomic adds (DW_ATOMIC)
  const int ksplit = (MODE == 2 && op.i[0] > 1) ? op.i[0] : 1;
  const int tiles_mn = op.ntiles / ksplit;
  const int ks = tile / tiles_mn, tmn = tile % tiles_mn;
  const int tm = tmn / op.tiles_n, tn = tmn % op.tiles_n;
  const int m0 = tm * BM, n0 = tn * BN;
  const int kc = (MODE == 2 && ksplit > 1) ? op.i[1] : 0;
  const float* __restrict__ A = ctx.base + op.a + (AKM ? (i64)ks * kc * op.a_sk : 0);
  const float* __restrict__ Bp = ctx.base + op.b + (BKM && MODE == 2 ? (i64)ks * kc * op.b_sk : 0);
  const int lda = AKM ? op.a_sk : op.a_sm;
  const int ldb = BKM ? op.b_sk : op.b_sn;
  const bool a_vec = op.a_vec != 0, b_vec = op.b_vec != 0;
  const int M = op.M, N = op.N;
  const int K = (ksplit > 1) ? min(kc, op.K - ks * kc) : op.K;
  const bool bias_tile = BSUM && (tn == 0) && (op.pb >= 0);
  const int nk = (K + GEMM_BK - 1) / GEMM_BK;
  SACX_TSTAMP(0);

  const int kg = tid / C::TPG, t = tid % C::TPG;
  const int ty = t / C::TX, tx = t % C::TX;
  float acc[8][8];
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;
  float bsum[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) bsum[i] = 0.f;
  EpiPre pre;
  pre.valid = false;
  float bpre[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};        // bias-row operands (p, m, v, target, step size, bc2, tau, 1 - tau) of dW

  // epilogue operands travel while the pipeline fills
  if (C::NV == 1) epi_prefetch<MODE>(op, ctx, m0 + tid / (BN / 4), n0 + (tid % (BN / 4)) * 4, pre);
  if (bias_tile && (op.flags & DW_ADAM) && tid < BM && m0 + tid < M) {
    bpre[0] = __ldcg(ctx.base + op.pb + m0 + tid);
    bpre[1] = __ldcg(ctx.base + op.pbm + m0 + tid);
    bpre[2] = __ldcg(ctx.base + op.pbv + m0 + tid);
    if (op.flags & DW_POLYAK) bpre[3] = __ldcg(ctx.base + op.pbt + m0 + tid);
    bpre[4] = __ldcg(&ctx.scal->adam_step_size[op.opt]);
    bpre[5] = __ldcg(&ctx.scal->adam_bc2_sqrt[op.opt]);
    if (op.flags & DW_POLYAK) { bpre[6] = __ldcg(&ctx.scal->tau); bpre[7] = __ldcg(&ctx.scal->one_minus_tau); }
  }

  // NS-deep cp.async ring as ONE rolled loop (one copy of the load and math code per variant keeps the
  // instruction footprint small: instruction-fetch stalls were 30% of this kernel's samples). Iteration j issues
  // stage j and consumes stage j-(NS-1); for K <= 192 the whole K range is in flight before the first wait.
  float a_cur[8][4];
#pragma unroll 1
  for (int j = 0; j < nk + GEMM_NS - 1; ++j) {
    const int it = j - (GEMM_NS - 1);
    if (it >= 0) {
      cp_async_wait<GEMM_NS - 3>();          // stages it and it+1 have landed
      __syncthreads();                       // ... for everyone; slot (it-1) % NS is free again
      if (it == 0) SACX_TSTAMP(1);
    }
    if (j < nk) {
      float* st = smem + (j % GEMM_NS) * C::STAGE_FLOATS;
      stage_load<BM, AKM>(st, A, lda, a_vec, m0, M, j * GEMM_BK, K);
      stage_load<BN, BKM>(st + C::A_FLOATS, Bp, ldb, b_vec, n0, N, j * GEMM_BK, K);
    }
    cp_async_commit();
    if (it >= 0) {
      const float* st = smem + (it % GEMM_NS) * C::STAGE_FLOATS;
      stage_math<C, AKM, BKM, BSUM>(st, st, false, kg, ty, tx, a_cur, acc, bsum);
    }
  }
  cp_async_wait<0>();
  __syncthreads();                         // all stages consumed: the ring can be reused for the reduction
  SACX_TSTAMP(2);

  // intra-CTA split-K reduction through shared memory
  float* red = smem;
  float* myred = red + kg * C::RBLK;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int r = AKM ? ((i >> 2) * (BM / 2) + 4 * ty + (i & 3)) : (ty + C::TY * i);
    if (BKM) {
#pragma unroll
      for (int h = 0; h < 2; ++h)
        *reinterpret_cast<float4*>(&myred[r * RS + h * (BN / 2) + 4 * tx]) =
            make_float4(acc[i][h * 4 + 0], acc[i][h * 4 + 1], acc[i][h * 4 + 2], acc[i][h * 4 + 3]);
    } else {
#pragma unroll
      for (int j = 0; j < 8; ++j) myred[r * RS + tx + C::TX * j] = acc[i][j];
    }
    if (BSUM) { if (bias_tile && tx == 0) myred[r * RS + BN] = bsum[i]; }
  }
  __syncthreads();
  SACX_TSTAMP(3);
#pragma unroll
  for (int i = 0; i < C::NV; ++i) {
    const int g = tid + i * 256;
    const int row = g / (BN / 4), c4 = (g % (BN / 4)) * 4;
    float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int q = 0; q < KG; ++q) {
      const float4 p = *reinterpret_cast<const float4*>(&red[q * C::RBLK + row * RS + c4]);
      s.x += p.x; s.y += p.y; s.z += p.z; s.w += p.w;
    }
    epilogue_row4<MODE>(op, ctx, m0 + row, n0 + c4, s, pre, C::NV == 1);
  }
  if (BSUM) {
    if (bias_tile && tid < BM) {
      float s = 0.f;
#pragma unroll
      for (int q = 0; q < KG; ++q) s += red[q * C::RBLK + tid * RS + BN];
      epilogue_bias(op, ctx, m0 + tid, s, bpre);
    }
  }
  __syncthreads();   // smem is reused by the next tile
  SACX_TSTAMP(4);
}

template <class C>
__device__ __forceinline__ void gemm_tile(const Op& op, const EpiCtx& ctx, int tile, float* __restrict__ smem) {
  if (op.epi == EPI_FWD) gemm_tile_impl<C, 0>(op, ctx, tile, smem);
  else if (op.epi == EPI_DACT) gemm_tile_impl<C, 1>(op, ctx, tile, smem);
  else gemm_tile_impl<C, 2>(op, ctx, tile, smem);
}

}  // namespace sacx
