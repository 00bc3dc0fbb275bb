// Row-parallel kernel for the single-agent SAC update (latency path).
//
// The tile-parallel plan (sacx_run_kernel) spreads every layer over all SMs and therefore needs a grid-wide barrier
// after each of the ~16 dependent layers of one update; at batch 256 the barriers, the first L2 round trip of every
// tile and the FFMA K loop add up to ~18K cycles per phase. Here the batch is cut into row blocks of 16 rows (one
// m16 MMA tile) and a GROUP of 8 CTAs owns a row block through the whole forward/backward chain:
//   * every layer's output columns are split 8 ways: CTA `rank` computes the 16 x (N/8) slice with 3xTF32
//     mma.sync.m16n8k8 tensor-core tiles (hi/lo split of both operands, fp32 accumulate: fp32-level accuracy),
//   * slices are exchanged through L2: each CTA stores its slice, the 8 CTAs meet at a group barrier (one L2 atomic
//     per CTA, polled by all eight) and pull the full 16 x N rows back with cp.async,
//   * the narrow heads (policy 2A outputs, critic 1 output, dQ/da) never travel as activations: the producing tile
//     projects its slice onto the head weights and only the 8 partial sums per row are exchanged,
//   * weight slices stream from L2 into a 3-slot shared-memory ring two jobs ahead (they do not depend on data),
//   * the per-row SAC arithmetic (tanh-Gaussian sample/log-prob, Bellman target, loss gradients, head backward) is
//     evaluated redundantly by every CTA of the group from the reduced partials -- cheaper than another barrier.
// Groups are formed in software rather than as hardware thread-block clusters: a cluster of 8 must sit inside one
// GPC, and only 15 such clusters are co-resident on a B200 at this shared-memory footprint (tools/cluster_probe.cu),
// one short of the 16 row blocks of a 256-row batch -- the unbalanced second round cost more than the ~1K cycles a
// software barrier adds over barrier.cluster. Any 128 of the 148 SMs can form 16 groups.
// Only the weight gradients need all rows: dW + Adam (+ Polyak) stay tile-parallel in two grid-wide phases -- 3xTF32 tiles
// with TMA-staged operands (rp_dw_tile_tc), 128-column vector tiles for one-row layers (rp_dw_vec_tile), the FFMA tiles of
// sacx_gemm.cuh as the fallback -- on a grid sized to the widest of them (CTAs past the row groups only work there).
// One update = 4 grid barriers + 7 group barriers instead of 16 grid barriers. Reference semantics: sac/agent.py:195-327, sac/models.py:73-87 (SURVEY section 8 a4-a12).
#pragma once
#include "sacx_kernels.cuh"

namespace sacx {

constexpr int RP_CS = 8;                         // CTAs per group = column slices per layer
constexpr int RP_RB = 16;                        // rows per row block
constexpr int RP_HMAX = 256;                     // widest hidden layer
constexpr int RP_NABUF = 4;                      // full-row activation buffers [16][lda], lda = widest hidden + 4 (== 4 mod 32)
constexpr int RP_NWSLOT = 3;                     // weight slots (forward slice [N/8][K+4] / backward [K][N/8])
constexpr int RP_MAXA = 8;                       // action dimension handled by the row ops
constexpr int RP_MAX_GROUPS = 32;
constexpr int RP_MAX_JOBS = 40, RP_MAX_STEPS = 28, RP_MAX_LOADS = 48, RP_MAX_DW_OPS = 16;

enum RpRowOp : int { RPR_NONE = 0, RPR_GATHER, RPR_PI_HEADS, RPR_TARGET_CRITIC, RPR_RELOAD, RPR_ACTOR_Q, RPR_PI_BWD };
enum RpSrc : int { RPS_ABUF0 = 0, RPS_XSA = 4, RPS_XS2 = 5, RPS_XPI = 6 };
enum RpSlot : int { RPP_PI_T = 0, RPP_PI_A, RPP_Q1, RPP_Q2, RPP_QT1, RPP_QT2, RPP_DA1, RPP_DA2, RPP_N };

struct RpJob {
  int bkm;                 // 0 forward: B(k,n) = W[n0+n][k];  1 backward dA: B(k,n) = W[k][n0+n]
  int a_src;               // RpSrc
  int K, Kp, N;            // reduction length (padded to 8), full output width (slice NS = N / 8)
  int ns_log2;             // log2(NS), NS in {8, 16, 32}
  int act;                 // forward: activation;  backward: activation whose derivative multiplies the result
  int w_ld;                // leading dimension of W in global memory
  int out_ld, aux_ld;
  int proj_J, proj_slot, proj_sj, proj_sn;      // projection of the output slice onto J weight vectors (0: none)
  int tma, map;            // tma = 1: the weight slice arrives by TMA (tensor map `map`, 128B-swizzled tiles) instead of cp.async
  i64 w, bias, out, aux, proj_w;                // arena offsets (-1: unused)
  // pair = 1: a second, independent forward GEMM of the same shape rides in this job (pi(s') / pi(s), Q1 / Q2): its own input
  // rows (a_src2), output, projection slot and -- when w2_off > 0 -- its own weight slice (at slot + w2_off, tensor map map2)
  // and bias (epilogue operand + 32). Each half keeps the single job's k-groups and summation order: same bits.
  int pair, a_src2, proj_slot2, map2, w2_off, pad_p;
  i64 w2, bias2, out2;
};
struct RpLoad { i64 off; int ld, K, abuf, pad; };
struct RpStep { int row_op, job0, njobs, load0, nloads, pad0, pad1, pad2; };

struct RpProgram {
  int n_steps_a, n_steps_c, n_jobs, n_loads;
  int n_row_groups, pad_g;                     // groups that own row blocks (CTAs past 8 x n_row_groups only work in the tile-parallel phases)
  // shared-memory layout (float offsets into the dynamic region)
  int sm_abuf, sm_xbuf, ldx, sm_wslot, sm_red, sm_otile, sm_pw, sm_total;
  int lda, abuf_floats, wslot_floats, gldx;     // gldx: row stride of the batch buffers in the arena
  // geometry / activations
  int O, A, Hq, Hpi, ld_hq, ld_hpi, act_q, act_oq, act_pi, act_opi;
  int ab_q[2], ab_pi, part_stride;             // abuf indices of the delta generators; floats of partial scratch per group
  int part_off[RPP_N];                         // float offset of each partial slot inside a group's scratch: [rank][16][J]
  // arena offsets used by the row ops
  i64 x_sa, x_s2, x_pi, b_r, b_d, b_idx, b_eps1, b_eps2, b_lp2, b_lp, b_y, b_tq[2], b_q[2], b_qa[2], b_dout[2],
      b_loss[2], b_ploss, b_tz, b_se, b_mask, b_headz, b_dhead;
  i64 pi_bL, pi_WL, q_bL[2], q_WL[2], qt_bL[2];
  i64 dq_last[2], dp_last;
  RpStep steps[RP_MAX_STEPS];
  RpJob jobs[RP_MAX_JOBS];
  RpLoad loads[RP_MAX_LOADS];
};

struct RpRows {            // per-row state of the current row block (every CTA of the group holds a copy)
  float r[RP_RB], d[RP_RB], lp2[RP_RB], lp[RP_RB], coef[2][RP_RB];
  float eps1[RP_RB][RP_MAXA], eps2[RP_RB][RP_MAXA], tz[RP_RB][RP_MAXA], se[RP_RB][RP_MAXA], mk[RP_RB][RP_MAXA];
  float hz[RP_RB][2 * RP_MAXA], dh[RP_RB][2 * RP_MAXA];
};

// optional event trace of CTA 0 (profiling aid): (tag, clock64) pairs of the launch's last update
struct RpTrace { unsigned long long* buf; int n, cap; };

// (compiled into libsacx_debug.so only: ~180 trace points per update, each a load + branch in every warp, are not free in a
//  kernel whose every instruction costs latency; tools/phase_profile.py loads the debug library for the event trace)
#ifdef SACX_DEBUG_HOOKS
#define RP_TRACE(tag) do { if (c.tr->buf && threadIdx.x == 0 && c.tr->n < c.tr->cap) { \
  c.tr->buf[2 * c.tr->n] = (unsigned long long)(tag); c.tr->buf[2 * c.tr->n + 1] = clock64(); c.tr->n++; } } while (0)
#else
#define RP_TRACE(tag) do { } while (0)
#endif

struct RpCtx {
  float* base;
  AgentScalars* scal;
  const RunArgs* args;
  const RpProgram* P;
  RpRows* R;
  float* part;            // this group's partial scratch (global)
  unsigned* gbar;         // this group's barrier counter
  int rank, step, row0;
  RpTrace* tr;
  uint64_t* wbar;         // one mbarrier per weight slot (TMA-staged slices)
  const struct RpLaunch* L;   // per-launch constants (push count, stream keys, update counter at launch)
  i64* slots;             // ring slots of the current row block's rows (shared memory)
};

#define RP_SMEM extern __shared__ __align__(1024) float rp_dyn_smem[]; float* const smem_raw = rp_dyn_smem

// ---- shared-memory accessors (explicit state space: the helpers receive offsets, not generic pointers) ---------------
__device__ __forceinline__ uint32_t rp_saddr(const float* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ float rp_lds(uint32_t a) {
  float v;
  asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(a));
  return v;
}

__device__ __forceinline__ void rp_cp_async4(float* smem_dst, const float* gsrc) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(rp_saddr(smem_dst)), "l"(gsrc) : "memory");
}

// ---- TMA-staged weight slices (hidden width 256: NS = 32 columns per CTA) -------------------------------------------------
// One thread issues the whole slice (8 tile loads for a 32 x 256 forward slice, one for a 256 x 32 backward slice) and the
// copy runs behind the current job's math; the cp.async version blocks every thread for the ~2.4K cycles the L2 needs to
// deliver 32 KB to each of the 128 CTAs at once. Tiles are 128B-swizzled (32 floats per row): conflict-free fragment loads
// for the forward orientation, two-way conflicts for the backward one.
__device__ __forceinline__ void rp_mbar_init(uint64_t* b, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"((uint32_t)__cvta_generic_to_shared(b)), "r"(count));
}
__device__ __forceinline__ void rp_mbar_expect_tx(uint64_t* b, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"((uint32_t)__cvta_generic_to_shared(b)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void rp_mbar_wait(uint64_t* b, uint32_t parity) {
  uint32_t done;
  do {
    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                 : "=r"(done) : "r"((uint32_t)__cvta_generic_to_shared(b)), "r"(parity) : "memory");
  } while (!done);
}
__device__ __forceinline__ void rp_tma_load(float* dst, const void* map, uint64_t* bar, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
               ::"r"((uint32_t)__cvta_generic_to_shared(dst)), "l"(reinterpret_cast<uint64_t>(map)),
                 "r"((uint32_t)__cvta_generic_to_shared(bar)), "r"(c0), "r"(c1) : "memory");
}

// ---- 3xTF32 tensor-core arithmetic ------------------------------------------------------------------------------
// x = hi + lo with hi = x rounded to TF32 (half-ulp add, then the low 13 bits cleared); the tensor core ignores the low
// 13 mantissa bits of its inputs, so lo is passed as is (it loses at most 2^-21 |x|)
__device__ __forceinline__ void rp_split(float x, uint32_t& hi, uint32_t& lo) {
  hi = (__float_as_uint(x) + 0x1000u) & 0xffffe000u;
  lo = __float_as_uint(x - __uint_as_float(hi));
}
__device__ __forceinline__ void rp_mma(float (&c)[4], const uint32_t (&a)[4], const uint32_t (&b)[2]) {
  asm volatile("mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b[0]), "r"(b[1]));
}
// the three 3xTF32 terms of A(16x8) . B(8x8) go to separate accumulators: no tensor-core instruction waits on the
// previous one, and the small cross terms are summed before they meet the leading term
__device__ __forceinline__ void rp_mma3(float (&c0)[4], float (&c1)[4], float (&c2)[4], const float (&a)[4], const float (&b)[2]) {
  uint32_t ah[4], al[4], bh[2], bl[2];
#pragma unroll
  for (int i = 0; i < 4; ++i) rp_split(a[i], ah[i], al[i]);
#pragma unroll
  for (int i = 0; i < 2; ++i) rp_split(b[i], bh[i], bl[i]);
  rp_mma(c0, al, bh);
  rp_mma(c1, ah, bl);
  rp_mma(c2, ah, bh);
}

// ---- group barrier: 8 CTAs poll the arrival counter itself -- one L2 hop less than "last arriver publishes a flag" ---------
__device__ __forceinline__ void rp_group_barrier(unsigned* counter, unsigned& epoch) {
  __syncthreads();
  if (threadIdx.x == 0) {
    epoch += RP_CS;
    unsigned old, v;
    asm volatile("atom.add.release.gpu.global.u32 %0, [%1], 1;" : "=r"(old) : "l"(counter) : "memory");
    if (old + 1 != epoch) {
      do {
        asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(counter) : "memory");
      } while ((int)(v - epoch) < 0);
    } else {
      asm volatile("fence.acq_rel.gpu;" ::: "memory");
    }
  }
  __syncthreads();
}

// ---- everything job j needs, global (L2) -> its shared-memory slot, two jobs ahead of its use --------------------------
// slot = [weight slice | epilogue operand (bias[NS] or aux[16][NS]) | projection weights [J][NS]], all by cp.async (one
// commit group per job, committed by the caller). (1-D bulk copies were tried: ~90 cycles of issue per row copy on the
// single TMA queue -- 3.5K cycles for a 32-row slice -- against ~1.4K for 8 cp.async per thread.)
__device__ __forceinline__ void rp_issue_job(const RpJob& jb, float* __restrict__ slot, const RpCtx& c, int slot_idx) {
  const RpProgram& P = *c.P;
  const float* __restrict__ base = c.base;
  const int NS = 1 << jb.ns_log2, n0g = c.rank << jb.ns_log2, tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const float* __restrict__ W = base + jb.w;
  float* eps = slot + P.wslot_floats - 1024;
  float* pws = slot + P.wslot_floats - 512;
  const int J = jb.proj_J, cl = jb.ns_log2 - 2;            // chunks per NS-wide row = NS / 4 = 1 << cl
  const int B = c.args->hp.B;
  const bool sep = jb.pair && jb.w2_off > 0;               // a pair with a second weight slice (and bias) of its own
  if (jb.tma) {
    if (lane == 0) {
      // one 32 x 32 tile (4 KB) per warp: the issue cost (~100 cycles per tile on the TMA queue) is spread over the warps.
      // The slot was last READ with ordinary loads, all complete before the caller's barrier -- the usual consumer-release /
      // producer-acquire pattern of TMA pipelines, no proxy fence (it would also wait for the cp.async copies in flight).
      uint64_t* bar = c.wbar + slot_idx;
      const int slabs = (jb.K + 31) >> 5;                  // K <= 256: at most 8 (a pair with two slices: 2 x slabs <= 8)
      if (warp < (sep ? 2 * slabs : slabs)) {
        const bool h = warp >= slabs;                      // second slice of a pair: tiles at slot + w2_off
        const int wt = h ? warp - slabs : warp;
        const char* map = reinterpret_cast<const char*>(c.args->rp_maps) + (size_t)(h ? jb.map2 : jb.map) * 128;
        float* dst = slot + (h ? jb.w2_off : 0) + wt * 1024;
        rp_mbar_expect_tx(bar, 4096u);
        if (!jb.bkm) rp_tma_load(dst, map, bar, 32 * wt, n0g);
        else rp_tma_load(dst, map, bar, n0g, 32 * wt);
      } else {
        asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"((uint32_t)__cvta_generic_to_shared(bar)) : "memory");
      }
    }
    if (!jb.bkm) {
      if (tid < (1 << cl)) cp_async16(eps + (tid << 2), base + jb.bias + n0g + (tid << 2), 16);
      else if (sep && tid >= 32 && tid < 32 + (1 << cl)) cp_async16(eps + 32 + ((tid - 32) << 2), base + jb.bias2 + n0g + ((tid - 32) << 2), 16);
    } else if (tid < (RP_RB << cl)) {
      const int m = tid >> cl, cc = (tid & ((1 << cl) - 1)) << 2;
      const bool ok = c.row0 + m < B;
      cp_async16(eps + m * NS + cc, ok ? base + jb.aux + (i64)(c.row0 + m) * jb.aux_ld + n0g + cc : base, ok ? 16 : 0);
    }
  } else if (!jb.bkm) {
    const int ldw = jb.Kp + 4;
    for (int h = 0; h <= (int)sep; ++h) {
      const i64 wo = h ? jb.w2 : jb.w;
      const float* __restrict__ Wh = base + wo;
      float* sl = slot + (h ? jb.w2_off : 0);
      const bool vec = ((jb.K & 3) == 0) && ((wo & 3) == 0) && ((jb.w_ld & 3) == 0);
      if (vec) {
        const int cpr = jb.Kp >> 2;            // 16-byte chunks per row (the last one may be zero padding)
        for (int n = warp; n < NS; n += 8) {
          const float* src = Wh + (i64)(n0g + n) * jb.w_ld;
          float* dst = sl + n * ldw;
          for (int ch = lane; ch < cpr; ch += 32) {
            const int k = ch << 2;
            if (k < jb.K) cp_async16(dst + k, src + k, 16);
            else *reinterpret_cast<float4*>(dst + k) = make_float4(0.f, 0.f, 0.f, 0.f);
          }
        }
      } else {
        for (int n = warp; n < NS; n += 8)
          for (int k = lane; k < jb.Kp; k += 32)
            sl[n * ldw + k] = (k < jb.K) ? __ldcg(Wh + (i64)(n0g + n) * jb.w_ld + k) : 0.f;
      }
    }
    if (tid < (1 << cl)) cp_async16(eps + (tid << 2), base + jb.bias + n0g + (tid << 2), 16);
    else if (sep && tid >= 32 && tid < 32 + (1 << cl)) cp_async16(eps + 32 + ((tid - 32) << 2), base + jb.bias2 + n0g + ((tid - 32) << 2), 16);
  } else {
    // [K][NS], 8-column groups XOR-swizzled by the row so that the (k = t, n = g) fragment reads hit 32 banks
    const int sh = 5 - jb.ns_log2;
    const int ch = (tid & ((1 << cl) - 1)) << 2;
    const float* src = W + n0g + ch + (i64)(tid >> cl) * jb.w_ld;
    const i64 sstep = (i64)(256 >> cl) * jb.w_ld;
    for (int k = tid >> cl; k < jb.K; k += 256 >> cl, src += sstep) {
      const int sw = ((k & 3) >> sh) << 3;
      cp_async16(slot + k * NS + (ch ^ sw), src, 16);
    }
    if (tid < (RP_RB << cl)) {          // aux: saved activations of this CTA's own slice, [16][NS]
      const int m = tid >> cl, cc = (tid & ((1 << cl) - 1)) << 2;
      const bool ok = c.row0 + m < B;
      cp_async16(eps + m * NS + cc, ok ? base + jb.aux + (i64)(c.row0 + m) * jb.aux_ld + n0g + cc : base, ok ? 16 : 0);
    }
  }
  if (J > 0) {
    if (jb.proj_sn == 1) {
      const int i = tid - 128;           // threads 128.. : J rows of NS contiguous floats
      if (i >= 0 && i < (J << cl)) {
        const int j = i >> cl, cc = (i & ((1 << cl) - 1)) << 2;
        cp_async16(pws + j * NS + cc, base + jb.proj_w + (i64)j * jb.proj_sj + n0g + cc, 16);
      }
    } else {
      for (int i = tid; i < J * NS; i += 256)
        rp_cp_async4(pws + i, base + jb.proj_w + (i64)(i >> jb.ns_log2) * jb.proj_sj + (i64)(n0g + (i & (NS - 1))) * jb.proj_sn);
    }
  }
}

// full rows of a [B][ld] activation matrix -> activation buffer (rows past the batch are zero)
__device__ __forceinline__ void rp_issue_load(const RpLoad& ld, float* __restrict__ abuf, int lda, const float* __restrict__ base, int row0, int B) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, cpr = ld.K >> 2;
#pragma unroll
  for (int h = 0; h < 2; ++h) {
    const int m = warp + 8 * h;
    const bool ok = row0 + m < B;
    const float* src = base + ld.off + (i64)(row0 + m) * ld.ld;
    for (int ch = lane; ch < cpr; ch += 32) cp_async16(abuf + m * lda + (ch << 2), ok ? src + (ch << 2) : base, ok ? 16 : 0);
  }
}

// ---- one GEMM job: 16 x NS output slice, K reduction split over the warps --------------------------------------------
__device__ __forceinline__ void rp_job_math(const RpJob& jb, uint32_t As, int lda, uint32_t Bs, float* __restrict__ red) {
  const int NS = 1 << jb.ns_log2, ntl = jb.ns_log2 - 3, KG = 8 >> ntl;      // n-tiles per slice = NS/8, K groups = 8/NT
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
  const int nt = warp & ((1 << ntl) - 1), kg = warp >> ntl, n0 = nt << 3;
  const int ksteps = jb.Kp >> 3, per = (ksteps + KG - 1) >> (3 - ntl);
  const int ks0 = kg * per, ks1 = min(ksteps, ks0 + per);
  float c0[4] = {0.f, 0.f, 0.f, 0.f}, c1[4] = {0.f, 0.f, 0.f, 0.f}, c2[4] = {0.f, 0.f, 0.f, 0.f};
  float d0[4] = {0.f, 0.f, 0.f, 0.f}, d1[4] = {0.f, 0.f, 0.f, 0.f}, d2[4] = {0.f, 0.f, 0.f, 0.f};
  const uint32_t a0p = As + 4u * (uint32_t)(g * lda + t), a1p = a0p + 32u * (uint32_t)lda;
  uint32_t bp, bstep, b4;
  if (!jb.bkm) {
    bp = Bs + 4u * (uint32_t)((n0 + g) * (jb.Kp + 4) + t); bstep = 32u; b4 = 16u;
  } else {
    const int sw = (t >> (5 - jb.ns_log2)) << 3;
    bp = Bs + 4u * (uint32_t)(t * NS + ((n0 + g) ^ sw)); bstep = 32u * (uint32_t)NS; b4 = 16u * (uint32_t)NS;
  }
  uint32_t ao = 32u * (uint32_t)ks0, bo = bstep * (uint32_t)ks0;
  int ks = ks0;
  if (jb.tma) {
    // 128B-swizzled tiles (NS = 32). forward: slab (ks >> 2) of [32 rows n][32 floats k], element (n, kk) in 16-byte chunk
    // (kk >> 2) ^ (n & 7); backward: [K rows][32 floats n], element (k, n) in chunk (n >> 2) ^ (k & 7)
    const uint32_t nrow = (uint32_t)(n0 + g);
    if (!jb.bkm) {
      const uint32_t rowb = nrow * 128u + 4u * (uint32_t)t;
      while (ks < ks1) {
        const uint32_t sl = Bs + (uint32_t)(ks >> 2) * 4096u + rowb;
        if ((ks & 3) == 0 && ks + 4 <= ks1) {          // a whole slab: four k-steps at fixed offsets
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const float a[4] = {rp_lds(a0p + ao + 32u * q), rp_lds(a1p + ao + 32u * q), rp_lds(a0p + ao + 32u * q + 16u), rp_lds(a1p + ao + 32u * q + 16u)};
            const float b[2] = {rp_lds(sl + (((uint32_t)(2 * q) ^ (uint32_t)g) << 4)), rp_lds(sl + (((uint32_t)(2 * q + 1) ^ (uint32_t)g) << 4))};
            if (q & 1) rp_mma3(d0, d1, d2, a, b);
            else rp_mma3(c0, c1, c2, a, b);
          }
          ao += 128u; ks += 4;
        } else {
          const uint32_t ch = (uint32_t)(ks & 3) * 2u;
          const float a[4] = {rp_lds(a0p + ao), rp_lds(a1p + ao), rp_lds(a0p + ao + 16u), rp_lds(a1p + ao + 16u)};
          const float b[2] = {rp_lds(sl + ((ch ^ (uint32_t)g) << 4)), rp_lds(sl + (((ch + 1u) ^ (uint32_t)g) << 4))};
          if (ks & 1) rp_mma3(d0, d1, d2, a, b);
          else rp_mma3(c0, c1, c2, a, b);
          ao += 32u; ++ks;
        }
      }
    } else {
      const uint32_t nc = nrow >> 2, w = 4u * (nrow & 3u);
      const uint32_t off0 = (uint32_t)t * 128u + ((nc ^ (uint32_t)t) << 4) + w, off1 = (uint32_t)(t + 4) * 128u + ((nc ^ (uint32_t)(t + 4)) << 4) + w;
      uint32_t kb = Bs + (uint32_t)ks * 1024u;
      for (; ks + 1 < ks1; ks += 2) {
        const float a[4] = {rp_lds(a0p + ao), rp_lds(a1p + ao), rp_lds(a0p + ao + 16u), rp_lds(a1p + ao + 16u)};
        const float b[2] = {rp_lds(kb + off0), rp_lds(kb + off1)};
        const float a2[4] = {rp_lds(a0p + ao + 32u), rp_lds(a1p + ao + 32u), rp_lds(a0p + ao + 48u), rp_lds(a1p + ao + 48u)};
        const float b2[2] = {rp_lds(kb + 1024u + off0), rp_lds(kb + 1024u + off1)};
        rp_mma3(c0, c1, c2, a, b);
        rp_mma3(d0, d1, d2, a2, b2);
        ao += 64u; kb += 2048u;
      }
      if (ks < ks1) {
        const float a[4] = {rp_lds(a0p + ao), rp_lds(a1p + ao), rp_lds(a0p + ao + 16u), rp_lds(a1p + ao + 16u)};
        const float b[2] = {rp_lds(kb + off0), rp_lds(kb + off1)};
        rp_mma3(c0, c1, c2, a, b);
        ++ks;
      }
    }
  }
  for (; ks + 1 < ks1; ks += 2) {
    const float a[4] = {rp_lds(a0p + ao), rp_lds(a1p + ao), rp_lds(a0p + ao + 16u), rp_lds(a1p + ao + 16u)};
    const float b[2] = {rp_lds(bp + bo), rp_lds(bp + bo + b4)};
    const float a2[4] = {rp_lds(a0p + ao + 32u), rp_lds(a1p + ao + 32u), rp_lds(a0p + ao + 48u), rp_lds(a1p + ao + 48u)};
    const float b2[2] = {rp_lds(bp + bo + bstep), rp_lds(bp + bo + bstep + b4)};
    rp_mma3(c0, c1, c2, a, b);
    rp_mma3(d0, d1, d2, a2, b2);
    ao += 64u; bo += 2u * bstep;
  }
  if (ks < ks1) {
    const float a[4] = {rp_lds(a0p + ao), rp_lds(a1p + ao), rp_lds(a0p + ao + 16u), rp_lds(a1p + ao + 16u)};
    const float b[2] = {rp_lds(bp + bo), rp_lds(bp + bo + b4)};
    rp_mma3(c0, c1, c2, a, b);
  }
  const int RS = NS + 8;
  float* r = red + kg * 16 * RS;
  float acc[4];
#pragma unroll
  for (int q = 0; q < 4; ++q) acc[q] = ((c0[q] + d0[q]) + (c1[q] + d1[q])) + (c2[q] + d2[q]);
  *reinterpret_cast<float2*>(r + g * RS + n0 + 2 * t) = make_float2(acc[0], acc[1]);
  *reinterpret_cast<float2*>(r + (g + 8) * RS + n0 + 2 * t) = make_float2(acc[2], acc[3]);
}

__device__ __forceinline__ void rp_job(const RpJob& jb, const RpCtx& c, int wslot_idx) {
  RP_SMEM;
  const RpProgram& P = *c.P;
  const int tid = threadIdx.x, NS = 1 << jb.ns_log2, n0g = c.rank << jb.ns_log2, RS = NS + 8, KG = 64 >> jb.ns_log2;
  const int B = c.args->hp.B;
  const float* Bs = smem_raw + P.sm_wslot + wslot_idx * P.wslot_floats;
  const float* eps = Bs + P.wslot_floats - 1024;
  const float* pws = Bs + P.wslot_floats - 512;
  float* red = smem_raw + P.sm_red;
  const int red_half = KG * 16 * RS;                 // reduction floats of one half of a pair
  RP_TRACE(4500);
#pragma unroll 1
  for (int h = 0; h <= jb.pair; ++h) {               // the halves of a pair one after the other: the single job's registers
    const int src = h ? jb.a_src2 : jb.a_src;
    const float* As;
    int lda;
    if (src < RP_NABUF) { As = smem_raw + P.sm_abuf + src * P.abuf_floats; lda = P.lda; }
    else { As = smem_raw + P.sm_xbuf + (src - RPS_XSA) * RP_RB * P.ldx; lda = P.ldx; }
    rp_job_math(jb, rp_saddr(As), lda, rp_saddr(Bs + (h ? jb.w2_off : 0)), red + h * red_half);
  }
  RP_TRACE(4600);
  __syncthreads();
  RP_TRACE(4650);
  // thread owns outputs (m, n) and (m, n + 1) of the 16 x NS slice (of each half); the NS / 2 lanes of a row sit in one warp
  const int e = tid * 2, m = e >> jb.ns_log2, n = e & (NS - 1);
  // (a rolled loop over the halves on purpose: the kernel lives on instruction fetch, and an unrolled second copy of this
  //  epilogue made every job slower -- DESIGN.md section 4.2, round 5)
  if (e < RP_RB * NS) {               // warp-uniform
#pragma unroll 1
    for (int h = 0; h <= jb.pair; ++h) {
      const float* rh = red + h * red_half;
      float2 s = make_float2(0.f, 0.f);
      for (int q = 0; q < KG; ++q) {
        const float2 p = *reinterpret_cast<const float2*>(rh + (q * 16 + m) * RS + n);
        s.x += p.x; s.y += p.y;
      }
      float2 v;
      if (!jb.bkm) {
        const float2 bb = *reinterpret_cast<const float2*>(eps + (h && jb.w2_off ? 32 : 0) + n);
        v = make_float2(act_fwd(jb.act, s.x + bb.x), act_fwd(jb.act, s.y + bb.y));
      } else {
        const float2 ax = *reinterpret_cast<const float2*>(eps + m * NS + n);
        v = make_float2(s.x * act_dz(jb.act, ax.x), s.y * act_dz(jb.act, ax.y));
      }
      const i64 out = h ? jb.out2 : jb.out;
      if (c.row0 + m < B && out >= 0) *reinterpret_cast<float2*>(c.base + out + (i64)(c.row0 + m) * jb.out_ld + n0g + n) = v;
      const int J = jb.proj_J;
      if (J > 0) {
        // projection of the row's slice onto J weight vectors: butterfly over the row's lanes (fixed order: deterministic);
        // share of CTA `rank` goes to [rank][m][j] of the group's scratch, summed in rank order by every reader.
        // (Both halves of a pair that projects share the weight slice, hence the projection weights.)
        const int lpr = NS >> 1, r = (tid & 31) & (lpr - 1);
        float* dst = c.part + P.part_off[h ? jb.proj_slot2 : jb.proj_slot] + (c.rank * RP_RB + m) * J;
        if (J == 1) {                    // critic heads: one weight vector, one butterfly
          const float2 w = *reinterpret_cast<const float2*>(pws + n);
          float p1 = fmaf(v.x, w.x, v.y * w.y);
          for (int o = lpr >> 1; o > 0; o >>= 1) p1 += __shfl_xor_sync(0xffffffffu, p1, o);
          if (r == 0) dst[0] = p1;
        } else
        for (int j0 = 0; j0 < J; j0 += 8) {
          float p[8];
#pragma unroll
          for (int jj = 0; jj < 8; ++jj) {
            p[jj] = 0.f;
            if (j0 + jj < J) {
              const float2 w = *reinterpret_cast<const float2*>(pws + (j0 + jj) * NS + n);
              p[jj] = fmaf(v.x, w.x, v.y * w.y);
            }
          }
          for (int o = lpr >> 1; o > 0; o >>= 1) {
#pragma unroll
            for (int jj = 0; jj < 8; ++jj) p[jj] += __shfl_xor_sync(0xffffffffu, p[jj], o);
          }
#pragma unroll
          for (int jj = 0; jj < 8; ++jj)
            if (j0 + jj < J && r == ((j0 + jj) & (lpr - 1))) dst[j0 + jj] = p[jj];
        }
      }
    }
  }
}

// the 8 CTAs' shares of element (m, j) of a partial slot: loads first (independent L2 requests; __ldcg is a volatile asm,
// so a sum between two groups of loads would serialise their round trips), summed later in rank order (deterministic)
struct RpParts { float v[RP_CS]; };
__device__ __forceinline__ void rp_load_parts(const RpCtx& c, int slot, int J, int m, int j, RpParts& o) {
  const float* p = c.part + c.P->part_off[slot] + m * J + j;
#pragma unroll
  for (int r = 0; r < RP_CS; ++r) o.v[r] = __ldcg(p + r * RP_RB * J);
}
__device__ __forceinline__ float rp_add_parts(const RpParts& o) {
  float s = 0.f;
#pragma unroll
  for (int r = 0; r < RP_CS; ++r) s += o.v[r];
  return s;
}
__device__ __forceinline__ float rp_sum8(float v) {     // sum over the 8 lanes that share a row
  v += __shfl_xor_sync(0xffffffffu, v, 1);
  v += __shfl_xor_sync(0xffffffffu, v, 2);
  v += __shfl_xor_sync(0xffffffffu, v, 4);
  return v;
}

// ---- row ops --------------------------------------------------------------------------------------------------------
// ring records -> the three input buffers (a2/a3), the update's normals; rank 0 mirrors the batch into the arena.
// Warp 0 turns the 16 rows' logical indices into ring slots (host index stream, or the keyed Feistel bijection) while warps
// 1-7 draw the update's 2 x 16 x A normals (one Philox call per thread); then every thread pulls its share of the 16 packed
// records [s | s2 | a | r | d] -- consecutive threads read consecutive floats of a record -- with all its loads in flight
// before the first is used. Per-launch constants (push count, stream keys, update counter at launch) come from RpLaunch.
struct RpLaunch { i64 pushes, upd0, oldest_slot; unsigned long long rng_seed; unsigned rng_agent, pad; };

// NSTEP: the s2 columns come from the window's last record (slot2), r and d are the folded nr / nd (rp_nstep_fold)
template <int MAXE, bool NSTEP>
__device__ __forceinline__ void rp_gather_rows(const RpCtx& c, const i64* __restrict__ slots, const float* __restrict__ ring,
                                               i64 slot2 = 0, float nr = 0.f, float nd = 0.f) {
  RP_SMEM;
  const RunArgs& a = *c.args;
  const RpProgram& P = *c.P;
  RpRows& R = *c.R;
  const int tid = threadIdx.x, O = P.O, A = P.A, ldx = P.ldx;
  float* xsa = smem_raw + P.sm_xbuf, *xs2 = xsa + RP_RB * ldx, *xpi = xs2 + RP_RB * ldx;
  const bool w0 = c.rank == 0;
  const int W = 2 * O + A + 2, mm = tid >> 4, c0 = tid & 15, row = c.row0 + mm;
  const i64 slot = slots[mm];
  const float* __restrict__ rec = ring + a.ring_s + (slot >= 0 ? slot : 0) * a.ring_rs;      // record = [s | s2 | a | r | d]: ring_s is its first field
  const float* __restrict__ rec2 = NSTEP ? ring + a.ring_s + (slot >= 0 ? slot2 : 0) * a.ring_rs : rec;
  float v[MAXE];
#pragma unroll
  for (int u = 0; u < MAXE; ++u) {
    const int col = c0 + 16 * u;
    if (NSTEP) v[u] = (col < 2 * O + A && slot >= 0) ? __ldcs((col >= O && col < 2 * O ? rec2 : rec) + col) : 0.f;
    else v[u] = (col < W && slot >= 0) ? __ldcs(rec + col) : 0.f;
  }
  // padding columns (finite zeros: they meet zero-padded weights in the K loop)
  for (int col = O + c0; col < ldx; col += 16) {
    if (col >= O + A) xsa[mm * ldx + col] = 0.f;
    xs2[mm * ldx + col] = 0.f; xpi[mm * ldx + col] = 0.f;
  }
  const bool ok = w0 && slot >= 0;
  // the row's arena destinations, formed before the first store: the compiler cannot tell a store through a float pointer
  // from the program table or the context, and reloaded their fields after every store of the scatter
  const i64 grow = (i64)row * P.gldx;
  float* const gsa = c.base + P.x_sa + grow, *const gpi = c.base + P.x_pi + grow, *const gs2 = c.base + P.x_s2 + grow;
  float* const gr = c.base + P.b_r + row, *const gd = c.base + P.b_d + row;
#pragma unroll
  for (int u = 0; u < MAXE; ++u) {
    const int col = c0 + 16 * u;
    if (col < W) {
      const float x = v[u];
      if (col < O) {
        xsa[mm * ldx + col] = x; xpi[mm * ldx + col] = x;
        if (ok) { gsa[col] = x; gpi[col] = x; }
      } else if (col < 2 * O) {
        xs2[mm * ldx + col - O] = x;
        if (ok) gs2[col - O] = x;
      } else if (col < 2 * O + A) {
        xsa[mm * ldx + col - O] = x;                       // action columns sit behind the state in X_sa
        if (ok) gsa[col - O] = x;
      } else if (col == 2 * O + A) {
        const float y = NSTEP ? nr : x;
        R.r[mm] = y;
        if (ok) *gr = y;
      } else {
        const float y = NSTEP ? nd : x;
        R.d[mm] = y;
        if (ok) *gd = y;
      }
    }
  }
}

// n-step fold of the row block (hp.n_step > 1): thread (row mm = tid >> 4, offset i = tid & 15) loads r, d of logical
// j + i, a 16-lane ballot finds the window's end e = m - 1, and every thread of the row gets R, d_eff and the end slot --
// the same threads then gather the row (rp_gather_rows<.., true>), so nothing goes through shared memory. Out of line:
// the one-step gather keeps its code and its registers.
struct RpFold { i64 slot2; float r, d; };
__device__ __noinline__ RpFold rp_nstep_fold(const RpCtx& c, i64 slot) {
  const RunArgs& a = *c.args;
  const RpLaunch& L = *c.L;
  const int i = threadIdx.x & 15, ns = a.hp.n_step;
  const i64 cap = a.ring_capacity, len = L.pushes < cap ? L.pushes : cap;
  i64 j = slot - L.oldest_slot;                      // logical position of the row's first record
  if (j < 0) j += cap;
  i64 si = slot + i;
  if (si >= cap) si -= cap;
  float ri = 0.f, di = 0.f;
  bool stop = false;
  if (slot >= 0 && i < ns && j + i < len) {
    const float* rec = a.ring + si * a.ring_rs;
    ri = __ldcg(rec + a.ring_r);
    di = __ldcg(rec + a.ring_d);
    stop = nstep_stop(di, i, ns, j + i, len);
  }
  const unsigned bits = (__ballot_sync(0xffffffffu, stop) >> (threadIdx.x & 16)) & 0xffffu;
  const int e = bits ? __ffs(bits) - 1 : 0;
  const NstepFold f = nstep_fold(ri, di, e, ns, __ldcg(&c.scal->gamma), 16);
  i64 s2 = slot + e;
  if (s2 >= cap) s2 -= cap;
  return {s2, f.r, f.d};
}

__device__ __noinline__ void rp_gather_nstep(const RpCtx& c, const i64* __restrict__ slots, const float* __restrict__ ring, int W) {
  const RpFold f = rp_nstep_fold(c, slots[threadIdx.x >> 4]);
  if (W <= 64) rp_gather_rows<4, true>(c, slots, ring, f.slot2, f.r, f.d);
  else if (W <= 128) rp_gather_rows<8, true>(c, slots, ring, f.slot2, f.r, f.d);
  else rp_gather_rows<16, true>(c, slots, ring, f.slot2, f.r, f.d);
}

__device__ __noinline__ void rp_gather(const RpCtx& c, const RpLaunch& L, i64* __restrict__ slots) {
  const RunArgs& a = *c.args;
  const Hyper& hp = a.hp;
  const RpProgram& P = *c.P;
  RpRows& R = *c.R;
  const int tid = threadIdx.x, O = P.O, A = P.A, B = hp.B;
  const float* __restrict__ ring = a.ring;
  const i64 cap = a.ring_capacity;
  const bool w0 = c.rank == 0;
  const unsigned long long upd = (unsigned long long)(L.upd0 + c.step);
  if (tid < RP_RB) {
    const int row = c.row0 + tid;
    i64 slot = -1;
    if (row < B) {
      const i64 n = L.pushes < cap ? L.pushes : cap;
      i64 j;
      if (a.idx_ext) j = a.idx_ext[(i64)c.step * hp.B + row];
      else j = (i64)feistel_index((unsigned long long)(hp.row0_global + row), (unsigned long long)n, L.rng_seed, upd, L.rng_agent);
      slot = L.oldest_slot + j;                      // slot of the oldest survivor (computed once per launch) + logical position
      if (slot >= cap) slot -= cap;                  // both < cap: one conditional subtraction replaces the 64-bit modulo
      if (w0) reinterpret_cast<i64*>(c.base + P.b_idx)[row] = j;
    }
    slots[tid] = slot;
  } else if (tid >= 32) {
    // normals: element i = (which, row of the block, action dim < A) -- 2 x 16 x A draws over 224 threads: ONE round up to A = 7
    // (enumerating all RP_MAXA dims cost every update a second ~3.5 K-cycle Philox + Box-Muller round for 32 of the threads).
    // Columns A.. of the eps rows are never read.
    const int per = RP_RB * A;
    for (int i = tid - 32; i < 2 * per; i += 224) {
      const int which = i >= per ? 1 : 0, r = i - which * per, mm = r / A, j = r - mm * A, row = c.row0 + mm;
      float e = 0.f;
      if (row < B) {
        const float* ext = which ? a.eps2_ext : a.eps1_ext;
        if (ext) e = ext[((i64)c.step * hp.B + row) * A + j];
        else e = philox_normal(L.rng_seed, upd, 1 + which, (uint32_t)(hp.row0_global + row), (uint32_t)j, L.rng_agent);
        if (w0) c.base[(which ? P.b_eps2 : P.b_eps1) + (i64)row * A + j] = e;
      }
      if (which) R.eps2[mm][j] = e; else R.eps1[mm][j] = e;
    }
  }
  RP_TRACE(2100);
  __syncthreads();
  // the 16 records: 16 threads per record, thread (mm, c0) takes columns c0, c0 + 16, ... of record mm (W = 2O + A + 2 <= 256
  // -> at most 16 per thread; 4 at BipedalWalker shape); all loads of a thread are in flight before the first is used. The
  // body is instantiated for 4 / 8 / 16 columns per thread: with one 16-column body every update walked twelve predicated-off
  // copies of the scatter at BipedalWalker shape, all instruction-cache misses (`no_instruction` at this line in the ncu source view)
  const int W = 2 * O + A + 2;
  if (hp.n_step > 1) rp_gather_nstep(c, slots, ring, W);
  else if (W <= 64) rp_gather_rows<4, false>(c, slots, ring);
  else if (W <= 128) rp_gather_rows<8, false>(c, slots, ring);
  else rp_gather_rows<16, false>(c, slots, ring);
  RP_TRACE(2103);
  __syncthreads();
}

// policy heads of pi(s') and pi(s) from the reduced partials: rsample, tanh squash, log-prob (models.py:73-87)
__device__ __noinline__ void rp_pi_heads(const RpCtx& c) {
  RP_SMEM;
  const Hyper& hp = c.args->hp;
  const RpProgram& P = *c.P;
  RpRows& R = *c.R;
  const int tid = threadIdx.x, O = P.O, A = P.A, J = 2 * A, ldx = P.ldx, B = hp.B;
  float* xs2 = smem_raw + P.sm_xbuf + RP_RB * ldx, *xpi = xs2 + RP_RB * ldx;
  const bool w0 = c.rank == 0;
  // warps 0-3: target head (which = 0); warps 4-7: actor head (which = 1); 8 lanes per row
  const int which = tid >> 7, t = tid & 127, mm = t >> 3, j = t & 7, row = c.row0 + mm;
  const bool ok = row < B, act_lane = j < A;
  const int slot = which ? RPP_PI_A : RPP_PI_T;
  float lp = 0.f;
  bool bad = false;
  if (act_lane) {
    RpParts pm, pl;
    rp_load_parts(c, slot, J, mm, j, pm);
    rp_load_parts(c, slot, J, mm, A + j, pl);
    const float bm = __ldcg(c.base + P.pi_bL + j), bl = __ldcg(c.base + P.pi_bL + A + j);
    const float zm = rp_add_parts(pm) + bm;
    const float zl = rp_add_parts(pl) + bl;
    const float e = which ? R.eps2[mm][j] : R.eps1[mm][j];
    const SacSample s = sac_rsample(act_fwd(P.act_opi, zm), act_fwd(P.act_opi, zl), e, hp.log_std_min, hp.log_std_max);
    const float av = s.tz * hp.action_scale;
    lp = s.lp;
    bad = ok && s.bad;
    if (!which) {
      xs2[mm * ldx + O + j] = ok ? av : 0.f;
      if (w0 && ok) c.base[P.x_s2 + (i64)row * P.gldx + O + j] = av;
    } else {
      xpi[mm * ldx + O + j] = ok ? av : 0.f;
      if (w0 && ok) {
        c.base[P.x_pi + (i64)row * P.gldx + O + j] = av;
        c.base[P.b_tz + (i64)row * A + j] = s.tz;
        c.base[P.b_se + (i64)row * A + j] = s.sd * e;
        c.base[P.b_mask + (i64)row * A + j] = s.in_clamp ? 1.f : 0.f;
        c.base[P.b_headz + (i64)row * J + j] = zm;
        c.base[P.b_headz + (i64)row * J + A + j] = zl;
      }
    }
  }
  lp = rp_sum8(lp);
  if (j == 0) {
    if (!which) { R.lp2[mm] = lp; if (w0 && ok) c.base[P.b_lp2 + row] = lp; }
    else if (w0 && ok) c.base[P.b_lp + row] = lp;
  }
  if (bad && w0) atomicOr(&c.scal->nonfinite, 1);
  __syncthreads();
}

// in-place delta of the critics' last hidden layer: abuf[m][k] <- coef[m] * W_L[k] * act'(h[m][k]).
// wl[cc]: this thread's float4 of W_L (every iteration of a thread touches the same 4 columns: 256 % (H/4) == 0)
__device__ __forceinline__ void rp_delta_critics(const RpCtx& c, const float4 (&wl)[2], bool store) {
  RP_SMEM;
  const RpProgram& P = *c.P;
  const RpRows& R = *c.R;
  const int tid = threadIdx.x, H = P.Hq, NS = H / RP_CS, n0g = c.rank * NS, B = c.args->hp.B;
  const int cpr = H >> 2, k = (tid % cpr) << 2, m0 = tid / cpr, mstep = 256 / cpr;
  const bool mine = store && k >= n0g && k < n0g + NS;
  // loop operands in registers before the first store (see rp_gather_rows): the rows then cost shared-memory round trips only
  const int lda = P.lda, act = P.act_q, ld = P.ld_hq, nrows = min(RP_RB, B - c.row0);
#pragma unroll
  for (int cc = 0; cc < 2; ++cc) {
    float* ab = smem_raw + P.sm_abuf + P.ab_q[cc] * P.abuf_floats;
    float* const dq = c.base + P.dq_last[cc] + (i64)c.row0 * ld + k;
    const float* const coef = R.coef[cc];
    const float4 w = wl[cc];
    for (int mm = m0; mm < RP_RB; mm += mstep) {
      float4* p = reinterpret_cast<float4*>(ab + mm * lda + k);
      const float4 dv = sac_delta(coef[mm], w, *p, act);
      *p = dv;
      if (mine && mm < nrows) *reinterpret_cast<float4*>(dq + (i64)mm * ld) = dv;
    }
    RP_TRACE(2910 + cc);
  }
  __syncthreads();
}
__device__ __forceinline__ void rp_load_wl(const RpCtx& c, float4 (&wl)[2]) {
  const int cpr = c.P->Hq >> 2, k = (threadIdx.x % cpr) << 2;
#pragma unroll
  for (int cc = 0; cc < 2; ++cc) wl[cc] = __ldcg(reinterpret_cast<const float4*>(c.base + c.P->q_WL[cc] + k));
}

// soft Bellman target (agent.py:195-211) and the critics' loss gradient (agent.py:213-236) for the row block.
// WEIGHTED: per-row importance weights of prioritized replay (RunArgs::w_ext); the uniform instantiation has no weight load.
template <bool WEIGHTED>
__device__ __noinline__ void rp_target_critic(const RpCtx& c) {
  const Hyper& hp = c.args->hp;
  const RpProgram& P = *c.P;
  RpRows& R = *c.R;
  const int tid = threadIdx.x, B = hp.B;
  float4 wl[2];
  rp_load_wl(c, wl);
  RP_TRACE(2901);
  if (tid < RP_RB) {
    const int mm = tid, row = c.row0 + mm;
    const bool ok = row < B, w0 = c.rank == 0;
    RpParts pt[2], pq[2];
    rp_load_parts(c, RPP_QT1, 1, mm, 0, pt[0]); rp_load_parts(c, RPP_QT2, 1, mm, 0, pt[1]);
    rp_load_parts(c, RPP_Q1, 1, mm, 0, pq[0]); rp_load_parts(c, RPP_Q2, 1, mm, 0, pq[1]);
    const float alpha = __ldcg(&c.scal->alpha_f32);
    const float bt[2] = {__ldcg(c.base + P.qt_bL[0]), __ldcg(c.base + P.qt_bL[1])};
    const float bq[2] = {__ldcg(c.base + P.q_bL[0]), __ldcg(c.base + P.q_bL[1])};
    const float st[2] = {rp_add_parts(pt[0]), rp_add_parts(pt[1])};
    const float sq[2] = {rp_add_parts(pq[0]), rp_add_parts(pq[1])};
    const float tq[2] = {act_fwd(P.act_oq, st[0] + bt[0]), act_fwd(P.act_oq, st[1] + bt[1])};
    const float y = sac_target(R.r[mm], R.d[mm], __ldcg(&c.scal->gamma), alpha, tq[0], tq[1], R.lp2[mm]);
    const float wr = (WEIGHTED && ok) ? __ldcg(c.args->w_ext + row) : 1.f;
    if (w0 && ok) { c.base[P.b_y + row] = y; c.base[P.b_tq[0] + row] = tq[0]; c.base[P.b_tq[1] + row] = tq[1]; }
#pragma unroll
    for (int cc = 0; cc < 2; ++cc) {
      const SacCriticRow cr = sac_critic_row(P.act_oq, sq[cc] + bq[cc], y, wr, hp.B_global);
      R.coef[cc][mm] = ok ? cr.dout : 0.f;
      if (w0 && ok) { c.base[P.b_q[cc] + row] = cr.q; c.base[P.b_dout[cc] + (i64)row * 4] = cr.dout; c.base[P.b_loss[cc] + row] = cr.loss; }
    }
  }
  RP_TRACE(2902);
  __syncthreads();
  RP_TRACE(2903);
  rp_delta_critics(c, wl, true);
}

// phase C entry: the row block's (s, a~pi) rows and the saved head quantities come back from the arena
// (instantiated for 2 / 4 / 9 columns per lane: see rp_gather_rows)
template <int MAXC>
__device__ __forceinline__ void rp_reload_impl(const RpCtx& c) {
  RP_SMEM;
  const RpProgram& P = *c.P;
  RpRows& R = *c.R;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, O = P.O, A = P.A, ldx = P.ldx, B = c.args->hp.B;
  float* xpi = smem_raw + P.sm_xbuf + 2 * RP_RB * ldx;
  // warp w: rows 2w, 2w+1 of x_pi; loads first
  float v[2][MAXC];
#pragma unroll
  for (int h = 0; h < 2; ++h) {
    const int row = c.row0 + 2 * warp + h;
#pragma unroll
    for (int u = 0; u < MAXC; ++u) {
      const int col = lane + 32 * u;
      v[h][u] = (col < O + A && row < B) ? __ldcg(c.base + P.x_pi + (i64)row * P.gldx + col) : 0.f;
    }
  }
  float tz = 0.f, se = 0.f, mk = 0.f, hz0 = 0.f, hz1 = 0.f, lpv = 0.f;
  const int mm = tid >> 3, j = tid & 7;
  if (tid < RP_RB * RP_MAXA) {
    const int row = c.row0 + mm;
    if (row < B && j < A) {
      tz = __ldcg(c.base + P.b_tz + (i64)row * A + j);
      se = __ldcg(c.base + P.b_se + (i64)row * A + j);
      mk = __ldcg(c.base + P.b_mask + (i64)row * A + j);
      hz0 = __ldcg(c.base + P.b_headz + (i64)row * 2 * A + j);
      hz1 = __ldcg(c.base + P.b_headz + (i64)row * 2 * A + A + j);
    }
  } else if (tid < 128 + RP_RB) {
    const int row = c.row0 + tid - 128;
    if (row < B) lpv = __ldcg(c.base + P.b_lp + row);
  }
#pragma unroll
  for (int h = 0; h < 2; ++h)
#pragma unroll
    for (int u = 0; u < MAXC; ++u) {
      const int col = lane + 32 * u;
      if (col < ldx) xpi[(2 * warp + h) * ldx + col] = v[h][u];
    }
  if (tid < RP_RB * RP_MAXA) {
    R.tz[mm][j] = tz; R.se[mm][j] = se; R.mk[mm][j] = mk;
    if (j < A) { R.hz[mm][j] = hz0; R.hz[mm][A + j] = hz1; }
  } else if (tid < 128 + RP_RB) {
    R.lp[tid - 128] = lpv;
  }
  __syncthreads();
}
__device__ __noinline__ void rp_reload(const RpCtx& c) {
  const int ldx = c.P->ldx;               // columns per lane = ceil(ldx / 32), ldx <= 260
  if (ldx <= 64) rp_reload_impl<2>(c);
  else if (ldx <= 128) rp_reload_impl<4>(c);
  else rp_reload_impl<9>(c);
}

// critics on (s, a~pi): min, policy loss rows, routed dQ (agent.py:238-260)
__device__ __noinline__ void rp_actor_q(const RpCtx& c) {
  const Hyper& hp = c.args->hp;
  const RpProgram& P = *c.P;
  RpRows& R = *c.R;
  const int tid = threadIdx.x, B = hp.B;
  float4 wl[2];
  rp_load_wl(c, wl);
  if (tid < RP_RB) {
    const int mm = tid, row = c.row0 + mm;
    const bool ok = row < B, w0 = c.rank == 0;
    RpParts pq[2];
    rp_load_parts(c, RPP_Q1, 1, mm, 0, pq[0]); rp_load_parts(c, RPP_Q2, 1, mm, 0, pq[1]);
    const float alpha = __ldcg(&c.scal->alpha_f32);
    const float bq[2] = {__ldcg(c.base + P.q_bL[0]), __ldcg(c.base + P.q_bL[1])};
    const float sq[2] = {rp_add_parts(pq[0]), rp_add_parts(pq[1])};
    const float z[2] = {sq[0] + bq[0], sq[1] + bq[1]};
    const float q[2] = {act_fwd(P.act_oq, z[0]), act_fwd(P.act_oq, z[1])};
    const SacRoute g = sac_actor_route(P.act_oq, z[0], q[0], z[1], q[1], hp.B_global);
    R.coef[0][mm] = ok ? g.c1 : 0.f;
    R.coef[1][mm] = ok ? g.c2 : 0.f;
    if (w0 && ok) {
      c.base[P.b_qa[0] + row] = q[0]; c.base[P.b_qa[1] + row] = q[1];
      c.base[P.b_ploss + row] = sac_policy_loss_row(alpha, R.lp[mm], q[0], q[1]);
    }
  }
  __syncthreads();
  rp_delta_critics(c, wl, false);
}

// dQ/da from the layer-0 partials, closed-form head backward (SURVEY a8), delta of the policy's last hidden layer
// (instantiated for 2A <= 4 / 8 / 16 head columns: see rp_gather_rows)
template <int JM>
__device__ __forceinline__ void rp_pi_bwd_impl(const RpCtx& c) {
  RP_SMEM;
  const Hyper& hp = c.args->hp;
  const RpProgram& P = *c.P;
  RpRows& R = *c.R;
  const int tid = threadIdx.x, A = P.A, J = 2 * A, B = hp.B;
  const int H = P.Hpi, NS = H / RP_CS, n0g = c.rank * NS, cpr = H >> 2;
  const int k = (tid % cpr) << 2, m0 = tid / cpr, mstep = 256 / cpr;
  // this thread's 4 columns of the policy's output layer W_L [2A][H], in flight while the head backward runs
  float4 wl[JM];
#pragma unroll
  for (int j = 0; j < JM; ++j)
    wl[j] = (j < J) ? __ldcg(reinterpret_cast<const float4*>(c.base + P.pi_WL + (i64)j * H + k)) : make_float4(0.f, 0.f, 0.f, 0.f);
  if (tid < RP_RB * RP_MAXA) {
    const int mm = tid >> 3, j = tid & 7, row = c.row0 + mm;
    if (j < A) {
      const bool ok = row < B;
      RpParts d1, d2;
      rp_load_parts(c, RPP_DA1, A, mm, j, d1); rp_load_parts(c, RPP_DA2, A, mm, j, d2);
      const float alpha = __ldcg(&c.scal->alpha_f32);
      const float da = rp_add_parts(d1) + rp_add_parts(d2);
      const SacHeadGrad g = sac_head_bwd(P.act_opi, R.tz[mm][j], R.se[mm][j], R.mk[mm][j], da, alpha / (float)hp.B_global,
                                         hp.action_scale, R.hz[mm][j], R.hz[mm][A + j]);
      const float dmu = ok ? g.dmu : 0.f, dls = ok ? g.dls : 0.f;
      R.dh[mm][j] = dmu; R.dh[mm][A + j] = dls;
      if (c.rank == 0 && ok) { c.base[P.b_dhead + (i64)row * J + j] = dmu; c.base[P.b_dhead + (i64)row * J + A + j] = dls; }
    }
  }
  __syncthreads();
  float* ab = smem_raw + P.sm_abuf + P.ab_pi * P.abuf_floats;
  const bool mine = k >= n0g && k < n0g + NS;
  // loop operands in registers before the first store (see rp_gather_rows)
  const int lda = P.lda, act = P.act_pi, ld = P.ld_hpi, nrows = min(RP_RB, B - c.row0);
  float* const dp = c.base + P.dp_last + (i64)c.row0 * ld + k;
  for (int mm = m0; mm < RP_RB; mm += mstep) {
    float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int j = 0; j < JM; ++j) {
      if (j < J) {
        const float gj = R.dh[mm][j];
        s.x = fmaf(gj, wl[j].x, s.x); s.y = fmaf(gj, wl[j].y, s.y); s.z = fmaf(gj, wl[j].z, s.z); s.w = fmaf(gj, wl[j].w, s.w);
      }
    }
    float4* p = reinterpret_cast<float4*>(ab + mm * lda + k);
    const float4 dv = sac_dact(s, *p, act);
    *p = dv;
    if (mine && mm < nrows) *reinterpret_cast<float4*>(dp + (i64)mm * ld) = dv;
  }
  __syncthreads();
}
__device__ __noinline__ void rp_pi_bwd(const RpCtx& c) {
  const int J = 2 * c.P->A;
  if (J <= 4) rp_pi_bwd_impl<4>(c);
  else if (J <= 8) rp_pi_bwd_impl<8>(c);
  else rp_pi_bwd_impl<2 * RP_MAXA>(c);
}

// ---- weight-gradient tile on the tensor cores (phases B and D) ------------------------------------------------------------
// dW[32 x 32] = dy^T x over the whole batch (K = batch <= RP_DW_MAXK rows) with the same 3xTF32 m16n8k8 arithmetic as the
// forward / backward jobs. What bounds a dW tile here is not arithmetic but getting 2 x K x 128 B of operands from L2 into the SM:
// the FFMA tile of sacx_gemm.cuh (and a first tensor-core version of this one) staged them with 16-byte cp.async copies, which
// this SM issues at ~14 B/clk -- 9-10 K of a tile's 14 K cycles went to the copies. Here ONE thread asks the TMA unit for the
// operands, a [64 rows x 32 floats] box of dy and of x per 64-row chunk (tensor maps built at engine creation, sacx.cu:
// engine_setup_rp_tma; 128B swizzle; columns past M / N and rows past the batch arrive as zeros), one mbarrier per chunk.
// Both operands are batch-major in global memory -- dy [batch][out], x [batch][in] -- and stay that way in shared memory; the
// tile's 32 output rows / columns are assigned to MMA fragment positions through a permutation chosen so that, under the
// swizzle, every fragment load touches 32 distinct banks. Warp w owns k-step w of every chunk (8 MMA tiles x 3 terms per
// chunk), the eight warps' partial tiles meet in shared memory, and the epilogue is the FFMA tile's (gradient store / Adam /
// Polyak on the tile itself); its operands (p, m, v, target) travel into shared memory by cp.async while the chunks load --
// each thread copies exactly the four float4 it will consume. Bias gradient = column sums of dy, taken from the staged chunks.
constexpr int RP_DW_MAXK = 512, RP_DW_CHUNK = 64, RP_DW_BOX = RP_DW_CHUNK * 32, RP_DW_NBAR = RP_DW_MAXK / RP_DW_CHUNK;
constexpr int RP_DW_STAGE = 2 * RP_DW_MAXK * 32 + 4 * 1024;        // floats: dy boxes | x boxes | p, m, v, target tiles
constexpr int RP_DW_SMEM = ((WSM_FLOATS + 255) & ~255) + RP_DW_STAGE;
__device__ __forceinline__ bool rp_dw_tc_ok(const Op& op, const void* maps) {
  return maps != nullptr && op.epi == EPI_DW && op.i[2] > 0 && op.i[3] > 0 && op.K <= RP_DW_MAXK && !(op.flags & DW_ATOMIC) && op.i[0] <= 1;
}
// swizzled position of element (k, col) of a [64][32] box: the 16-byte piece index is XORed with the row's low three bits
__device__ __forceinline__ int rp_dw_sw(int k, int col) { return k * 32 + ((((col >> 2) ^ k) & 7) << 2) + (col & 3); }

__device__ __noinline__ void rp_dw_tile_tc(const Op& op, const EpiCtx& ctx, int tile, float* __restrict__ stage, const void* maps,
                                           uint64_t* bars, unsigned& parity) {
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, g = lane >> 2, t = lane & 3;
  const int M = op.M, N = op.N, K = op.K;
  const int tm = tile / op.tiles_n, tn = tile % op.tiles_n, m0 = tm * 32, n0 = tn * 32;
  float* base = ctx.base;
  float* As = stage;                                           // [chunk][64][32], swizzled
  float* Bs = stage + RP_DW_MAXK * 32;
  float* Es = stage + 2 * RP_DW_MAXK * 32;                     // [4][32][32]: p, m, v, target of this tile
  const bool bias_tile = (tn == 0) && (op.pb >= 0);
  const int nchunks = (K + RP_DW_CHUNK - 1) / RP_DW_CHUNK;
  if (tid == 0) {
    // the staging area was last written / read with ordinary accesses (previous tile's reduction, the row-parallel phase), all
    // complete before the barrier in front of this tile: order them before the TMA unit's writes
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    const char* ma = reinterpret_cast<const char*>(maps) + (size_t)(op.i[2] - 1) * 128;
    const char* mb = reinterpret_cast<const char*>(maps) + (size_t)(op.i[3] - 1) * 128;
    for (int c = 0; c < nchunks; ++c) {
      rp_mbar_expect_tx(bars + c, 2u * RP_DW_BOX * 4u);
      rp_tma_load(As + c * RP_DW_BOX, ma, bars + c, m0, c * RP_DW_CHUNK);
      rp_tma_load(Bs + c * RP_DW_BOX, mb, bars + c, n0, c * RP_DW_CHUNK);
    }
  }
  // epilogue operands: thread (row, c4) copies its own four float4
  const int erow = tid >> 3, ec4 = (tid & 7) << 2;
  const bool adam = (op.flags & DW_ADAM) != 0, polyak = (op.flags & DW_POLYAK) != 0;
  const bool evec = adam && (m0 + erow < M) && epi_vec_ok(op, n0 + ec4);
  if (evec) {
    const i64 e = (i64)(m0 + erow) * N + n0 + ec4;
    float* dst = Es + erow * 32 + ec4;
    cp_async16(dst, base + op.p + e, 16);
    cp_async16(dst + 1024, base + op.pm + e, 16);
    cp_async16(dst + 2048, base + op.pv + e, 16);
    if (polyak) cp_async16(dst + 3072, base + op.pt + e, 16);
  }
  cp_async_commit();
  float ss = 0.f, bc = 0.f, tau = 0.f, omt = 0.f;
  if (adam) {
    ss = __ldcg(&ctx.scal->adam_step_size[op.opt]);
    bc = __ldcg(&ctx.scal->adam_bc2_sqrt[op.opt]);
    if (polyak) { tau = __ldcg(&ctx.scal->tau); omt = __ldcg(&ctx.scal->one_minus_tau); }
  }
  float bpre[8] = {0.f, 0.f, 0.f, 0.f, ss, bc, tau, omt};
  if (bias_tile && adam && tid < 32 && m0 + tid < M) {
    bpre[0] = __ldcg(base + op.pb + m0 + tid);
    bpre[1] = __ldcg(base + op.pbm + m0 + tid);
    bpre[2] = __ldcg(base + op.pbv + m0 + tid);
    if (polyak) bpre[3] = __ldcg(base + op.pbt + m0 + tid);
  }
  float acc[2][4][4], small[2][4][4];
#pragma unroll
  for (int i = 0; i < 2; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j)
#pragma unroll
      for (int q = 0; q < 4; ++q) { acc[i][j][q] = 0.f; small[i][j][q] = 0.f; }
  float bsum = 0.f;                                            // (warp, lane): this warp's k rows of dy column m0 + lane
  // fragment position -> tile row / column. A rows: MMA block i, row g + 8h <-> tile row 16 (g >> 2) + 8 i + 4 h + (g & 3);
  // B / C columns: block j, column cn <-> tile column 16 (cn >> 2) + 4 j + (cn & 3). Under the swizzle a fragment load of 32 lanes
  // (g, t) then reads piece ((4 (g >> 2) + const) ^ t) at word g & 3: 32 distinct banks.
  const int arow = 16 * (g >> 2) + (g & 3), kb = warp * 8;
  for (int c = 0; c < nchunks; ++c) {
    rp_mbar_wait(bars + c, (parity >> c) & 1u);
    if (c * RP_DW_CHUNK + kb < K) {
      const float* a = As + c * RP_DW_BOX;
      const float* b = Bs + c * RP_DW_BOX;
      uint32_t ah[2][4], al[2][4];
#pragma unroll
      for (int i = 0; i < 2; ++i) {
        rp_split(a[rp_dw_sw(kb + t, arow + 8 * i)], ah[i][0], al[i][0]);
        rp_split(a[rp_dw_sw(kb + t, arow + 8 * i + 4)], ah[i][1], al[i][1]);
        rp_split(a[rp_dw_sw(kb + t + 4, arow + 8 * i)], ah[i][2], al[i][2]);
        rp_split(a[rp_dw_sw(kb + t + 4, arow + 8 * i + 4)], ah[i][3], al[i][3]);
      }
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        uint32_t bh[2], bl[2];
        rp_split(b[rp_dw_sw(kb + t, arow + 4 * j)], bh[0], bl[0]);
        rp_split(b[rp_dw_sw(kb + t + 4, arow + 4 * j)], bh[1], bl[1]);
#pragma unroll
        for (int i = 0; i < 2; ++i) {
          rp_mma(small[i][j], al[i], bh);
          rp_mma(small[i][j], ah[i], bl);
          rp_mma(acc[i][j], ah[i], bh);
        }
      }
      if (bias_tile) {
#pragma unroll
        for (int k = 0; k < 8; ++k) bsum += a[rp_dw_sw(kb + k, lane)];
      }
    }
  }
  parity ^= (1u << nchunks) - 1u;
  __syncthreads();                                             // all chunks consumed: the dy boxes become the reduction buffer
  float* red = stage;                                          // [warp][32][33] (+ [warp][32] bias partials behind them)
  float* bred = stage + 8 * 32 * 33;
#pragma unroll
  for (int i = 0; i < 2; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j)
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const int row = arow + 8 * i + 4 * (q >> 1), cn = 2 * t + (q & 1), col = 16 * (cn >> 2) + 4 * j + (cn & 3);
        red[(warp * 32 + row) * 33 + col] = acc[i][j][q] + small[i][j][q];
      }
  if (bias_tile) bred[warp * 32 + lane] = bsum;
  cp_async_wait<0>();                                          // this thread's epilogue operands
  __syncthreads();
  {
    float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int w = 0; w < 8; ++w) {
      const float* p = red + (w * 32 + erow) * 33 + ec4;
      s.x += p[0]; s.y += p[1]; s.z += p[2]; s.w += p[3];
    }
    EpiPre pre;
    pre.valid = evec;
    if (evec) {
      const float* src = Es + erow * 32 + ec4;
      pre.a = *reinterpret_cast<const float4*>(src);
      pre.b = *reinterpret_cast<const float4*>(src + 1024);
      pre.c = *reinterpret_cast<const float4*>(src + 2048);
      if (polyak) pre.d = *reinterpret_cast<const float4*>(src + 3072);
      pre.ss = ss; pre.bc = bc; pre.tau = tau; pre.omt = omt;
    } else if (!adam) {
      pre.valid = (m0 + erow < M) && epi_vec_ok(op, n0 + ec4);          // gradient store only: nothing to prefetch
    }
    epilogue_row4<2>(op, ctx, m0 + erow, n0 + ec4, s, pre, true);
  }
  if (bias_tile && tid < 32) {
    float s = 0.f;
#pragma unroll
    for (int w = 0; w < 8; ++w) s += bred[w * 32 + tid];
    epilogue_bias(op, ctx, m0 + tid, s, bpre);
  }
  __syncthreads();                                             // the staging area is reused by the next tile
}

// ---- weight gradient of a one-row output layer (the critics' heads: dW_L[n] = sum_k dout[k] h[k][n]) --------------------------
// As 32 x 32 tiles this layer was eight tiles per critic with one valid row each -- sixteen more tiles than the 128-CTA grid
// has CTAs, i.e. a second wave for the whole phase (every tile costs ~10 K cycles whatever it computes: operand delivery).
// Here ONE tile covers 128 columns: the x boxes [64 rows x 32 columns] of four column blocks arrive by TMA (same tensor map as
// the square tiles), thread (n, half) runs down half of the batch for column n, the halves meet in shared memory, and the
// Adam / Polyak epilogue is the square tiles'. Two tiles per critic; with the grid sized to the phase (148 tiles on 148 CTAs at
// BipedalWalker shape) the critics' dW phase is one wave.
constexpr int RP_DWV_COLS = 128, RP_DWV_MAXK = 256;
__device__ __noinline__ void rp_dw_vec_tile(const Op& op, const EpiCtx& ctx, int tile, float* __restrict__ stage, const void* maps,
                                            uint64_t* bars, unsigned& parity) {
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int N = op.N, K = op.K, n0 = tile * RP_DWV_COLS;
  float* base = ctx.base;
  const int nchunks = (K + RP_DW_CHUNK - 1) / RP_DW_CHUNK;          // <= 4
  float* xs = stage;                                                // [col block q][chunk c][64][32], swizzled
  float* dsm = stage + 4 * RP_DWV_MAXK * 32;                        // dout[k], then the two halves' partial sums
  float* red = dsm + RP_DWV_MAXK;
  if (tid == 0) {
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    for (int c = 0; c < nchunks; ++c) rp_mbar_expect_tx(bars + c, 4u * RP_DW_BOX * 4u);      // four column blocks per chunk
  }
  if (lane == 0) {
    const char* mb = reinterpret_cast<const char*>(maps) + (size_t)(op.i[3] - 1) * 128;
    if (tid != 0) asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    for (int b = warp; b < 4 * nchunks; b += 8) {                    // box b = (chunk, column block): chunk-major, so chunk 0 is complete first
      const int c = b >> 2, q = b & 3;
      rp_tma_load(xs + (q * nchunks + c) * RP_DW_BOX, mb, bars + c, n0 + 32 * q, c * RP_DW_CHUNK);
    }
  }
  for (int k = tid; k < RP_DWV_MAXK; k += 256) dsm[k] = (k < K) ? __ldcg(base + op.a + (i64)k * op.a_sk) : 0.f;
  const bool adam = (op.flags & DW_ADAM) != 0, polyak = (op.flags & DW_POLYAK) != 0;
  __syncthreads();                                                   // dout staged
  {
    const int n = tid & (RP_DWV_COLS - 1), half = tid >> 7, q = n >> 5, col = n & 31;
    const int cpt = (nchunks + 1) >> 1;                              // chunks per half
    float acc = 0.f;
    for (int c = half * cpt; c < min(nchunks, (half + 1) * cpt); ++c) {
      rp_mbar_wait(bars + c, (parity >> c) & 1u);
      const float* xb = xs + (q * nchunks + c) * RP_DW_BOX;
      const float* dk = dsm + c * RP_DW_CHUNK;
#pragma unroll 8
      for (int kk = 0; kk < RP_DW_CHUNK; ++kk) acc = fmaf(dk[kk], xb[rp_dw_sw(kk, col)], acc);
    }
    // every thread has to have seen every chunk barrier's phase before the next tile re-arms them
    for (int c = 0; c < nchunks; ++c) rp_mbar_wait(bars + c, (parity >> c) & 1u);
    red[tid] = acc;
  }
  parity ^= (1u << nchunks) - 1u;
  __syncthreads();
  if (tid < RP_DWV_COLS / 4) {                                       // 32 threads, four columns each: the square tiles' epilogue
    const float4 g = make_float4(red[4 * tid] + red[128 + 4 * tid], red[4 * tid + 1] + red[128 + 4 * tid + 1], red[4 * tid + 2] + red[128 + 4 * tid + 2],
                                 red[4 * tid + 3] + red[128 + 4 * tid + 3]);
    EpiPre pre;
    pre.valid = false;
    if (n0 + 4 * tid < N) epilogue_row4<2>(op, ctx, 0, n0 + 4 * tid, g, pre, false);
  }
  if (tile == 0 && op.pb >= 0 && warp == 1) {                        // bias gradient = sum of dout (lane-strided, then butterfly)
    float sacc = 0.f;
    for (int k = lane; k < K; k += 32) sacc += dsm[k];
    sacc = warp_sum(sacc);
    if (lane == 0) {
      float bpre[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
      if (adam) {
        bpre[0] = __ldcg(base + op.pb); bpre[1] = __ldcg(base + op.pbm); bpre[2] = __ldcg(base + op.pbv);
        if (polyak) bpre[3] = __ldcg(base + op.pbt);
        bpre[4] = __ldcg(&ctx.scal->adam_step_size[op.opt]); bpre[5] = __ldcg(&ctx.scal->adam_bc2_sqrt[op.opt]);
        if (polyak) { bpre[6] = __ldcg(&ctx.scal->tau); bpre[7] = __ldcg(&ctx.scal->one_minus_tau); }
      }
      epilogue_bias(op, ctx, 0, sacc, bpre);
    }
  }
  __syncthreads();                                                   // the staging area is reused by the next tile
}

// ---- the step interpreter ---------------------------------------------------------------------------------------------
struct RpSync {            // barrier state that lives across phases and updates
  unsigned gepoch;         // group barrier epoch
  unsigned wphase;         // parity bit per weight slot (TMA mbarriers)
};

// (forceinline on purpose: a single out-of-line copy shared by phases A and C measured 19% SLOWER -- 158.6 vs 133.8 us per
//  update -- although it shrinks the kernel from 389 KB to 276 KB of SASS: the instruction footprint is not what limits it)
__device__ __forceinline__ void rp_run_steps(const RpCtx& c, int s0, int s1, RpSync& sy) {
  RP_SMEM;
  const RpProgram& P = *c.P;
  const int jbeg = P.steps[s0].job0, jend = P.steps[s1 - 1].job0 + P.steps[s1 - 1].njobs;
  float* wring = smem_raw + P.sm_wslot;
  const int B = c.args->hp.B;
  for (int j = jbeg; j < jbeg + 2; ++j) {
    if (j < jend) rp_issue_job(P.jobs[j], wring + (j % RP_NWSLOT) * P.wslot_floats, c, j % RP_NWSLOT);
    cp_async_commit();
  }
  for (int s = s0; s < s1; ++s) {
    const RpStep st = P.steps[s];
    RP_TRACE(1000 + s);
    if (st.nloads > 0) {
      for (int l = st.load0; l < st.load0 + st.nloads; ++l)
        rp_issue_load(P.loads[l], smem_raw + P.sm_abuf + P.loads[l].abuf * P.abuf_floats, P.lda, c.base, c.row0, B);
      cp_async_commit();
      cp_async_wait<0>();
      __syncthreads();
    }
    RP_TRACE(2000 + st.row_op);
    switch (st.row_op) {
      case RPR_GATHER: rp_gather(c, *c.L, c.slots); break;
      case RPR_PI_HEADS: rp_pi_heads(c); break;
      case RPR_TARGET_CRITIC: if (c.args->w_ext) rp_target_critic<true>(c); else rp_target_critic<false>(c); break;
      case RPR_RELOAD: rp_reload(c); break;
      case RPR_ACTOR_Q: rp_actor_q(c); break;
      case RPR_PI_BWD: rp_pi_bwd(c); break;
      default: break;
    }
    RP_TRACE(3000);
    for (int j = st.job0; j < st.job0 + st.njobs; ++j) {
      const int sl = j % RP_NWSLOT;
      cp_async_wait<1>();                      // this thread's share of job j has landed (job j + 1 may still be in flight)
      if (P.jobs[j].tma) {                     // ... and the TMA-staged weight slice
        rp_mbar_wait(c.wbar + sl, (sy.wphase >> sl) & 1u);
        sy.wphase ^= 1u << sl;
      }
      __syncthreads();                         // ... everyone's has; and everyone is done with job j - 1
      RP_TRACE(3500);
      // slot of job j + 2 == slot of job j - 1: free now
      if (j + 2 < jend) rp_issue_job(P.jobs[j + 2], wring + ((j + 2) % RP_NWSLOT) * P.wslot_floats, c, (j + 2) % RP_NWSLOT);
      cp_async_commit();
      RP_TRACE(4000 + j);
      const RpJob jb = P.jobs[j];
      rp_job(jb, c, sl);
      RP_TRACE(5000 + j);
    }
    if (s + 1 < s1) rp_group_barrier(c.gbar, sy.gepoch);
    RP_TRACE(6000 + s);
  }
  cp_async_wait<0>();
  __syncthreads();
}

// program and dW ops -> shared memory: 16-byte loads, all of a thread's loads in flight before its first store (with 4-byte
// loads in two dependent loops this was 4 K of the 7 K cycles a launch spends before its first step). Out of line: its
// registers are its own.
__device__ __noinline__ void rp_stage_program(const Plan* __restrict__ gplan, const RpProgram* __restrict__ gprog, RpProgram* sprog, Op* sops) {
  const int tid = threadIdx.x;
  constexpr int PW = (int)(sizeof(RpProgram) / 16), OW = (int)(RP_MAX_DW_OPS * sizeof(Op) / 16);
  static_assert(sizeof(RpProgram) % 4 == 0 && (RP_MAX_DW_OPS * sizeof(Op)) % 16 == 0 && sizeof(Plan) % 16 == 0 && offsetof(Plan, ops) % 16 == 0,
                "16-byte copies of the program / the dW ops");
  const int4* src = reinterpret_cast<const int4*>(gprog);
  int4* dst = reinterpret_cast<int4*>(sprog);
  const int4* osrc = reinterpret_cast<const int4*>(gplan->ops);
  int4* odst = reinterpret_cast<int4*>(sops);
  constexpr int NP = (PW + 255) / 256, NO = (OW + 255) / 256;
  int4 vp[NP], vo[NO];
#pragma unroll
  for (int u = 0; u < NP; ++u) if (tid + 256 * u < PW) vp[u] = __ldg(src + tid + 256 * u);
#pragma unroll
  for (int u = 0; u < NO; ++u) if (tid + 256 * u < OW) vo[u] = __ldg(osrc + tid + 256 * u);
  if (tid < (int)(sizeof(RpProgram) % 16) / 4)      // tail words of the program
    reinterpret_cast<int*>(sprog)[PW * 4 + tid] = __ldg(reinterpret_cast<const int*>(gprog) + PW * 4 + tid);
#pragma unroll
  for (int u = 0; u < NP; ++u) if (tid + 256 * u < PW) dst[tid + 256 * u] = vp[u];
#pragma unroll
  for (int u = 0; u < NO; ++u) if (tid + 256 * u < OW) odst[tid + 256 * u] = vo[u];
}

// grid = n_groups x 8 CTAs (cooperative launch: all co-resident). gplan: phase 0 = critics' dW + Adam + Polyak tiles,
// phase 1 = policy dW + Adam tiles and the final op (loss means, temperature step, update counter).
__global__ void __launch_bounds__(256, 1) sacx_rp_kernel(const Plan* __restrict__ gplan, const RpProgram* __restrict__ gprog, const RunArgs args) {
  RP_SMEM;
  __shared__ __align__(16) RpProgram sprog;
  __shared__ RpRows rows;
  __shared__ __align__(16) Op sops[RP_MAX_DW_OPS];
  __shared__ Phase sphase[2];
  __shared__ RpTrace trace;
  __shared__ __align__(8) uint64_t wbar[RP_NWSLOT];
  __shared__ __align__(8) uint64_t dwbar[RP_DW_NBAR];
  __shared__ RpLaunch launch;
  __shared__ i64 row_slots[RP_RB];
  __shared__ RunArgs sargs;       // the argument block and the dW tiles' context, read by the helpers (see below)
  __shared__ EpiCtx sec;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
#ifdef SACX_DEBUG_HOOKS
  const long long t_entry = clock64();
#endif
  if (tid == 0) {
    for (int i = 0; i < RP_NWSLOT; ++i) rp_mbar_init(&wbar[i], 8);      // one arrival per warp and job
    for (int i = 0; i < RP_DW_NBAR; ++i) rp_mbar_init(&dwbar[i], 1);    // one arrival (the issuing thread's expect_tx) per dW chunk
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    if (args.rp_maps && (((uint32_t)__cvta_generic_to_shared(smem_raw)) & 1023u)) __trap();   // swizzled tiles need 1024 B alignment
  }
  rp_stage_program(gplan, gprog, &sprog, sops);
  {
    if (tid < 2) sphase[tid] = gplan->phases[tid];
    if (tid == 0) {
      trace.buf = nullptr; trace.n = 0; trace.cap = 0;
      // constant for the whole launch: nothing pushes into the ring or touches the stream keys while the kernel runs
      const AgentScalars* sc = reinterpret_cast<const AgentScalars*>(args.arena + args.scal_off);
      launch.pushes = args.ring ? reinterpret_cast<const RingMeta*>(args.ring)->pushes : 0;
      launch.upd0 = sc->updates; launch.rng_seed = sc->rng_seed; launch.rng_agent = sc->rng_agent; launch.pad = 0;
      launch.oldest_slot = launch.pushes > args.ring_capacity ? (launch.pushes - args.ring_capacity) % args.ring_capacity : 0;
    }
    // the next launch's barrier counters (the two sets alternate): zeroed here, off the critical path, instead of by a memset
    // operation in front of every launch
    if (blockIdx.x == 0 && args.barrier_next)
      for (int i = tid; i < 64 * (1 + RP_MAX_GROUPS); i += 256) args.barrier_next[i] = 0u;
  }
  if (tid == 32) {            // (another warp than the launch constants' thread)
    sargs = args;             // a plain struct copy: &args would bring the stack copy back
    float* b0 = args.arena;
    sec = EpiCtx{b0, reinterpret_cast<AgentScalars*>(b0 + args.scal_off), &sargs.hp, nullptr};
  }
  __syncthreads();
  const int rank = blockIdx.x % RP_CS, gid = blockIdx.x / RP_CS, ngr = sprog.n_row_groups;
  float* base = args.arena;
  AgentScalars* scal = reinterpret_cast<AgentScalars*>(base + args.scal_off);
  const int B = args.hp.B, nrb = (B + RP_RB - 1) / RP_RB;
  // A copy of the argument block (and the dW tiles' context) lives in SHARED memory: as a kernel-local copy -- forced by taking
  // &args -- it sat on the local-memory stack (472 B per thread, 118 KB per CTA: more than the L1 left beside 192 KB of shared
  // memory), and every `c.args->...` in a helper was a local load that regularly missed to L2: 600-800 cycles for a handful of
  // instructions (profiles/r02c_rp_hot_lines.txt). The row-parallel context `c` (104 B) stays per thread: a shared copy whose
  // fields point at the other shared objects made nvcc 12.9 drop those objects.
  // dW phases reuse the tile code of the tile-parallel kernel; their shared memory aliases the row-parallel buffers
  float* wsm = smem_raw;
  float* gsm = smem_raw + WSM_FLOATS;
  float* dwstage = smem_raw + ((WSM_FLOATS + 255) & ~255);      // 1 KB aligned: swizzled TMA boxes
  unsigned dwparity = 0u;
  RpCtx c{base, scal, &sargs, &sprog, &rows, args.rp_part + (i64)gid * sprog.part_stride, args.barrier + 64 * (1 + gid), rank, 0, 0, &trace, wbar, &launch, row_slots};
  const EpiCtx& ec = sec;
  RowCtx rc{base, scal, &sargs, 0, 0, wsm + warp * 4 * SACX_MAX_ACT, gsm, CfgSmall::SMEM_FLOATS, nullptr};      // (no OP_GATHER here: gcache stays null)
  unsigned epoch = 0;
  RpSync sy{0u, 0u};
  unsigned* counter = args.barrier;
  const int sa = sprog.n_steps_a, sc = sprog.n_steps_c;
  for (int step = 0; step < args.n_steps; ++step) {
    c.step = step; rc.step = step;
#ifdef SACX_DEBUG_HOOKS
    if (tid == 0 && args.dbg2 && blockIdx.x == 0 && step + 1 == args.n_steps) {
      trace.buf = args.dbg2 + 1; trace.cap = 1000; trace.n = 0;
      if (step == 0) { trace.buf[0] = 100ull; trace.buf[1] = (unsigned long long)t_entry; trace.n = 1; }      // kernel entry (one-update launches)
      RP_TRACE(101);
    }
#endif
    // optional per-phase timestamps: [step][4 phases][CTA][arrive, release]
    unsigned long long* dbg = (args.dbg && tid == 0) ? args.dbg + ((size_t)step * 4 * gridDim.x + blockIdx.x) * 2 : nullptr;
    const size_t dstride = (size_t)gridDim.x * 2;
    if (blockIdx.x == 0 && tid < 3) {
      Op po; po.mode = 7;
      op_prologue(po, rc, tid);
    }
    for (int ph = 0; ph < 4; ++ph) {
      if ((ph & 1) == 0) {          // row-parallel phases: A (target, critics' forward/backward), C (actor)
        const int s0 = ph ? sa : 0, s1 = ph ? sa + sc : sa;
        if (gid < ngr)                  // (the extra CTAs of a grid sized for the dW phases wait at the phase barrier)
          for (int rb = gid; rb < nrb; rb += ngr) { c.row0 = rb * RP_RB; rp_run_steps(c, s0, s1, sy); }
      } else {                      // tile-parallel phases: dW + Adam (+ Polyak) of the critics (B) / the policy (D)
        const Phase p = sphase[ph >> 1];
        for (int t = blockIdx.x; t < p.ntiles; t += gridDim.x) {
          int oi = p.op0;
          while (oi + 1 < p.op0 + p.nops && t >= sops[oi + 1].tile0) ++oi;
          const Op& op = sops[oi];
          const int lt = t - op.tile0;
          if (op.type == OP_GEMM) {                 // only dW tiles live in these phases
            if (op.i[5] == 1) rp_dw_vec_tile(op, ec, lt, dwstage, args.rp_maps, dwbar, dwparity);      // one-row layer: 128 columns per tile
            else if (rp_dw_tc_ok(op, args.rp_maps)) rp_dw_tile_tc(op, ec, lt, dwstage, args.rp_maps, dwbar, dwparity);
            else gemm_tile_impl<CfgSmall, 2>(op, ec, lt, gsm);
          }
          else if (op.type == OP_FINAL) {
            op_final_par(op, rc, wsm);
            if (warp == 0) {
              if (args.metrics_host && step + 1 == args.n_steps) {
                // the step's result goes straight into pinned host memory (visible to the host once the kernel has completed):
                // no device-to-host copy operation behind the launch
                __syncwarp();
                __threadfence();
                const float* src = reinterpret_cast<const float*>(scal);
                for (int i = lane; i < (int)(sizeof(AgentScalars) / 4); i += 32) args.metrics_host[i] = __ldcg(src + i);
                __threadfence_system();
              }
            }
          }
        }
      }
      const bool very_last = (ph == 3) && (step + 1 == args.n_steps);
      RP_TRACE(7000 + ph);
      if (dbg) dbg[ph * dstride] = clock64();
      if (!very_last) group_barrier_counter(counter, epoch);
      if (dbg) dbg[ph * dstride + 1] = clock64();
    }
  }
  RP_TRACE(9999);
#ifdef SACX_DEBUG_HOOKS
  if (tid == 0 && trace.buf) args.dbg2[0] = (unsigned long long)trace.n;
#endif
}

}  // namespace sacx
