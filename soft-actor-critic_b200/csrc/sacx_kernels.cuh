// The persistent fused update kernel and the small standalone kernels (ring scatter/gather, batch
// load, rollout-side policy / critic forwards).
#pragma once
#include "sacx_gemm.cuh"
#include "sacx_rowops.cuh"

namespace sacx {

constexpr int SMEM_OPS = 64;                                   // ops of the active phase range cached in smem
constexpr int WSM_FLOATS = 8 * 4 * SACX_MAX_ACT;               // per-warp scratch for the row ops

// Barriers among the gridDim.x CTAs that work on the same agent (cooperative launch => co-resident), on a monotonic
// arrival counter with release/acquire at gpu scope.
// Flag form (tile-parallel kernel): arrivals on one line, release flag on another, so pollers do not queue behind the atomics.
__device__ __forceinline__ void group_barrier_flag(unsigned* counter, unsigned& epoch) {
  __syncthreads();
  if (gridDim.x > 1) {
    if (threadIdx.x == 0) {
      epoch += gridDim.x;
      unsigned v, old;
      unsigned* flag = counter + 32;
      asm volatile("atom.add.release.gpu.global.u32 %0, [%1], 1;" : "=r"(old) : "l"(counter) : "memory");
      if (old + 1 == epoch) {
        asm volatile("st.release.gpu.global.u32 [%0], %1;" ::"l"(flag), "r"(epoch) : "memory");
      } else {
        do {
          asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(flag) : "memory");
        } while ((int)(v - epoch) < 0);
      }
    }
    __syncthreads();
  }
}
// Counter form (row-parallel kernel's grid barrier): every CTA polls the arrival counter itself, one L2 hop less than waiting
// for a flag. Thread 0's fences make the CTA's global writes visible and drop stale L1 lines before the other threads continue.
__device__ __forceinline__ void group_barrier_counter(unsigned* counter, unsigned& epoch) {
  __syncthreads();
  if (gridDim.x > 1) {
    if (threadIdx.x == 0) {
      epoch += gridDim.x;
      unsigned v;
      __threadfence();
      atomicAdd(counter, 1u);
      do {
        asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(counter) : "memory");
      } while (v < epoch);
      __threadfence();
    }
    __syncthreads();
  }
}

template <bool LARGE>
__global__ void __launch_bounds__(256, 1) sacx_run_kernel(const Plan* __restrict__ gplan, const RunArgs args) {
  using C = typename std::conditional<LARGE, CfgLarge, CfgSmall>::type;
  extern __shared__ __align__(16) float smem_raw[];
  Op* sops = reinterpret_cast<Op*>(smem_raw);
  float* wsm = smem_raw + (SMEM_OPS * sizeof(Op)) / 4;
  float* gsm = wsm + WSM_FLOATS;
  __shared__ Phase sphase[MAX_PHASES];
  __shared__ uint32_t gcache[8 * GCACHE_WORDS];            // OP_GATHER: per-warp cache of the sampler keys / ring header
  // the argument block the context structs point at is a SHARED copy: &args would put a 328-byte copy on every thread's
  // local-memory stack, and the helpers' reads of it miss the small L1 that is left beside the shared-memory carve-out
  __shared__ RunArgs sargs;
  if (threadIdx.x == 0) sargs = args;
  if (threadIdx.x < 8 * GCACHE_WORDS) gcache[threadIdx.x] = 0xffffffffu;

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int op_lo = gplan->phases[args.phase_begin].op0;
  const int op_hi = gplan->phases[args.phase_end - 1].op0 + gplan->phases[args.phase_end - 1].nops;
  const bool cached = (op_hi - op_lo) <= SMEM_OPS;
  if (cached) {
    const int words = (op_hi - op_lo) * (int)(sizeof(Op) / 4);
    const int* src = reinterpret_cast<const int*>(gplan->ops + op_lo);
    int* dst = reinterpret_cast<int*>(sops);
    for (int i = tid; i < words; i += 256) dst[i] = src[i];
  }
  for (int i = tid; i < gplan->n_phases; i += 256) sphase[i] = gplan->phases[i];
  __syncthreads();
  const Op* ops = cached ? (sops - op_lo) : gplan->ops;

  unsigned epoch = 0;
  unsigned* counter = args.barrier + blockIdx.y * 64;
  for (int agent = blockIdx.y; agent < args.n_agents; agent += gridDim.y) {
    float* base = args.arena + (i64)agent * args.agent_stride;
    AgentScalars* scal = reinterpret_cast<AgentScalars*>(base + args.scal_off);
    RowCtx rc{base, scal, &sargs, agent, 0, wsm + warp * 4 * SACX_MAX_ACT, gsm, C::SMEM_FLOATS, nullptr};
    rc.gcache = gcache + warp * GCACHE_WORDS;
    EpiCtx ec{base, scal, &sargs.hp, nullptr};
    const bool last_agent = (agent + (int)gridDim.y >= args.n_agents);
    for (int step = 0; step < args.n_steps; ++step) {
      rc.step = step;
      for (int p = args.phase_begin; p < args.phase_end; ++p) {
        const Phase ph = sphase[p];
        if (args.dbg2) rc.t = ec.t = args.dbg2 + (((size_t)step * (args.phase_end - args.phase_begin) + (p - args.phase_begin)) * gridDim.x + blockIdx.x) * 8;
        for (int t = blockIdx.x; t < ph.ntiles; t += gridDim.x) {
          int oi = ph.op0;
          while (oi + 1 < ph.op0 + ph.nops && t >= ops[oi + 1].tile0) ++oi;
          const Op& op = ops[oi];
          const int lt = t - op.tile0;
          switch (op.type) {
            case OP_GEMM: if (!(args.tc_skip && (op.cfg & 2))) gemm_tile<C>(op, ec, lt, gsm); break;
            case OP_GATHER: op_gather(op, rc, lt * ROWS_PER_TILE + warp, lane); break;
            case OP_PI_HEAD: tile_pi_head<0>(op, rc, lt); __syncthreads(); break;
            case OP_PI_TAIL: tile_pi_tail(op, rc, lt); break;
            case OP_Q_TAIL: tile_q_tail(op, rc, lt); break;
            case OP_DELTA: tile_delta(op, rc, lt); break;
            case OP_Q_ROW: tile_q_row<0>(op, rc, lt); __syncthreads(); break;
            case OP_ACTOR_Q: tile_actor_q<0>(op, rc, lt); __syncthreads(); break;
            case OP_ACTOR_BWD: tile_actor_bwd<0>(op, rc, lt); __syncthreads(); break;
            case OP_PROLOGUE: if (tid < 3) op_prologue(op, rc, tid); break;
            case OP_FINAL: if (warp == 0) op_final(op, rc, lane); break;
            case OP_POLYAK: op_polyak(op, rc, lt); break;
            case OP_ADAM_FLAT: op_adam_flat(op, rc, lt); break;
            default: break;
          }
        }
        const bool very_last = last_agent && (step + 1 == args.n_steps) && (p + 1 == args.phase_end);
        unsigned long long* dbg = nullptr;
        if (args.dbg && tid == 0) {
          dbg = args.dbg + (((size_t)step * (args.phase_end - args.phase_begin) + (p - args.phase_begin)) * gridDim.x + blockIdx.x) * 2;
          dbg[0] = clock64();
        }
        if (!very_last) group_barrier_flag(counter, epoch);
        if (dbg) dbg[1] = clock64();
      }
    }
  }
}

// Light kernel for the phases of a large-batch plan that hold no FFMA GEMM tile (row ops, gather, flat optimiser ops): the
// persistent kernel above needs 255 registers and ~200 KB of shared memory, i.e. one CTA (8 rows in flight) per SM; at
// batch 65536 the row phases are then bound by the latency of a tile's dependent loads. Same tile functions (their
// own copy, V = 1), 3 CTAs per SM. One phase per launch, single agent or blockIdx.y = agent.
// forward layer with a very short reduction (first layer of a low-dimensional observation: K = obs (+ act) <= 32 with rows
// TMA cannot address, e.g. K = 5): 64x64 tile of the op's tile grid, thread = one output column x 16 rows, the weight row
// in registers, the input rows as warp-wide broadcast loads. Memory-bound on the output write.
constexpr int SMALLK_MAX = 32;
__device__ __forceinline__ bool small_fwd_ok(const Op& o) {
  return o.type == OP_GEMM && o.epi == EPI_FWD && o.K <= SMALLK_MAX && o.zout < 0 && o.a_sk == 1 && o.b_sk == 1 && o.cfg >= 1;
}
// K <= KB: the reduction is unrolled over KB register-resident weights; the tile's 64 input rows are staged (zero-padded to
// KB) in shared memory first, so the inner loop has no global load and no predicate. (Profile history: one 32-wide bucket
// ran 32 predicated steps per output for a K = 5 layer -- instruction-bound; per-row global loads -- latency-bound.)
// Called by all 256 threads of the CTA (two barriers inside); xs: 64 * KB floats of shared memory.
// Tiles are enumerated ROW-BLOCK-minor (tile = tn * tiles_m + tm): with gridDim.x dividing tiles_m a CTA keeps its row block
// while it walks the column tiles -- and the second critic of the phase, which reads the same input -- so the 64 x K input rows
// are staged ONCE per CTA (`reuse_x`: the caller saw the same input matrix and row block in its previous tile) instead of once
// per tile behind two barriers and a dependent global round trip (8 per CTA before: ~400 us per phase for a 1024-agent
// population against a 90 us store floor).
template <int KB>
__device__ __forceinline__ void small_fwd_tile_k(const Op& op, float* __restrict__ base, int tile, float* __restrict__ xs, bool reuse_x) {
  // the op lives in shared memory: its fields go to registers once (left in place the compiler re-read them around every global
  // store -- the profile of this tile showed ~50 instructions per output row, most of them such reloads and address arithmetic)
  const int M = op.M, N = op.N, K = op.K, ldc = op.ldc, a_sm = op.a_sm, b_sn = op.b_sn, act = op.act;
  const i64 oa = op.a, ob = op.b, oc = op.c, obias = op.bias;
  const int tiles_m = (M + 63) >> 6;
  const int tm = tile % tiles_m, tn = tile / tiles_m;
  if (!reuse_x) {
    __syncthreads();
    for (int i = threadIdx.x; i < 64 * KB; i += 256) {
      const int r = i / KB, k = i % KB, m = tm * 64 + r;
      xs[i] = (m < M && k < K) ? __ldcg(base + oa + (i64)m * a_sm + k) : 0.f;
    }
    __syncthreads();
  }
  const int n = tn * 64 + (threadIdx.x & 63), r0 = (threadIdx.x >> 6) * 16;
  if (n >= N) return;
  float w[KB];
#pragma unroll
  for (int k = 0; k < KB; ++k) w[k] = (k < K) ? __ldg(base + ob + (i64)n * b_sn + k) : 0.f;
  const float bias = __ldg(base + obias + n);
  float* __restrict__ out = base + oc + (i64)(tm * 64 + r0) * ldc + n;
  const int rows = min(16, M - (tm * 64 + r0));
  const bool relu = act == SACX_ACT_RELU;
#pragma unroll
  for (int r = 0; r < 16; ++r) {
    // the row is the same address in every lane of the warp: 16-byte broadcast loads, KB / 4 per row instead of KB
    const float4* x4 = reinterpret_cast<const float4*>(xs + (r0 + r) * KB);
    float s = bias;
#pragma unroll
    for (int q = 0; q < KB / 4; ++q) {
      const float4 xv = x4[q];
      s = fmaf(xv.x, w[4 * q], s); s = fmaf(xv.y, w[4 * q + 1], s); s = fmaf(xv.z, w[4 * q + 2], s); s = fmaf(xv.w, w[4 * q + 3], s);
    }
    const float o = relu ? fmaxf(s, 0.f) : act_fwd(act, s);
    if (r < rows) { *out = o; }
    out += ldc;
  }
}
// (a 4 x 4 output block per thread with 16-byte stores was tried for K <= 8: its weight reads from shared memory are
//  16-way bank-conflicted at this K and it measured 45% slower -- 584 vs 402 us per phase for a 1024-agent population)
__device__ __forceinline__ void small_fwd_tile(const Op& op, float* __restrict__ base, int tile, float* __restrict__ xs, bool reuse_x) {
  if (op.K <= 8) small_fwd_tile_k<8>(op, base, tile, xs, reuse_x);
  else if (op.K <= 16) small_fwd_tile_k<16>(op, base, tile, xs, reuse_x);
  else small_fwd_tile_k<SMALLK_MAX>(op, base, tile, xs, reuse_x);
}

// weight gradient of a narrow output layer whose delta rows TMA cannot address (policy head with 2A not a multiple of 4:
// row stride 8 or 24 bytes): dW[m][n] = sum_b dy[b][m] x[b][n] (+ db[m] = sum_b dy[b][m]), M <= 8 rows, 64-column tile of the
// op's tile grid, batch range split over 4 thread groups and reduced through shared memory, optimiser epilogue as in
// sacx_gemm.cuh. Called by all 256 threads; xs: >= 4 * 64 * 9 floats.
constexpr int SMALLM_MAX = 8, SMALLDW_MAXK = 4096;
__device__ __forceinline__ bool small_dw_ok(const Op& o) {
  return o.type == OP_GEMM && o.epi == EPI_DW && o.M <= SMALLM_MAX && o.K <= SMALLDW_MAXK && o.a_sm == 1 && o.b_sn == 1 && o.cfg >= 1 &&
         !(o.flags & DW_ATOMIC) && o.i[0] <= 1;
}
__device__ __forceinline__ void small_dw_tile(const Op& op, float* __restrict__ base, const AgentScalars* scal, const Hyper& hp, int tile,
                                              float* __restrict__ xs) {
  const int tn = tile % op.tiles_n, c = threadIdx.x & 63, kg = threadIdx.x >> 6, n = tn * 64 + c;
  const int kper = (op.K + 3) >> 2, b0 = kg * kper, b1 = min(op.K, b0 + kper);
  float acc[SMALLM_MAX + 1];
#pragma unroll
  for (int m = 0; m <= SMALLM_MAX; ++m) acc[m] = 0.f;
  if (n < op.N) {
    int b = b0;
    for (; b + 3 < b1; b += 4) {              // four batch rows per step: their loads are in flight together
      float x[4], d[4][SMALLM_MAX];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        x[u] = __ldcg(base + op.b + (i64)(b + u) * op.b_sk + n);
        const float* dy = base + op.a + (i64)(b + u) * op.a_sk;
#pragma unroll
        for (int m = 0; m < SMALLM_MAX; ++m) d[u][m] = (m < op.M) ? __ldcg(dy + m) : 0.f;
      }
#pragma unroll
      for (int u = 0; u < 4; ++u)
#pragma unroll
        for (int m = 0; m < SMALLM_MAX; ++m) acc[m] = fmaf(d[u][m], x[u], acc[m]);
    }
    for (; b < b1; ++b) {
      const float x = __ldcg(base + op.b + (i64)b * op.b_sk + n);
      const float* dy = base + op.a + (i64)b * op.a_sk;
#pragma unroll
      for (int m = 0; m < SMALLM_MAX; ++m)
        if (m < op.M) acc[m] = fmaf(__ldcg(dy + m), x, acc[m]);
    }
  }
  if (tn == 0 && c < op.M)                      // bias gradient: column c of dy
    for (int b = b0; b < b1; ++b) acc[SMALLM_MAX] += __ldcg(base + op.a + (i64)b * op.a_sk + c);
  __syncthreads();
#pragma unroll
  for (int m = 0; m <= SMALLM_MAX; ++m) xs[(kg * 64 + c) * (SMALLM_MAX + 1) + m] = acc[m];
  __syncthreads();
  if (kg == 0) {
    const float ss = (op.flags & DW_ADAM) ? __ldcg(&scal->adam_step_size[op.opt]) : 0.f;
    const float bc = (op.flags & DW_ADAM) ? __ldcg(&scal->adam_bc2_sqrt[op.opt]) : 1.f;
    const float tau = __ldcg(&scal->tau), omt = __ldcg(&scal->one_minus_tau);
    auto apply = [&](float g, i64 p, i64 pm, i64 pv, i64 pt, i64 pg) {
      if (op.flags & DW_STORE_GRAD) base[pg] = g;
      if (op.flags & DW_ADAM) {
        float w = base[p], mm = base[pm], vv = base[pv];
        adam_update(g, w, mm, vv, ss, bc);
        base[p] = w; base[pm] = mm; base[pv] = vv;
        if ((op.flags & DW_POLYAK) && pt >= 0) base[pt] = polyak_mix(tau, omt, w, base[pt]);
      }
    };
    for (int m = 0; m <= SMALLM_MAX; ++m) {
      float g = 0.f;
      for (int q = 0; q < 4; ++q) g += xs[(q * 64 + c) * (SMALLM_MAX + 1) + m];
      if (m < op.M && n < op.N) {
        const i64 e = (i64)m * op.N + n;
        apply(g, op.p + e, op.pm + e, op.pv + e, op.pt >= 0 ? op.pt + e : -1, op.pg + e);
      } else if (m == SMALLM_MAX && tn == 0 && c < op.M && op.pb >= 0) {
        apply(g, op.pb + c, op.pbm + c, op.pbv + c, op.pbt >= 0 ? op.pbt + c : -1, op.pbg + c);
      }
    }
  }
}

constexpr int ROWS_SMEM_OPS = 8;
__global__ void __launch_bounds__(256, 3) sacx_rows_kernel(const Plan* __restrict__ gplan, const RunArgs args, int tsm_floats) {
  extern __shared__ __align__(16) float rows_raw[];
  __shared__ Op sops[ROWS_SMEM_OPS];
  __shared__ float fred[8];
  __shared__ uint32_t gcache[8 * GCACHE_WORDS];            // OP_GATHER: per-warp cache of the sampler keys / ring header
  __shared__ RunArgs sargs;                                // (shared copy of the argument block: see sacx_run_kernel)
  if (threadIdx.x == 0) sargs = args;
  if (threadIdx.x < 8 * GCACHE_WORDS) gcache[threadIdx.x] = 0xffffffffu;
  float* wsm = rows_raw;
  float* tsm = rows_raw + WSM_FLOATS;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const Phase ph = gplan->phases[args.phase_begin];
  const bool cached = ph.nops <= ROWS_SMEM_OPS;
  if (cached) {
    const int words = ph.nops * (int)(sizeof(Op) / 4);
    const int* src = reinterpret_cast<const int*>(gplan->ops + ph.op0);
    int* dst = reinterpret_cast<int*>(sops);
    for (int i = tid; i < words; i += 256) dst[i] = src[i];
  }
  __syncthreads();
  const Op* ops = cached ? (sops - ph.op0) : gplan->ops;
  for (int agent = blockIdx.y; agent < args.n_agents; agent += gridDim.y) {
    float* base = args.arena + (i64)agent * args.agent_stride;
    AgentScalars* scal = reinterpret_cast<AgentScalars*>(base + args.scal_off);
    RowCtx rc{base, scal, &sargs, agent, 0, wsm + warp * 4 * SACX_MAX_ACT, tsm, tsm_floats, nullptr};
    rc.gcache = gcache + warp * GCACHE_WORDS;
    int last_oi = -1;
    i64 sm_a = -1;                                  // input matrix / row block of the small-K tile staged last (uniform over the CTA)
    int sm_ld = 0, sm_k = 0, sm_tm = -1;
    rc.pf_rows = 2 * (int)gridDim.x * ROWS_PER_TILE;
    for (int t = blockIdx.x; t < ph.ntiles; t += gridDim.x) {
      int oi = ph.op0;
      while (oi + 1 < ph.op0 + ph.nops && t >= ops[oi + 1].tile0) ++oi;
      const Op& op = ops[oi];
      const int lt = t - op.tile0;
      // head weights are staged once per (agent, op) run of tiles, not once per 8 rows; between two tiles of the same op the
      // warps are NOT synchronised (each owns its row and its scratch), so a warp whose row is done moves on to the next
      // tile's loads -- the CTA-wide barrier sits only where the staging area changes hands
      rc.fresh = (oi != last_oi);
      if (rc.fresh && last_oi != -1) __syncthreads();
      last_oi = oi;
      switch (op.type) {
        case OP_GEMM:
          if (op.cfg & 2) break;                      // tensor-core kernel
          if (small_fwd_ok(op)) {                   // (these tiles use the staging area themselves)
            const int tm_ = lt % ((op.M + 63) >> 6);
            const bool reuse = last_oi == -3 && sm_a == op.a && sm_ld == op.a_sm && sm_k == op.K && sm_tm == tm_;
            small_fwd_tile(op, base, lt, tsm, reuse);
            sm_a = op.a; sm_ld = op.a_sm; sm_k = op.K; sm_tm = tm_;
            last_oi = -3;                           // -3: the staging area holds a small-K input tile (any other op re-stages)
          }
          else if (small_dw_ok(op)) { small_dw_tile(op, base, scal, sargs.hp, lt, tsm); last_oi = -2; }
          break;
        case OP_GATHER: op_gather(op, rc, lt * ROWS_PER_TILE + warp, lane); break;
        case OP_PI_HEAD: tile_pi_head<1>(op, rc, lt); break;
        case OP_PI_TAIL: tile_pi_tail(op, rc, lt); break;
        case OP_Q_TAIL: tile_q_tail(op, rc, lt); break;
        case OP_DELTA: tile_delta(op, rc, lt); break;
        case OP_Q_ROW: tile_q_row<1>(op, rc, lt); break;
        case OP_ACTOR_Q: tile_actor_q<1>(op, rc, lt); break;
        case OP_ACTOR_BWD: tile_actor_bwd<1>(op, rc, lt); break;
        case OP_PROLOGUE: if (tid < 3) op_prologue(op, rc, tid); break;
        case OP_FINAL: op_final_impl<true>(op, rc, tid, fred); break;      // all 256 threads: B terms per mean
        case OP_POLYAK: op_polyak(op, rc, lt); break;
        case OP_ADAM_FLAT: op_adam_flat(op, rc, lt); break;
        default: break;        // GEMM ops of this phase run on the tensor-core kernel
      }
    }
  }
}

// ---------------------------------------------------------------- ring kernels
struct StageHdr {
  int agent, pad;
  i64 push_no;
};

// Ring layout: one PACKED record per slot, [s (O) | s2 (O) | a (A) | r | d | pad] = RS floats (RS = 2O + A + 2 rounded up to a
// multiple of 4, so records start 16-byte aligned; BipedalWalker: 56 floats = 224 B = seven 32-byte sectors). A sampled
// transition is one contiguous read instead of five pieces in five arrays: the round-1 SoA ring moved 2.9x the algorithmic
// bytes from DRAM on a 1M-row gather (every piece cost its own 64-byte granules). Field f of slot k lives at
// rb[off_f + k * RS + i]; off_* are the field offsets inside the record plus the ring header.

// staged host rows [s | a | r | s2 | d] -> ring records (slot = push_no % capacity); bumps the agent's push count
__global__ void ring_scatter_kernel(float* __restrict__ ring, i64 ring_stride, i64 cap, i64 off_s, i64 off_a, i64 off_r,
                                    i64 off_s2, i64 off_d, int RS, int O, int A, const float* __restrict__ rows,
                                    const StageHdr* __restrict__ hdr, int n) {
  const int W = 2 * O + A + 2;
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= n) return;
  const StageHdr h = hdr[row];
  float* rb = ring + (i64)h.agent * ring_stride;
  float* rec = rb + (h.push_no % cap) * RS;
  const float* src = rows + (i64)row * W;
  for (int k = lane; k < O; k += 32) {
    rec[off_s + k] = src[k];
    rec[off_s2 + k] = src[O + A + 1 + k];
  }
  for (int k = lane; k < A; k += 32) rec[off_a + k] = src[O + k];
  if (lane == 0) {
    rec[off_r] = src[O + A];
    rec[off_d] = src[2 * O + A + 1];
    atomicMax(reinterpret_cast<unsigned long long*>(&reinterpret_cast<RingMeta*>(rb)->pushes),
              (unsigned long long)(h.push_no + 1));
  }
}

// rows already on the device (SoA inputs) for one agent
__global__ void ring_scatter_dev_kernel(float* __restrict__ rb, i64 cap, i64 off_s, i64 off_a, i64 off_r, i64 off_s2,
                                        i64 off_d, int RS, int O, int A, const float* __restrict__ s, const float* __restrict__ a,
                                        const float* __restrict__ r, const float* __restrict__ s2,
                                        const float* __restrict__ d, i64 push0, int n) {
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= n) return;
  float* rec = rb + ((push0 + row) % cap) * RS;
  for (int k = lane; k < O; k += 32) {
    rec[off_s + k] = s[(i64)row * O + k];
    rec[off_s2 + k] = s2[(i64)row * O + k];
  }
  for (int k = lane; k < A; k += 32) rec[off_a + k] = a[(i64)row * A + k];
  if (lane == 0) {
    rec[off_r] = r[row];
    rec[off_d] = d[row];
    if (row == n - 1)
      atomicMax(reinterpret_cast<unsigned long long*>(&reinterpret_cast<RingMeta*>(rb)->pushes),
                (unsigned long long)(push0 + n));
  }
}

// uniform-index gather, any dimensions: one warp per sampled row; logical deque position -> ring slot.
// Streaming loads (ld.global.cs): every row is touched once per update and the 1M-row ring does not fit L2.
__global__ void ring_gather_kernel(const float* __restrict__ rb, i64 cap, i64 off_s, i64 off_a, i64 off_r, i64 off_s2,
                                   i64 off_d, int RS, int O, int A, const i64* __restrict__ idx, int B, float* __restrict__ s,
                                   float* __restrict__ a, float* __restrict__ r, float* __restrict__ s2,
                                   float* __restrict__ d) {
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= B) return;
  const i64 pushes = reinterpret_cast<const RingMeta*>(rb)->pushes;
  const i64 oldest = pushes > cap ? pushes - cap : 0;
  const i64 j = idx[row];
  const bool in = j >= 0 && j < (pushes < cap ? pushes : cap);          // a position outside the deque reads nothing: zero row
  const float* rec = rb + ((oldest + (in ? j : 0)) % cap) * RS;
  if (s) for (int k = lane; k < O; k += 32) s[(i64)row * O + k] = in ? __ldcs(rec + off_s + k) : 0.f;
  if (s2) for (int k = lane; k < O; k += 32) s2[(i64)row * O + k] = in ? __ldcs(rec + off_s2 + k) : 0.f;
  if (a) for (int k = lane; k < A; k += 32) a[(i64)row * A + k] = in ? __ldcs(rec + off_a + k) : 0.f;
  if (lane == 0) {
    if (r) r[row] = in ? __ldcs(rec + off_r) : 0.f;
    if (d) d[row] = in ? __ldcs(rec + off_d) : 0.f;
  }
}

// The same gather with one THREAD per 16-byte piece of the record (obs and act dimensions multiples of 4): a BipedalWalker
// record is 14 pieces -> 16 threads, two rows per warp, the whole record in flight at once and read as consecutive sectors.
// Piece p of the record holds 4 floats of s (p < O/4), of s2, of a, or the (r, d, pad, pad) tail.
__global__ void ring_gather_vec_kernel(const float* __restrict__ rb, i64 cap, i64 oldest_slot, i64 n_valid, i64 off_s, int RS, int O, int A,
                                       const i64* __restrict__ idx, int B, float* __restrict__ s, float* __restrict__ a,
                                       float* __restrict__ r, float* __restrict__ s2, float* __restrict__ d, int tpr_log2) {
  // every thread owns the same 16-byte piece of TWO rows (row, row + ceil(B / 2)): two independent record reads in flight per
  // thread before the first store
  const i64 gt = (i64)blockIdx.x * blockDim.x + threadIdx.x;
  const int half = (B + 1) >> 1;
  const int row0 = (int)(gt >> tpr_log2), piece = (int)(gt & ((1 << tpr_log2) - 1));
  if (row0 >= half) return;
  const int cs = O >> 2, ca = A >> 2;
  if (piece > 2 * cs + ca) return;
  // slot of the oldest survivor and the deque length come from the host (it owns the push counter): no header read, and one
  // conditional subtraction instead of a 64-bit modulo per thread
  int rows[2] = {row0, row0 + half};
  float4 v[2];
#pragma unroll
  for (int u = 0; u < 2; ++u) {
    v[u] = make_float4(0.f, 0.f, 0.f, 0.f);
    if (rows[u] < B) {
      const i64 j = __ldg(idx + rows[u]);
      if (j >= 0 && j < n_valid) {                                        // a position outside the deque reads nothing: zero row
        i64 slot = oldest_slot + j;
        if (slot >= cap) slot -= cap;
        v[u] = __ldcs(reinterpret_cast<const float4*>(rb + off_s + slot * RS) + piece);
      }
    }
  }
#pragma unroll
  for (int u = 0; u < 2; ++u) {
    const int row = rows[u];
    if (row >= B) continue;
    if (piece < cs) {
      if (s) __stcs(reinterpret_cast<float4*>(s + (i64)row * O) + piece, v[u]);
    } else if (piece < 2 * cs) {
      if (s2) __stcs(reinterpret_cast<float4*>(s2 + (i64)row * O) + piece - cs, v[u]);
    } else if (piece < 2 * cs + ca) {
      if (a) __stcs(reinterpret_cast<float4*>(a + (i64)row * A) + piece - 2 * cs, v[u]);
    } else {
      if (r) r[row] = v[u].x;
      if (d) d[row] = v[u].y;
    }
  }
}

__global__ void ring_indices_kernel(const float* __restrict__ rb, i64 cap, unsigned long long seed,
                                    unsigned long long counter, int agent, int B, i64* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B) return;
  const i64 pushes = reinterpret_cast<const RingMeta*>(rb)->pushes;
  const i64 n = pushes < cap ? pushes : cap;
  out[i] = (i64)feistel_index((unsigned long long)i, (unsigned long long)n, seed, counter, (uint32_t)agent);
}

// ---- device-side observation assembly of the DonkeyVae producer (SURVEY 8f-4) ------------------------------------------------
// reference: DonkeyCarEnv/donkey_gym/envs/vae_env.py:175-210 (postprocessing_step) and :253-266 (reset). The VAE latent is
// already on the device (ae/autoencoder.py encodes on cuda); the 2 x n_command_history command history is rolled, the
// [latent | history] frame appended to the n_stack frame stack (zeroed first when the episode ended), and the transition
// (previous stack, action, reward, new stack, done) is left in device staging for sacx_ring_push_n_dev -- no host bounce.
//   hist  [n_cmd * n_hist]        command history (oldest first)
//   stack [n_stack * frame]       frame stack (oldest first), frame = z + n_cmd * n_hist
//   prev  [n_stack * frame]       out: the stack before this step (the transition's state)
// One CTA; every thread reads what it needs before the barrier and writes after it (in-place roll).
__global__ void obs_assemble_kernel(float* __restrict__ hist, float* __restrict__ stack, float* __restrict__ prev, float* __restrict__ act_out,
                                    float* __restrict__ rd_out, const float* __restrict__ latent, const float* __restrict__ action,
                                    float a0, float a1, float reward, int done, int reset, int z, int n_cmd, int n_hist, int n_stack) {
  extern __shared__ float sm[];
  const int H = n_cmd * n_hist, F = z + H, S = n_stack * F;
  float* nh = sm;            // new history [H]
  float* ns = sm + H;        // new stack [S]
  for (int i = threadIdx.x; i < H; i += blockDim.x) {
    float v;
    if (reset) v = 0.f;
    else if (i < H - n_cmd) v = hist[i + n_cmd];                                  // np.roll(history, -n_cmd)
    else { const int j = i - (H - n_cmd); v = action ? action[j] : (j == 0 ? a0 : a1); }      // history[-n_cmd:] = action
    nh[i] = v;
  }
  for (int i = threadIdx.x; i < S; i += blockDim.x) prev[i] = stack[i];
  __syncthreads();
  for (int i = threadIdx.x; i < S; i += blockDim.x) {
    float v;
    if (i >= S - F) { const int j = i - (S - F); v = j < z ? latent[j] : nh[j - z]; }          // newest frame = [latent | history]
    else v = (reset || done) ? 0.f : prev[i + F];                                 // np.roll(stack, -F); zeroed on reset / done
    ns[i] = v;
  }
  __syncthreads();
  for (int i = threadIdx.x; i < H; i += blockDim.x) hist[i] = nh[i];
  for (int i = threadIdx.x; i < S; i += blockDim.x) stack[i] = ns[i];
  if (threadIdx.x < n_cmd && act_out) act_out[threadIdx.x] = action ? action[threadIdx.x] : (threadIdx.x == 0 ? a0 : a1);
  if (threadIdx.x == 0 && rd_out) { rd_out[0] = reward; rd_out[1] = done ? 1.f : 0.f; }
}

// external batch -> the arena's batch buffers (staged API): X_sa=[s|a], X_pi=[s|.], X_s2=[s2|.], r, d
__global__ void load_batch_kernel(float* __restrict__ base, i64 x_sa, i64 x_s2, i64 x_pi, i64 r_off, i64 d_off, int ldx,
                                  int O, int A, int B, const float* __restrict__ s, const float* __restrict__ a,
                                  const float* __restrict__ r, const float* __restrict__ s2, const float* __restrict__ d) {
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= B) return;
  if (s) for (int k = lane; k < O; k += 32) {
    const float v = s[(i64)row * O + k];
    base[x_sa + (i64)row * ldx + k] = v;
    base[x_pi + (i64)row * ldx + k] = v;
  }
  if (s2) for (int k = lane; k < O; k += 32) base[x_s2 + (i64)row * ldx + k] = s2[(i64)row * O + k];
  if (a) for (int k = lane; k < A; k += 32) base[x_sa + (i64)row * ldx + O + k] = a[(i64)row * A + k];
  if (lane == 0) {
    if (r) base[r_off + row] = r[row];
    if (d) base[d_off + row] = d[row];
  }
}

__global__ void copy_out_kernel(const float* __restrict__ src, float* __restrict__ dst, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) dst[i] = src[i];
}

// ---------------------------------------------------------------- rollout-side forwards (a13, _log_q_values)
struct NetRef {          // one MLP inside an agent arena
  int n_lin, in_dim, out_dim, act_h, act_o;
  int dims[SACX_MAX_HIDDEN + 2];
  i64 W[SACX_MAX_HIDDEN + 1], b[SACX_MAX_HIDDEN + 1];
};

// one CTA per row: activations ping-pong in shared memory, one warp per output neuron
__device__ __forceinline__ const float* mlp_row(const float* __restrict__ base, const NetRef& net, float* buf0, float* buf1) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  float* in = buf0;
  float* out = buf1;
  for (int l = 0; l < net.n_lin; ++l) {
    const int K = net.dims[l], N = net.dims[l + 1];
    const int act = (l + 1 < net.n_lin) ? net.act_h : net.act_o;
    for (int o = warp; o < N; o += nw) {
      const float* w = base + net.W[l] + (i64)o * K;
      float s = 0.f;
      for (int k = lane; k < K; k += 32) s = fmaf(in[k], __ldg(w + k), s);
      s = warp_sum(s);
      if (lane == 0) out[o] = act_fwd(act, s + __ldg(base + net.b[l] + o));
    }
    __syncthreads();
    float* t = in; in = out; out = t;
  }
  return in;
}

__global__ void act_kernel(const float* __restrict__ base, NetRef net, int maxw, const float* __restrict__ s,
                           const float* __restrict__ eps, int deterministic, float* __restrict__ a_out, int A,
                           float lo, float hi, float scale, i64 scal_off, unsigned long long counter,
                           int agent0, i64 agent_stride) {
  // grid (rows per agent, agents): blockIdx.y walks a population (vectorised rollouts: one launch for every agent's action)
  extern __shared__ float sm[];
  float* b0 = sm;
  float* b1 = sm + maxw;
  const int agent = agent0 + blockIdx.y;
  base += (i64)agent * agent_stride;
  const AgentScalars* scal = reinterpret_cast<const AgentScalars*>(base + scal_off);      // the agent's own stream keys
  const int row = blockIdx.y * gridDim.x + blockIdx.x;
  for (int k = threadIdx.x; k < net.in_dim; k += blockDim.x) b0[k] = s[(i64)row * net.in_dim + k];
  __syncthreads();
  const float* head = mlp_row(base, net, b0, b1);
  for (int j = threadIdx.x; j < A; j += blockDim.x) {
    const float mu = head[j];
    float v;
    if (deterministic) {
      v = tanhf(mu) * scale;                                     // models.py:89-92
    } else {
      const float e = eps ? eps[(i64)row * A + j]
                          : philox_normal(scal->rng_seed, counter, 3, (uint32_t)blockIdx.x, (uint32_t)j, scal->rng_agent);
      v = sac_rsample(mu, head[A + j], e, lo, hi).tz * scale;     // models.py:79-84
    }
    a_out[(i64)row * A + j] = v;
  }
}

__global__ void qvalue_kernel(const float* __restrict__ base, NetRef q1, NetRef q2, int maxw, int O, int A,
                              const float* __restrict__ s, const float* __restrict__ a, float* __restrict__ q1_out,
                              float* __restrict__ q2_out) {
  extern __shared__ float sm[];
  float* b0 = sm;
  float* b1 = sm + maxw;
  const int row = blockIdx.x;
  const NetRef& net = blockIdx.y == 0 ? q1 : q2;
  for (int k = threadIdx.x; k < O + A; k += blockDim.x)
    b0[k] = k < O ? s[(i64)row * O + k] : a[(i64)row * A + (k - O)];
  __syncthreads();
  const float* out = mlp_row(base, net, b0, b1);
  if (threadIdx.x == 0) (blockIdx.y == 0 ? q1_out : q2_out)[row] = out[0];
}

}  // namespace sacx
