// libsacx.so -- C ABI (include/sacx.h) over the B200-native SAC update engine.
// Compile: nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -shared -Xcompiler -fPIC
#include "../../include/sacx.h"

#include <cuda_runtime.h>

#include <cmath>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "sacx_engine.cuh"
#include "sacx_pbt.cuh"
#include "sacx_per.cuh"

namespace sacx {

thread_local std::string g_err;
int fail(int code, const std::string& msg) {
  g_err = msg;
  return code;
}

// ------------------------------------------------------------------------------------------ ring
constexpr int STAGE_ROWS = 4096;

struct Ring {
  int O, A, n_agents, W;
  i64 cap, stride;                      // float words per agent block
  i64 off_s, off_a, off_r, off_s2, off_d;   // field offsets inside a packed record, ring header included
  int RS = 0;                           // floats per record
  float* dev = nullptr;
  bool own = false;
  float* h_rows = nullptr;              // pinned staging [STAGE_ROWS, W]
  StageHdr* h_hdr = nullptr;
  float* d_rows = nullptr;
  StageHdr* d_hdr = nullptr;
  int staged = 0;
  int stage_limit = STAGE_ROWS;          // <= capacity: two staged rows never target the same slot
  std::vector<i64> pushes;              // host mirror of RingMeta.pushes (includes staged rows)
  cudaStream_t stream = 0;
  cudaEvent_t stage_free = nullptr;     // staging block may be overwritten once this event has fired
  bool stage_busy = false;
  // scratch for the host gather
  void* scr_dev = nullptr; size_t scr_dev_bytes = 0;
  void* scr_host = nullptr; size_t scr_host_bytes = 0;
  long long launches = 0;

  // packed records [s | s2 | a | r | d | pad], RS = align4(2O + A + 2) floats each, behind the 32-byte ring header
  static int record_floats(int O, int A) { return (2 * O + A + 2 + 3) & ~3; }
  static void offsets(int O, int A, i64 cap, i64& s, i64& a, i64& r, i64& s2, i64& d, i64& total) {
    const i64 hdr = (i64)(sizeof(RingMeta) / 4);
    s = hdr; s2 = hdr + O; a = hdr + 2 * O; r = hdr + 2 * O + A; d = r + 1;
    total = (hdr + cap * record_floats(O, A) + 127) & ~(i64)127;
  }
  i64 len(int agent) const { return std::min(pushes[agent], cap); }
  float* block(int agent) const { return dev + (i64)agent * stride; }

  int wait_stage() {
    if (stage_busy) {
      SACX_CUDA(cudaEventSynchronize(stage_free));
      stage_busy = false;
    }
    return SACX_OK;
  }
  int flush() {
    if (staged == 0) return SACX_OK;
    SACX_CUDA(cudaMemcpyAsync(d_rows, h_rows, (size_t)staged * W * sizeof(float), cudaMemcpyHostToDevice, stream));
    SACX_CUDA(cudaMemcpyAsync(d_hdr, h_hdr, (size_t)staged * sizeof(StageHdr), cudaMemcpyHostToDevice, stream));
    ring_scatter_kernel<<<(staged + 7) / 8, 256, 0, stream>>>(dev, stride, cap, off_s, off_a, off_r, off_s2, off_d, RS, O, A,
                                                              d_rows, d_hdr, staged);
    ++launches;
    SACX_CUDA(cudaGetLastError());
    SACX_CUDA(cudaEventRecord(stage_free, stream));
    stage_busy = true;
    staged = 0;
    return SACX_OK;
  }
  int push(int agent, const float* s, const float* a, float r, const float* s2, float d) {
    if (agent < 0 || agent >= n_agents) return fail(SACX_ERR_INVALID, "ring push: agent out of range");
    if (staged == 0) { int rc = wait_stage(); if (rc) return rc; }
    float* row = h_rows + (size_t)staged * W;
    memcpy(row, s, O * sizeof(float));
    memcpy(row + O, a, A * sizeof(float));
    row[O + A] = r;
    memcpy(row + O + A + 1, s2, O * sizeof(float));
    row[2 * O + A + 1] = d;
    h_hdr[staged].agent = agent;
    h_hdr[staged].pad = 0;
    h_hdr[staged].push_no = pushes[agent]++;
    if (++staged >= stage_limit) return flush();
    return SACX_OK;
  }
  int ensure_scratch(size_t bytes) {
    if (bytes > scr_dev_bytes) {
      if (scr_dev) cudaFree(scr_dev);
      if (scr_host) cudaFreeHost(scr_host);
      scr_dev = scr_host = nullptr; scr_dev_bytes = scr_host_bytes = 0;
      SACX_CUDA(cudaMalloc(&scr_dev, bytes));
      SACX_CUDA(cudaMallocHost(&scr_host, bytes));
      scr_dev_bytes = scr_host_bytes = bytes;
    }
    return SACX_OK;
  }
};

// ------------------------------------------------------------------------------------------ prioritized replay tree
// Host side of sacx_per.cuh: owns the tree's device memory (the agent arena is untouched) and issues per_refresh_kernel.
// Every call is one cooperative launch on the attached agent's stream (else the ring's). The write-back of an agent update
// is deferred into the next launch (the next update's sample, or a read of the priorities); every launch that can overwrite
// the arena's per-row q / y flushes it first (engine_launch, engine_launch_rp).
struct Per {
  Ring* ring = nullptr;
  Engine* agent = nullptr;
  float alpha = 0.6f, eps = 1e-6f;
  double beta0 = 0.4;
  i64 beta_steps = 0;
  int max_batch = 0, depth = 0, grid_max = 1;
  i64 nodes[PER_MAX_LEVELS + 1] = {};
  i64 internal = 0;                    // internal nodes over all levels
  float* d_leaf = nullptr;
  float* d_tree = nullptr;             // sums of levels 1..depth, then mins
  unsigned* d_mark = nullptr;
  unsigned long long* d_win = nullptr;
  PerState* d_st = nullptr;
  i64* d_idx = nullptr; float* d_w = nullptr; i64* d_slots = nullptr;   // [max_batch]: the agent update's batch
  unsigned epoch = 0;
  i64 seen_hint = 0;                   // host view of PerState::seen (sizes the grid only)
  bool rebuild = true;                 // internal nodes not valid yet (create, load_priorities)
  int pend_n = 0;                      // deferred write-back: rows of the last agent update
  const float *pend_q1 = nullptr, *pend_q2 = nullptr, *pend_y = nullptr;

  cudaStream_t stream() const { return agent ? agent->stream : ring->stream; }

  PerArgs base() {
    PerArgs a;
    memset(&a, 0, sizeof a);
    a.leaf = d_leaf;
    i64 off = 0;
    for (int l = 1; l <= depth; ++l) {
      a.sum[l] = d_tree + off; a.mn[l] = d_tree + internal + off; a.mark[l] = d_mark + off;
      off += nodes[l];
    }
    for (int l = 0; l <= depth; ++l) a.nodes[l] = nodes[l];
    a.depth = depth; a.win = d_win; a.st = d_st; a.hdr = reinterpret_cast<const RingMeta*>(ring->block(0)); a.cap = ring->cap;
    a.alpha = alpha; a.eps = eps; a.beta0 = beta0; a.beta_steps = beta_steps;
    if (pend_n) {
      a.wb_n = pend_n; a.wb_slots = d_slots; a.wb_q1 = pend_q1; a.wb_q2 = pend_q2; a.wb_y = pend_y;
    }
    return a;
  }
  int run(PerArgs& a) {
    int rc = ring->flush();
    if (rc) return rc;
    if (ring->stream != stream()) SACX_CUDA(cudaStreamSynchronize(ring->stream));
    const i64 pushes = ring->pushes[0], n_new = pushes - seen_hint;
    const bool full = rebuild || n_new < 0 || n_new >= ring->cap;
    const i64 work = full ? ring->cap : std::max<i64>(a.B, a.wb_n + n_new);
    a.rebuild = rebuild ? 1 : 0;
    a.epoch = ++epoch;
    // one warp per row / touched leaf: the sampler's walk and the propagation are chains of dependent L2 reads, so the
    // rows run side by side rather than one after another on fewer warps (B 256: 32 CTAs)
    const int blocks = (int)std::max<i64>(1, std::min<i64>(grid_max, (work + 7) / 8));
    void* args[] = {(void*)&a};
    SACX_CUDA(cudaLaunchCooperativeKernel((const void*)per_refresh_kernel, dim3(blocks), dim3(256), args, 0, stream()));
    if (agent) ++agent->launches;
    seen_hint = pushes; rebuild = false; pend_n = 0;
    return SACX_OK;
  }
  int flush() { PerArgs a = base(); return run(a); }
};

// ------------------------------------------------------------------------------------------ engine runtime
static int per_flush_pending(Engine* e) { return (e->per && e->per->pend_n) ? e->per->flush() : SACX_OK; }

static int engine_launch(Engine* e, int plan_id, int pb, int pe, int n_steps, const RunArgs& proto, bool per_phase) {
  { int rc = per_flush_pending(e); if (rc) return rc; }
  const Plan& hp = e->h_plans[plan_id];
  if (pe < 0) pe = hp.n_phases;
  RunArgs a = proto;
  a.arena = e->arena; a.agent_stride = e->stride; a.scal_off = e->scal_off; a.hp = e->hp;
  a.n_agents = e->cfg.n_agents; a.barrier = e->d_barrier; a.ctas_per_agent = e->grid_x;
  if (e->ring) {
    Ring* r = e->ring;
    a.ring = r->dev; a.ring_stride = r->stride; a.ring_capacity = r->cap;
    a.ring_s = r->off_s; a.ring_a = r->off_a; a.ring_r = r->off_r; a.ring_s2 = r->off_s2; a.ring_d = r->off_d; a.ring_rs = r->RS;
  }
  const Plan* dplan = e->d_plans + plan_id;
  auto launch = [&](int p0, int p1, int steps, dim3 grid, bool coop) -> int {
    a.phase_begin = p0; a.phase_end = p1; a.n_steps = steps;
    void* args[] = {(void*)&dplan, (void*)&a};
    const void* fn = e->large ? (const void*)sacx_run_kernel<true> : (const void*)sacx_run_kernel<false>;
    if (coop) {
      SACX_CUDA(cudaMemsetAsync(e->d_barrier, 0, sizeof(unsigned) * 64 * (size_t)std::max(1, (int)grid.y), e->stream));
      SACX_CUDA(cudaLaunchCooperativeKernel(fn, grid, dim3(256), args, (size_t)e->smem_bytes, e->stream));
    } else {
      SACX_CUDA(cudaLaunchKernel(fn, grid, dim3(256), args, (size_t)e->smem_bytes, e->stream));
    }
    ++e->launches;
    return SACX_OK;
  };
  if (e->tc && !per_phase) {
    bool any = false;      // something to gain: a tensor-core GEMM, or a GEMM-free phase for the light row kernel
    for (int p = pb; p < pe; ++p) any = any || !e->tc_phases[plan_id][p].groups.empty() || e->tc_phases[plan_id][p].light;
    if (any) {
      // tensor-core plan walk: runs of phases without TC ops go through the persistent kernel (cooperative when the run
      // has more than one phase); a phase with TC ops launches the tcgen05 kernel per group of <= 4 GEMMs (+ the dW
      // reduce/optimiser kernel) and, when it also holds row ops, the persistent kernel with the TC GEMMs masked out
      const i64 nb = (i64)e->cfg.n_agents * e->cfg.batch_size;
      for (int s = 0; s < n_steps; ++s) {
        if (proto.idx_ext) a.idx_ext = proto.idx_ext + s * nb;
        if (proto.eps1_ext) a.eps1_ext = proto.eps1_ext + s * nb * e->cfg.act_dim;
        if (proto.eps2_ext) a.eps2_ext = proto.eps2_ext + s * nb * e->cfg.act_dim;
        auto launch_rows = [&](int p) -> int {
          a.phase_begin = p; a.phase_end = p + 1; a.n_steps = 1; a.tc_skip = 1;
          const int tiles = std::max(1, hp.phases[p].ntiles);
          // ~8 waves of CTAs over the chip; a CTA keeps to one agent and walks its tiles, so head weights are staged once
          const int na = e->cfg.n_agents, slots = e->n_sms * e->rows_ctas_per_sm;
          const int gx = na == 1 ? std::min(tiles, slots) : std::min(tiles, std::max(1, (8 * slots + na - 1) / na));
          sacx_rows_kernel<<<dim3(gx, std::min(na, 65535)), 256, e->rows_smem_bytes, e->stream>>>(
              dplan, a, e->rows_tsm_floats);
          ++e->launches;
          return SACX_OK;
        };
        int p = pb;
        while (p < pe) {
          Engine::TcPhase& tp = e->tc_phases[plan_id][p];
          if (tp.groups.empty()) {
            if (tp.light) { launch_rows(p); ++p; continue; }
            int q = p + 1;
            while (q < pe && e->tc_phases[plan_id][q].groups.empty() && !e->tc_phases[plan_id][q].light) ++q;
            a.tc_skip = 0;
            int rc = launch(p, q, 1, dim3(e->grid_x, e->grid_y), e->grid_x > 1 && q - p > 1);
            if (rc) return rc;
            p = q;
            continue;
          }
          if (tp.other_ops) {
            if (tp.light) launch_rows(p);
            else {
              a.tc_skip = 1;
              int rc = launch(p, p + 1, 1, dim3(e->grid_x, e->grid_y), false);
              if (rc) return rc;
              a.tc_skip = 0;
            }
          }
          for (Engine::TcGroup& g : tp.groups) {
            sacx_tc_kernel<<<g.grid, TC_THREADS, TC_SMEM_BYTES, e->stream>>>(g.p, g.maps);
            ++e->launches; ++e->tc_launches;
            if (g.has_red) {
              tc_dw_reduce_kernel<<<dim3(g.red_blocks, g.red.n_ops, e->cfg.n_agents), 256, 0, e->stream>>>(g.red);
              ++e->launches;
            }
          }
          SACX_CUDA(cudaGetLastError());
          ++p;
        }
      }
      return SACX_OK;
    }
  }
  if (per_phase) {
    // one launch per phase, no in-kernel barrier: grid.x covers the phase's tiles, grid.y the agents
    for (int s = 0; s < n_steps; ++s) {
      RunArgs keep = a;
      // external per-step arrays advance on the host
      const i64 nb = (i64)e->cfg.n_agents * e->cfg.batch_size;
      if (proto.idx_ext) a.idx_ext = proto.idx_ext + s * nb;
      if (proto.eps1_ext) a.eps1_ext = proto.eps1_ext + s * nb * e->cfg.act_dim;
      if (proto.eps2_ext) a.eps2_ext = proto.eps2_ext + s * nb * e->cfg.act_dim;
      for (int p = pb; p < pe; ++p) {
        const int tiles = std::max(1, hp.phases[p].ntiles);
        int rc = launch(p, p + 1, 1, dim3(std::min(tiles, 65535), std::min(e->cfg.n_agents, 65535)), false);
        if (rc) return rc;
      }
      a = keep;
    }
    return SACX_OK;
  }
  const bool coop = e->grid_x > 1;
  const bool single_pass = (pe - pb == 1) && n_steps == 1 && e->grid_y >= e->cfg.n_agents;
  return launch(pb, pe, n_steps, dim3(e->grid_x, e->grid_y), coop && !single_pass);
}

// Row-parallel launch: n_groups x 8 CTAs, cooperative (all CTAs co-resident: grid and group barriers spin).

static int engine_launch_rp(Engine* e, int n_steps, const RunArgs& proto) {
  { int rc = per_flush_pending(e); if (rc) return rc; }
  RunArgs a = proto;
  a.arena = e->arena; a.agent_stride = e->stride; a.scal_off = e->scal_off; a.hp = e->hp;
  a.n_agents = 1; a.barrier = e->d_barrier; a.ctas_per_agent = e->rp_grid;
  a.n_steps = n_steps; a.phase_begin = 0; a.phase_end = 2;
  if (e->ring) {
    Ring* r = e->ring;
    a.ring = r->dev; a.ring_stride = r->stride; a.ring_capacity = r->cap;
    a.ring_s = r->off_s; a.ring_a = r->off_a; a.ring_r = r->off_r; a.ring_s2 = r->off_s2; a.ring_d = r->off_d; a.ring_rs = r->RS;
  }
  a.rp_part = e->d_rp_part;
  a.rp_maps = e->d_rp_maps;
  // two counter sets of its own (behind the tile-parallel kernel's region of d_barrier): launch L spins on set L & 1 and zeroes the
  // other one for launch L + 1; both start zeroed at create. When the caller captures the stream into a graph, replays would
  // freeze that alternation: a captured launch uses the first set and zeroes it in front of the kernel instead.
  {
    unsigned* sets = e->d_barrier + 64 * 2048;
    const size_t set_words = 64 * (1 + RP_MAX_GROUPS);
    const int cur = (int)(e->rp_launch_no & 1);
    a.barrier = sets + cur * set_words;
    a.barrier_next = sets + (cur ^ 1) * set_words;
    cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
    if (cudaStreamIsCapturing(e->stream, &cs) == cudaSuccess && cs != cudaStreamCaptureStatusNone) {
      a.barrier = e->d_barrier; a.barrier_next = nullptr;
      SACX_CUDA(cudaMemsetAsync(e->d_barrier, 0, sizeof(unsigned) * set_words, e->stream));
    } else {
      ++e->rp_launch_no;
    }
  }
  const Plan* dplan = e->d_plans + PLAN_RP;
  const RpProgram* dprog = e->d_prog;
  void* kargs[] = {(void*)&dplan, (void*)&dprog, (void*)&a};
  SACX_CUDA(cudaLaunchCooperativeKernel((const void*)sacx_rp_kernel, dim3(e->rp_grid), dim3(256), kargs, (size_t)e->rp_smem_bytes, e->stream));
  ++e->launches;
  return SACX_OK;
}

static int engine_setup_rp(Engine* e) {
  if (!e->rp) return SACX_OK;
  auto off = [&](const std::string& why) { e->rp = false; e->rp_why = why; cudaGetLastError(); return SACX_OK; };
  cudaFuncAttributes fa;
  if (cudaFuncGetAttributes(&fa, sacx_rp_kernel) != cudaSuccess) return off("cudaFuncGetAttributes failed");
  e->rp_smem_bytes = e->h_prog.sm_total * 4;
  int dev = 0, max_optin = 0;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&max_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
  if ((size_t)e->rp_smem_bytes + fa.sharedSizeBytes > (size_t)max_optin) return off("shared memory budget exceeded");
  if (cudaFuncSetAttribute(sacx_rp_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, e->rp_smem_bytes) != cudaSuccess)
    return off("cannot raise the dynamic shared memory limit");
  const int nrb = (e->cfg.batch_size + RP_RB - 1) / RP_RB;
  int per_sm = 0;
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, sacx_rp_kernel, 256, (size_t)e->rp_smem_bytes) != cudaSuccess || per_sm < 1)
    return off("row-parallel kernel does not fit on an SM");
  int n_groups = std::min(e->n_sms / RP_CS, RP_MAX_GROUPS);
  const char* env = getenv("SACX_RP_GROUPS");
  if (env && atoi(env) > 0) n_groups = std::min(n_groups, atoi(env));
  if (n_groups < 1) return off("fewer than 8 SMs");
  // balanced rounds: with 16 row blocks and 18 possible groups, 16 groups do one round each
  const int rounds = (nrb + n_groups - 1) / n_groups;
  n_groups = (nrb + rounds - 1) / rounds;
  e->rp_grid = n_groups * RP_CS;
  e->h_prog.n_row_groups = n_groups;
  if (e->d_rp_part) { cudaFree(e->d_rp_part); e->d_rp_part = nullptr; }       // (second call: plans rebuilt after a failed tensor-core setup)
  if (e->d_prog) { cudaFree(e->d_prog); e->d_prog = nullptr; }
  SACX_CUDA(cudaMalloc((void**)&e->d_rp_part, sizeof(float) * (size_t)RP_MAX_GROUPS * e->h_prog.part_stride));
  SACX_CUDA(cudaMemset(e->d_rp_part, 0, sizeof(float) * (size_t)RP_MAX_GROUPS * e->h_prog.part_stride));
  SACX_CUDA(cudaMalloc((void**)&e->d_prog, sizeof(RpProgram)));
  SACX_CUDA(cudaMemcpy(e->d_prog, &e->h_prog, sizeof(RpProgram), cudaMemcpyHostToDevice));
  return SACX_OK;
}

// ---- tensor-core path setup: mark the eligible GEMM ops of every plan, encode their TMA descriptors ------------------------
typedef CUresult (*TcEncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                               const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                               CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

// fp32 tensor [outer][inner] with row stride ld (floats); out-of-range box elements read as zero / are not written.
// swz: 0 = 128B swizzle (epilogue tiles, 32-float rows), 1 = 128B swizzle with 32B atoms (MN-major operands), 2 = 64B
// swizzle (K-major operands, 16-float rows)
// (the third dimension is the agent: slices `agent_stride` floats apart)
static bool tc_encode(TcEncodeFn enc, CUtensorMap* map, const float* base, uint64_t inner, uint64_t outer, uint64_t ld,
                      uint32_t box_in, uint32_t box_out, int swz, uint64_t n_agents, uint64_t agent_stride) {
  cuuint64_t dims[3] = {inner, outer, n_agents};
  cuuint64_t strides[2] = {ld * 4, std::max<uint64_t>(agent_stride, 4) * 4};
  cuuint32_t box[3] = {box_in, box_out, 1};
  cuuint32_t estr[3] = {1, 1, 1};
  return enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<float*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
             swz == 1 ? CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B : swz == 2 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_128B,
             CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
             CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

static int engine_setup_tc(Engine* e) {
  e->tc = e->tc_wanted(e->tc_why);
  if (!e->tc) return SACX_OK;
  auto off = [&](const std::string& why) { e->tc = false; e->tc_why = why; e->tc_phases.clear(); cudaGetLastError(); return SACX_OK; };
#ifdef SACX_DEBUG_HOOKS      // failure injection for tests/test_gpu_tc.py (libsacx_debug.so only)
  if (getenv("SACX_TC_FAIL")) return off("forced setup failure (SACX_TC_FAIL, test hook)");
#endif
  void* fn = nullptr;
  cudaDriverEntryPointQueryResult qres;
  if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres) != cudaSuccess || !fn)
    return off("cuTensorMapEncodeTiled is not available");
  TcEncodeFn enc = (TcEncodeFn)fn;
  if (cudaFuncSetAttribute(sacx_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, TC_SMEM_BYTES) != cudaSuccess)
    return off("cannot raise the dynamic shared memory limit of the tensor-core kernel");
  auto rup = [](int x, int m) { return (x + m - 1) / m * m; };
  const uint64_t NA = (uint64_t)e->cfg.n_agents, AS = (uint64_t)e->stride;
  uint64_t sstride = 4;                  // scratch floats per agent (known after pass 0)
  {  // light row kernel: staging area for the widest head (falls back to global reads beyond 48 KB)
    const int A = e->cfg.act_dim, Kp = e->pi.dims[e->pi.L()], Kq = e->q1.dims[e->q1.L()], H0 = e->q1.dims[1];
    int need = std::max(std::max(2 * A * Kp + 2 * A, 4 * Kq), 2 * A * H0 + 2 * A * Kp);
    const int small_floats = std::max(2 * 64 * SMALLK_MAX, 4 * 64 * (SMALLM_MAX + 1));  // small-K forward input + weight tiles / narrow dW reduction
    need = std::max(need, small_floats);
    e->rows_tsm_floats = std::max(std::min(rup(need, 4), 12288), small_floats);
    e->rows_smem_bytes = (WSM_FLOATS + e->rows_tsm_floats) * 4;
    if (cudaFuncSetAttribute(sacx_rows_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, e->rows_smem_bytes) != cudaSuccess)
      return off("cannot size the row kernel's shared memory");
    int per_sm = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, sacx_rows_kernel, 256, (size_t)e->rows_smem_bytes) != cudaSuccess || per_sm < 1)
      return off("row kernel does not fit on an SM");
    e->rows_ctas_per_sm = per_sm;
  }
  // pass 0 sizes the scratch (dW partial tiles), pass 1 builds descriptors against the allocated scratch
  for (int pass = 0; pass < 2; ++pass) {
    size_t need = 0;
    bool ok = true;
    e->tc_phases.assign(N_PLANS, std::vector<Engine::TcPhase>());
    for (int id = 0; id < N_PLANS; ++id) {
      Plan& pl = e->h_plans[id];
      if (id == PLAN_RP) continue;
      e->tc_phases[id].resize(pl.n_phases);
      for (int ph = 0; ph < pl.n_phases; ++ph) {
        Engine::TcPhase& tp = e->tc_phases[id][ph];
        std::vector<int> elig;
        for (int i = pl.phases[ph].op0; i < pl.phases[ph].op0 + pl.phases[ph].nops; ++i) {
          if (e->tc_op_eligible(pl.ops[i])) { elig.push_back(i); pl.ops[i].cfg |= 2; }
          else {
            tp.other_ops = true;
            const int ty = pl.ops[i].type;
            const Op& oo = pl.ops[i];
            const bool small_fwd = ty == OP_GEMM && oo.epi == EPI_FWD && oo.K <= SMALLK_MAX && oo.zout < 0 && oo.a_sk == 1 &&
                                   oo.b_sk == 1 && oo.cfg >= 1;      // the light kernel's small_fwd_tile (64x64 tile grid)
            const bool small_dw = ty == OP_GEMM && oo.epi == EPI_DW && oo.M <= SMALLM_MAX && oo.K <= SMALLDW_MAXK && oo.a_sm == 1 && oo.b_sn == 1 &&
                                  oo.cfg >= 1 && !(oo.flags & DW_ATOMIC) && oo.i[0] <= 1;         // the light kernel's small_dw_tile
            if ((ty == OP_GEMM && !small_fwd && !small_dw) || ty == OP_LOAD_EXT || ty == OP_NONE) tp.light = false;
            if (pass == 1 && id == PLAN_FUSED && ty == OP_GEMM && !small_fwd && !small_dw && getenv("SACX_TC_VERBOSE"))
              fprintf(stderr, "sacx: FFMA leftover in the fused plan: phase %d epi %d M %d N %d K %d a_sm %d a_sk %d b_sk %d b_sn %d\n", ph, oo.epi,
                      oo.M, oo.N, oo.K, oo.a_sm, oo.a_sk, oo.b_sk, oo.b_sn);
          }
        }
        size_t so = 0;                       // scratch offset inside this phase (floats)
        for (size_t g0 = 0; g0 < elig.size(); g0 += TC_MAX_OPS) {
          tp.groups.emplace_back();
          Engine::TcGroup& g = tp.groups.back();
          memset(&g.p, 0, sizeof g.p); memset(&g.maps, 0, sizeof g.maps); memset(&g.red, 0, sizeof g.red);
          g.p.arena = e->arena; g.p.scratch = e->d_tc_scratch;
          g.p.n_agents = (int)NA; g.p.agent_stride = (i64)AS; g.p.scratch_stride = (i64)sstride;
#ifdef SACX_DEBUG_HOOKS
          { const char* dv = getenv("SACX_TC_DBG"); g.p.dbg = dv ? atoi(dv) : 0; }
#endif
          g.red.arena = e->arena; g.red.scratch = e->d_tc_scratch; g.red.scal_off = e->scal_off; g.red.hp = e->hp;
          g.red.agent_stride = (i64)AS; g.red.scratch_stride = (i64)sstride;
          int tiles = 0;
          for (size_t k = g0; k < std::min(elig.size(), g0 + TC_MAX_OPS); ++k) {
            const Op& o = pl.ops[elig[k]];
            const int j = g.p.n_ops++;
            TcOp& t = g.p.ops[j];
            t.kind = o.epi; t.act = o.act; t.M = o.M; t.N = o.N; t.K = o.K;
            t.n_mma = rup(o.N, 16);
            t.a_bytes = TC_A_BYTES;
            t.m_tiles = (o.M + TC_BM - 1) / TC_BM;
            t.splits = 1; t.k_per_split = rup(o.K, TC_BK);
            t.bias = o.bias; t.bias_part = -1;
            t.proj_w = o.o[28]; t.proj_out = o.o[29]; t.proj_b = o.o[30];      // critic head riding on this layer (blank(): -1)
            const float* A = e->arena + o.a;
            const float* Bm = e->arena + o.b;
            if (o.epi == EPI_FWD || o.epi == EPI_DACT) {
              ok = ok && tc_encode(enc, &g.maps.a[j], A, o.K, o.M, o.a_sm, TC_BK, TC_BM, 2, NA, AS);
              // (a width that is not a multiple of 4 floats: store the zero columns of the 16-byte padded rows as well)
              ok = ok && tc_encode(enc, &g.maps.c[j], e->arena + o.c, (o.N & 3) ? std::min(rup(o.N, 4), o.ldc) : o.N, o.M, o.ldc, 32, TC_BM, 0, NA, AS);
              if (o.epi == EPI_FWD) {
                t.b_rows = t.n_mma; t.b_bytes = t.n_mma * TC_BK * 4;
                ok = ok && tc_encode(enc, &g.maps.b[j], Bm, o.K, o.N, o.b_sn, TC_BK, t.n_mma, 2, NA, AS);
              } else {
                t.b_mn = 1; t.b_rows = (t.n_mma + 31) / 32; t.b_bytes = t.b_rows * TC_SLAB; t.has_aux = 1;
                ok = ok && tc_encode(enc, &g.maps.b[j], Bm, o.N, o.K, o.b_sk, 32, TC_BK, 1, NA, AS);
                ok = ok && tc_encode(enc, &g.maps.aux[j], e->arena + o.aux, o.N, o.M, o.ld_aux, 32, TC_BM, 0, NA, AS);
              }
            } else {
              t.a_mn = t.b_mn = 1;
              t.b_rows = (t.n_mma + 31) / 32; t.b_bytes = t.b_rows * TC_SLAB;
              t.k_per_split = std::min(1024, std::max(256, rup((o.K + 63) / 64, TC_BK)));
              t.splits = (o.K + t.k_per_split - 1) / t.k_per_split;
              const int m_pad = t.m_tiles * TC_BM, n_ld = rup(o.N, 4);
              TcRedOp& r = g.red.ops[g.red.n_ops++];
              r.op = o; r.splits = t.splits; r.m_pad = m_pad; r.n_ld = n_ld;
              r.part = (i64)so; so += (size_t)t.splits * m_pad * n_ld;
              r.bias_part = (i64)so; so += (size_t)t.splits * m_pad * TC_SPLIT_WARPS;
              t.bias_part = o.pb >= 0 ? r.bias_part : -1;
              g.has_red = true;
              g.red_blocks = std::max(g.red_blocks, std::min(1024, (o.M * ((o.N + 3) / 4) + o.M + 255) / 256));
              ok = ok && tc_encode(enc, &g.maps.a[j], A, o.M, o.K, o.a_sk, 32, TC_BK, 1, NA, AS);
              ok = ok && tc_encode(enc, &g.maps.b[j], Bm, o.N, o.K, o.b_sk, 32, TC_BK, 1, NA, AS);
              if (pass == 1)
                ok = ok && tc_encode(enc, &g.maps.c[j], e->d_tc_scratch + r.part, n_ld, (uint64_t)t.splits * m_pad, n_ld, 32, TC_BM, 0, NA, sstride);
            }
            t.idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)t.a_mn << 15) | ((uint32_t)t.b_mn << 16) |
                      ((uint32_t)(t.n_mma >> 3) << 17) | ((uint32_t)(TC_BM >> 4) << 24);
            t.tile0 = tiles; t.ntiles = t.m_tiles * t.splits;
            tiles += t.ntiles;
          }
          g.p.tiles_per_agent = tiles;
          g.p.total_tiles = tiles * (int)NA;
          g.grid = std::max(1, std::min(g.p.total_tiles, e->n_sms));
        }
        need = std::max(need, so);
      }
    }
    if (!ok) return off("cuTensorMapEncodeTiled rejected an operand layout");
    if (pass == 0) {
      sstride = (uint64_t)((need + 63) / 64 * 64 + 64);
      e->tc_scratch_floats = (size_t)sstride * NA;
      SACX_CUDA(cudaMalloc((void**)&e->d_tc_scratch, e->tc_scratch_floats * sizeof(float)));
      SACX_CUDA(cudaMemset(e->d_tc_scratch, 0, e->tc_scratch_floats * sizeof(float)));
    }
  }
  return SACX_OK;
}

// tensor maps of the row-parallel kernel: the TMA-staged weight slices of the jobs, then the dW tiles' operands (needs the arena
// address). Either set failing to encode leaves its consumers on their cp.async path.
static int engine_setup_rp_tma(Engine* e) {
  if (!e->rp) return SACX_OK;
  RpProgram& P = e->h_prog;
  Plan& plan = e->h_plans[PLAN_RP];
  void* fn = nullptr;
  cudaDriverEntryPointQueryResult qres;
  const bool have = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres) == cudaSuccess && fn;
  const int nj = 2 * P.n_jobs;                                   // job j: map 2j, and 2j + 1 for the second slice of a pair
  std::vector<CUtensorMap> maps(nj + 2 * plan.n_ops);
  memset(maps.data(), 0, sizeof(CUtensorMap) * maps.size());
  bool ok = have;
  for (int j = 0; ok && j < P.n_jobs; ++j) {
    const RpJob& jb = P.jobs[j];
    if (!jb.tma) continue;
    cuuint64_t dims[2], strides[1] = {(cuuint64_t)jb.w_ld * 4};
    cuuint32_t box[2], estr[2] = {1, 1};
    box[0] = 32; box[1] = 32;                                   // 32 x 32 tiles (4 KB), one per warp
    if (!jb.bkm) { dims[0] = jb.K; dims[1] = jb.N; }            // W [N][K]: 32 rows n x 32 k
    else { dims[0] = jb.N; dims[1] = jb.K; }                    // W [K][N]: 32 rows k x 32 columns n
    for (int h = 0; ok && h <= (jb.pair && jb.w2_off > 0 ? 1 : 0); ++h)
      ok = ((TcEncodeFn)fn)(&maps[h ? jb.map2 : jb.map], CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, e->arena + (h ? jb.w2 : jb.w), dims, strides, box, estr,
                            CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                            CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
  }
  if (!ok) { for (int j = 0; j < P.n_jobs; ++j) P.jobs[j].tma = 0; cudaGetLastError(); }
  // dW operands: dy [batch][M] and x [batch][N], boxes of 64 batch rows x 32 columns
  const char* dw_env = getenv("SACX_RP_DW_TMA");               // 0: keep the dW tiles on the FFMA / cp.async tile (A/B measurements)
  bool ok_dw = have && !(dw_env && atoi(dw_env) == 0);
  for (int k = 0; k < plan.n_ops; ++k) { plan.ops[k].i[2] = 0; plan.ops[k].i[3] = 0; }
  for (int k = 0; ok_dw && k < plan.n_ops; ++k) {
    Op& o = plan.ops[k];
    if (o.type != OP_GEMM || o.epi != EPI_DW || o.a_sm != 1 || o.b_sn != 1 || (o.a & 3) || (o.b & 3) || (o.a_sk & 3) || (o.b_sk & 3)) continue;
    if (o.K > RP_DW_MAXK || o.cfg != 0) continue;            // (cfg 0: the 32 x 32 tile grid this kernel walks)
    for (int w = 0; ok_dw && w < 2; ++w) {
      cuuint64_t dims[2] = {(cuuint64_t)(w ? o.N : o.M), (cuuint64_t)o.K}, strides[1] = {(cuuint64_t)(w ? o.b_sk : o.a_sk) * 4};
      cuuint32_t box[2] = {32, (cuuint32_t)RP_DW_CHUNK}, estr[2] = {1, 1};
      ok_dw = ((TcEncodeFn)fn)(&maps[nj + 2 * k + w], CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, e->arena + (w ? o.b : o.a), dims, strides, box, estr,
                               CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                               CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
    }
    if (ok_dw) { o.i[2] = nj + 2 * k + 1; o.i[3] = nj + 2 * k + 2; }
  }
  if (!ok_dw) { for (int k = 0; k < plan.n_ops; ++k) { plan.ops[k].i[2] = 0; plan.ops[k].i[3] = 0; } cudaGetLastError(); }
  // one-row output layers (the critics' heads) as 128-column vector tiles (rp_dw_vec_tile) instead of 32 x 32 tiles with one valid
  // row each; then the tile offsets of the two dW phases are recomputed and the grid grows to the widest phase (up to one CTA per
  // SM): the extra CTAs own no row block and only work in the tile-parallel phases.
  const char* vec_env = getenv("SACX_RP_DW_VEC");
  if (ok_dw && !(vec_env && atoi(vec_env) == 0)) {
    for (int k = 0; k < plan.n_ops; ++k) {
      Op& o = plan.ops[k];
      o.i[5] = 0;
      if (o.type == OP_GEMM && o.epi == EPI_DW && o.i[3] > 0 && o.M == 1 && o.K <= RP_DWV_MAXK && o.N >= 64 && !(o.flags & DW_ATOMIC) && o.i[0] <= 1) {
        o.i[5] = 1; o.tiles_n = (o.N + RP_DWV_COLS - 1) / RP_DWV_COLS; o.ntiles = o.tiles_n;
      }
    }
    int widest = 0;
    for (int ph = 0; ph < plan.n_phases; ++ph) {
      Phase& p = plan.phases[ph];
      p.ntiles = 0;
      for (int k = p.op0; k < p.op0 + p.nops; ++k) { plan.ops[k].tile0 = p.ntiles; p.ntiles += plan.ops[k].ntiles; }
      widest = std::max(widest, p.ntiles);
    }
    e->rp_grid = std::min(e->n_sms, std::max(e->rp_grid, widest));
  }
  if (e->d_rp_maps) { cudaFree(e->d_rp_maps); e->d_rp_maps = nullptr; }
  bool up = cudaMalloc(&e->d_rp_maps, sizeof(CUtensorMap) * maps.size()) == cudaSuccess;
  up = up && cudaMemcpy(e->d_rp_maps, maps.data(), sizeof(CUtensorMap) * maps.size(), cudaMemcpyHostToDevice) == cudaSuccess;
  if (!up) {
    for (int j = 0; j < P.n_jobs; ++j) P.jobs[j].tma = 0;
    for (int k = 0; k < plan.n_ops; ++k) { plan.ops[k].i[2] = 0; plan.ops[k].i[3] = 0; }
    if (e->d_rp_maps) { cudaFree(e->d_rp_maps); e->d_rp_maps = nullptr; }
    cudaGetLastError();
  }
  SACX_CUDA(cudaMemcpy(e->d_prog, &e->h_prog, sizeof(RpProgram), cudaMemcpyHostToDevice));
  return SACX_OK;
}

static int engine_init_scalars(Engine* e) {
  AgentScalars s;
  memset(&s, 0, sizeof s);
  s.log_alpha = std::log(e->cfg.alpha);
  // auto: alpha = exp(log_alpha) in f64 (agent.py:50); fixed: torch.tensor(alpha) is f32 (agent.py:55)
  s.alpha = e->cfg.auto_entropy_tuning ? std::exp(s.log_alpha) : (double)(float)e->cfg.alpha;
  s.alpha_f32 = (float)s.alpha;
  s.metrics[4] = (float)s.alpha;
  s.metrics[5] = (float)s.log_alpha;
  // per-agent hyper-parameters start at the config's values (lr 0 = "use Hyper.lr"); the device RNG streams are keyed by
  // (train.seed, GLOBAL agent id): agents that share a local index on different ranks draw different streams
  s.gamma = e->hp.gamma; s.tau = e->hp.tau; s.one_minus_tau = e->hp.one_minus_tau;
  s.rng_seed = e->hp.seed;
  std::vector<AgentScalars> all((size_t)e->cfg.n_agents, s);
  for (int ag = 0; ag < e->cfg.n_agents; ++ag) {
    all[ag].rng_agent = (unsigned)(e->cfg.agent_id_base + ag);
    SACX_CUDA(cudaMemcpyAsync(e->arena + (i64)ag * e->stride + e->scal_off, &all[ag], sizeof s, cudaMemcpyHostToDevice, e->stream));
  }
  SACX_CUDA(cudaStreamSynchronize(e->stream));
  return SACX_OK;
}

static int validate(const sacx_config* c) {
  if (!c) return fail(SACX_ERR_INVALID, "null config");
  if (c->n_hidden_pi <= 0 || c->n_hidden_q <= 0) return fail(SACX_ERR_EMPTY_HIDDEN, "hidden_sizes cannot be empty");
  if (c->n_hidden_pi > SACX_MAX_HIDDEN || c->n_hidden_q > SACX_MAX_HIDDEN)
    return fail(SACX_ERR_INVALID, "more than SACX_MAX_HIDDEN hidden layers");
  if (c->obs_dim <= 0 || c->act_dim <= 0 || c->act_dim > SACX_MAX_ACT) return fail(SACX_ERR_INVALID, "obs_dim/act_dim out of range (act_dim <= 32)");
  if (c->batch_size <= 0 || c->n_agents <= 0) return fail(SACX_ERR_INVALID, "batch_size and n_agents must be positive");
  for (int i = 0; i < c->n_hidden_pi; ++i) if (c->hidden_pi[i] <= 0 || c->hidden_pi[i] > 8192) return fail(SACX_ERR_INVALID, "policy hidden size out of range");
  for (int i = 0; i < c->n_hidden_q; ++i) if (c->hidden_q[i] <= 0 || c->hidden_q[i] > 8192) return fail(SACX_ERR_INVALID, "q hidden size out of range");
  const int acts[4] = {c->act_hidden_pi, c->act_out_pi, c->act_hidden_q, c->act_out_q};
  for (int a : acts) if (a < 0 || a > SACX_ACT_SELU) return fail(SACX_ERR_ACTIVATION, "unknown activation id");
  if (!(c->alpha > 0.0)) return fail(SACX_ERR_INVALID, "alpha must be positive");
  if (c->n_step < 0 || c->n_step > 16) return fail(SACX_ERR_INVALID, "n_step out of range (0..16, 0 = 1)");
  return SACX_OK;
}

// ------------------------------------------------------------------------------------------ population-based training
// span 0 starts with the scalar block and runs through Adam v; span 1 holds the target critics (sacx_pbt.cuh)
static i64 pbt_span0(const Engine& e) { return e.P0 + 3 * e.blk - e.scal_off; }
static i64 pbt_span1(const Engine& e) { return align4(e.n_critic); }
static PbtEnd pbt_arena(const Engine& e) { return PbtEnd{e.arena, e.stride, e.scal_off, e.T0}; }
static PbtEnd pbt_buffer(const Engine& e, const float* buf) {
  return PbtEnd{const_cast<float*>(buf), pbt_span0(e) + pbt_span1(e), 0, pbt_span0(e)};
}

static int pbt_check_agents(const Engine& e, const int32_t* ids, int n, const char* what) {
  for (int i = 0; i < n; ++i)
    if (ids[i] < 0 || ids[i] >= e.cfg.n_agents)
      return fail(SACX_ERR_INVALID, std::string("pbt: ") + what + " agent " + std::to_string(ids[i]) + " out of range [0, " +
                                        std::to_string(e.cfg.n_agents) + ")");
  return SACX_OK;
}

static int pbt_check_destinations(const Engine& e, const int32_t* dst, int n, const int32_t* src /* nullable */) {
  std::vector<char> is_dst((size_t)e.cfg.n_agents, 0);
  for (int i = 0; i < n; ++i) {
    if (is_dst[dst[i]]) return fail(SACX_ERR_INVALID, "pbt: agent " + std::to_string(dst[i]) + " is a destination twice");
    is_dst[dst[i]] = 1;
  }
  if (src)
    for (int i = 0; i < n; ++i)
      if (is_dst[src[i]])
        return fail(SACX_ERR_INVALID, "pbt: agent " + std::to_string(src[i]) + " is both a source and a destination");
  return SACX_OK;
}

static int pbt_check_record(const Engine& e, const sacx_pbt_record& r) {
  const unsigned all = SACX_PBT_ALPHA | SACX_PBT_ALPHA_LR | SACX_PBT_ACTOR_LR | SACX_PBT_CRITIC_LR | SACX_PBT_TAU | SACX_PBT_GAMMA;
  auto pos = [](double x) { return x > 0.0 && std::isfinite(x); };
  if (r.set & ~all) return fail(SACX_ERR_INVALID, "pbt: unknown record bits");
  if (r.set & SACX_PBT_ALPHA) {
    if (e.cfg.auto_entropy_tuning)
      return fail(SACX_ERR_INVALID, "pbt: with auto_entropy_tuning the temperature is learner state; a record cannot set it");
    if (!pos(r.alpha) || !pos(r.alpha_f32) || !std::isfinite(r.log_alpha)) return fail(SACX_ERR_INVALID, "pbt: alpha must be positive and finite");
  }
  if ((r.set & SACX_PBT_ALPHA_LR) && !pos(r.alpha_lr)) return fail(SACX_ERR_INVALID, "pbt: alpha_lr must be positive and finite");
  if ((r.set & SACX_PBT_ACTOR_LR) && !pos(r.actor_lr)) return fail(SACX_ERR_INVALID, "pbt: actor_lr must be positive and finite");
  if ((r.set & SACX_PBT_CRITIC_LR) && !pos(r.critic_lr)) return fail(SACX_ERR_INVALID, "pbt: critic_lr must be positive and finite");
  if ((r.set & SACX_PBT_TAU) && !(pos(r.tau) && r.tau <= 1.f && r.one_minus_tau >= 0.f && r.one_minus_tau <= 1.f))
    return fail(SACX_ERR_INVALID, "pbt: tau must be in (0, 1]");
  if ((r.set & SACX_PBT_GAMMA) && !pos(r.gamma)) return fail(SACX_ERR_INVALID, "pbt: gamma must be positive and finite");
  return SACX_OK;
}

// validated pairs -> one pbt_copy_kernel launch on the agent's stream (the pair list goes up through a pinned block)
static int pbt_launch(Engine& e, const PbtEnd& src, const PbtEnd& dst, bool dst_arena, const int32_t* s, const int32_t* d, int n,
                      const sacx_pbt_record* rec) {
  if (n == 0) return SACX_OK;
  if (e.P0 != e.scal_off + SCAL_WORDS || ((uintptr_t)e.arena & 15))
    return fail(SACX_ERR_INVALID, "pbt: the arena does not hold the learner state as two 16-byte aligned spans");
  if (rec)
    for (int i = 0; i < n; ++i) {
      int rc = pbt_check_record(e, rec[i]);
      if (rc) return rc;
    }
  const size_t bytes = (size_t)n * sizeof(PbtPair);
  if (!e.pbt_copied) SACX_CUDA(cudaEventCreateWithFlags(&e.pbt_copied, cudaEventDisableTiming));
  SACX_CUDA(cudaEventSynchronize(e.pbt_copied));         // the previous pair list has left the pinned block
  if (bytes > e.pbt_bytes) {
    if (e.pbt_pinned) { cudaFreeHost(e.pbt_pinned); e.pbt_pinned = nullptr; }
    if (e.pbt_dev) { SACX_CUDA(cudaStreamSynchronize(e.stream)); cudaFree(e.pbt_dev); e.pbt_dev = nullptr; }
    e.pbt_bytes = 0;
    SACX_CUDA(cudaMallocHost(&e.pbt_pinned, bytes));
    SACX_CUDA(cudaMalloc(&e.pbt_dev, bytes));
    e.pbt_bytes = bytes;
  }
  PbtPair* p = static_cast<PbtPair*>(e.pbt_pinned);
  for (int i = 0; i < n; ++i) {
    memset(&p[i], 0, sizeof p[i]);
    p[i].src = s[i]; p[i].dst = d[i];
    if (rec) p[i].rec = rec[i];
  }
  SACX_CUDA(cudaMemcpyAsync(e.pbt_dev, e.pbt_pinned, bytes, cudaMemcpyHostToDevice, e.stream));
  SACX_CUDA(cudaEventRecord(e.pbt_copied, e.stream));
  const i64 n0 = pbt_span0(e) / 4, n1 = pbt_span1(e) / 4;
  const dim3 grid((unsigned)((n0 + n1 + PBT_CHUNK - 1) / PBT_CHUNK), (unsigned)std::min(n, 65535));
  pbt_copy_kernel<<<grid, PBT_THREADS, 0, e.stream>>>(src, dst, n0, n1, dst_arena ? 1 : 0, static_cast<const PbtPair*>(e.pbt_dev), n);
  ++e.launches;
  SACX_CUDA(cudaGetLastError());
  return SACX_OK;
}

}  // namespace sacx

using namespace sacx;

struct sacx_ring_s { Ring r; };
struct sacx_agent_s { Engine e; };
struct sacx_per_s { Per p; };

extern "C" {

const char* sacx_last_error(void) { return g_err.c_str(); }
int sacx_version(void) { return SACX_VERSION; }
int sacx_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
  return n;
}

int sacx_sizeof_config(void) { return (int)sizeof(sacx_config); }
int sacx_sizeof_metrics(void) { return (int)sizeof(sacx_metrics); }
int sacx_sizeof_tensor_desc(void) { return (int)sizeof(sacx_tensor_desc); }

int sacx_activation_id(const char* name) {
  if (!name) return SACX_ERR_ACTIVATION;
  static const char* names[] = {"identity", "relu", "tanh", "elu", "leaky_relu", "gelu", "selu"};
  for (int i = 0; i < 7; ++i) if (strcmp(name, names[i]) == 0) return i;
  return fail(SACX_ERR_ACTIVATION, std::string("unknown activation: ") + name);
}

// ---------------------------------------------------------------------------------------- ring API
int64_t sacx_ring_bytes(int32_t O, int32_t A, int64_t cap, int32_t n_agents) {
  i64 s, a, r, s2, d, total;
  Ring::offsets(O, A, cap, s, a, r, s2, d, total);
  return total * 4 * (int64_t)n_agents;
}

int sacx_ring_create(int32_t O, int32_t A, int64_t cap, int32_t n_agents, void* dev_mem, sacx_ring_t* out) {
  if (!out || O <= 0 || A <= 0 || cap <= 0 || n_agents <= 0) return fail(SACX_ERR_INVALID, "ring_create: bad arguments");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
    cudaGetLastError();
    return fail(SACX_ERR_CUDA, "no CUDA device: the replay ring is device-resident and has no CPU fallback");
  }
  sacx_ring_s* h = new sacx_ring_s();
  Ring& r = h->r;
  r.O = O; r.A = A; r.cap = cap; r.n_agents = n_agents; r.W = 2 * O + A + 2;
  i64 total;
  Ring::offsets(O, A, cap, r.off_s, r.off_a, r.off_r, r.off_s2, r.off_d, total);
  r.RS = Ring::record_floats(O, A);
  r.stride = total;
  r.pushes.assign(n_agents, 0);
  r.stage_limit = (int)std::min<i64>(STAGE_ROWS, cap);
  if (dev_mem) r.dev = (float*)dev_mem;
  else {
    SACX_CUDA(cudaMalloc((void**)&r.dev, (size_t)total * 4 * n_agents));
    r.own = true;
  }
  for (int ag = 0; ag < n_agents; ++ag) SACX_CUDA(cudaMemset(r.block(ag), 0, sizeof(RingMeta)));
  SACX_CUDA(cudaMallocHost((void**)&r.h_rows, (size_t)STAGE_ROWS * r.W * sizeof(float)));
  SACX_CUDA(cudaMallocHost((void**)&r.h_hdr, (size_t)STAGE_ROWS * sizeof(StageHdr)));
  SACX_CUDA(cudaMalloc((void**)&r.d_rows, (size_t)STAGE_ROWS * r.W * sizeof(float)));
  SACX_CUDA(cudaMalloc((void**)&r.d_hdr, (size_t)STAGE_ROWS * sizeof(StageHdr)));
  SACX_CUDA(cudaEventCreateWithFlags(&r.stage_free, cudaEventDisableTiming));
  *out = h;
  return SACX_OK;
}

int sacx_ring_destroy(sacx_ring_t h) {
  if (!h) return SACX_OK;
  Ring& r = h->r;
  cudaStreamSynchronize(r.stream);
  if (r.own && r.dev) cudaFree(r.dev);
  if (r.h_rows) cudaFreeHost(r.h_rows);
  if (r.h_hdr) cudaFreeHost(r.h_hdr);
  if (r.d_rows) cudaFree(r.d_rows);
  if (r.d_hdr) cudaFree(r.d_hdr);
  if (r.scr_dev) cudaFree(r.scr_dev);
  if (r.scr_host) cudaFreeHost(r.scr_host);
  if (r.stage_free) cudaEventDestroy(r.stage_free);
  delete h;
  return SACX_OK;
}

int sacx_ring_set_stream(sacx_ring_t h, void* stream) {
  if (!h) return fail(SACX_ERR_INVALID, "null ring");
  Ring& r = h->r;
  int rc = r.flush();
  if (rc) return rc;
  if ((cudaStream_t)stream != r.stream) {
    // work already queued on the old stream (the flush's scatter, earlier pushes) must be ordered before anything the new
    // stream does with the ring: record on the old stream, make the new one wait
    cudaEvent_t ev;
    SACX_CUDA(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
    SACX_CUDA(cudaEventRecord(ev, r.stream));
    SACX_CUDA(cudaStreamWaitEvent((cudaStream_t)stream, ev, 0));
    SACX_CUDA(cudaEventDestroy(ev));
  }
  r.stream = (cudaStream_t)stream;
  return SACX_OK;
}

int sacx_ring_push_host(sacx_ring_t h, int32_t agent, const float* s, const float* a, float reward, const float* s2, float done) {
  if (!h || !s || !a || !s2) return fail(SACX_ERR_INVALID, "ring_push: null pointer");
  return h->r.push(agent, s, a, reward, s2, done);
}

int sacx_ring_push_n_host(sacx_ring_t h, int32_t agent, int64_t n, const float* s, const float* a, const float* reward,
                          const float* s2, const float* done) {
  if (!h || !s || !a || !s2 || !reward || !done || n < 0) return fail(SACX_ERR_INVALID, "ring_push_n: bad arguments");
  Ring& r = h->r;
  for (int64_t i = 0; i < n; ++i) {
    int rc = r.push(agent, s + i * r.O, a + i * r.A, reward[i], s2 + i * r.O, done[i]);
    if (rc) return rc;
  }
  return SACX_OK;
}

int sacx_ring_push_n_dev(sacx_ring_t h, int32_t agent, int64_t n, const float* s, const float* a, const float* reward,
                         const float* s2, const float* done) {
  if (!h || !s || !a || !s2 || !reward || !done || n < 0) return fail(SACX_ERR_INVALID, "ring_push_n_dev: bad arguments");
  Ring& r = h->r;
  if (agent < 0 || agent >= r.n_agents) return fail(SACX_ERR_INVALID, "ring push: agent out of range");
  if (n > r.cap) return fail(SACX_ERR_INVALID, "ring_push_n_dev: n exceeds capacity");
  if (n == 0) return SACX_OK;
  int rc = r.flush();
  if (rc) return rc;
  ring_scatter_dev_kernel<<<(unsigned)((n + 7) / 8), 256, 0, r.stream>>>(r.block(agent), r.cap, r.off_s, r.off_a, r.off_r, r.off_s2,
                                                                         r.off_d, r.RS, r.O, r.A, s, a, reward, s2, done, r.pushes[agent], (int)n);
  ++r.launches;
  SACX_CUDA(cudaGetLastError());
  r.pushes[agent] += n;
  return SACX_OK;
}

int sacx_ring_flush(sacx_ring_t h) { return h ? h->r.flush() : fail(SACX_ERR_INVALID, "null ring"); }
int64_t sacx_ring_len(sacx_ring_t h, int32_t agent) { return (h && agent >= 0 && agent < h->r.n_agents) ? h->r.len(agent) : -1; }
int64_t sacx_ring_pushes(sacx_ring_t h, int32_t agent) { return (h && agent >= 0 && agent < h->r.n_agents) ? h->r.pushes[agent] : -1; }

// exact resume (SURVEY 8f-3): after the caller has copied a saved ring image back into the device block, re-derive the
// host-side push counters from the ring headers (RingMeta.pushes of every agent)
int sacx_ring_resync(sacx_ring_t h) {
  if (!h) return fail(SACX_ERR_INVALID, "null ring");
  Ring& r = h->r;
  int rc = r.flush();
  if (rc) return rc;
  SACX_CUDA(cudaStreamSynchronize(r.stream));
  for (int ag = 0; ag < r.n_agents; ++ag) {
    RingMeta m;
    SACX_CUDA(cudaMemcpy(&m, r.dev + (i64)ag * r.stride, sizeof m, cudaMemcpyDeviceToHost));
    if (m.pushes < 0) return fail(SACX_ERR_INVALID, "ring_resync: corrupt ring header");
    r.pushes[ag] = m.pushes;
  }
  return SACX_OK;
}

// rollout-noise counter of the engine (device Philox stream of sacx_act): part of an exact-resume snapshot
int64_t sacx_agent_act_counter(sacx_agent_t h, int64_t set_to) {
  if (!h) return -1;
  if (set_to >= 0) h->e.act_calls = (unsigned long long)set_to;
  return (int64_t)h->e.act_calls;
}

int sacx_ring_gather(sacx_ring_t h, int32_t agent, const int64_t* idx_dev, int32_t B, float* s, float* a, float* rr, float* s2, float* d) {
  if (!h || !idx_dev || B <= 0) return fail(SACX_ERR_INVALID, "ring_gather: bad arguments");
  Ring& r = h->r;
  if (agent < 0 || agent >= r.n_agents) return fail(SACX_ERR_INVALID, "ring_gather: agent out of range");
  if (r.len(agent) < B)
    return fail(SACX_ERR_UNDERFILLED, "Not enough samples in the replay buffer to sample " + std::to_string(B) +
                                          " transitions. Current size: " + std::to_string(r.len(agent)));
  int rc = r.flush();
  if (rc) return rc;
  auto al16 = [](const void* p) { return (((uintptr_t)p) & 15) == 0; };
  const bool vec = (r.O % 4 == 0) && (r.A % 4 == 0) && al16(r.block(agent)) && al16(s) && al16(s2) && al16(a) && r.RS / 4 <= 256;
  if (vec) {
    const int pieces = r.RS / 4;                // 16-byte pieces of a packed record (the last one holds r, d)
    int tl = 0;
    while ((1 << tl) < pieces) ++tl;
    const i64 threads = (i64)((B + 1) / 2) << tl;     // two rows per thread
    const i64 pushes = r.pushes[agent];               // everything staged was flushed above: the device header holds the same count
    const i64 oldest_slot = pushes > r.cap ? (pushes - r.cap) % r.cap : 0;
    ring_gather_vec_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, r.stream>>>(r.block(agent), r.cap, oldest_slot, std::min(pushes, r.cap), r.off_s,
                                                                                    r.RS, r.O, r.A, (const i64*)idx_dev, B, s, a, rr, s2, d, tl);
  } else {
    ring_gather_kernel<<<(B + 7) / 8, 256, 0, r.stream>>>(r.block(agent), r.cap, r.off_s, r.off_a, r.off_r, r.off_s2, r.off_d, r.RS, r.O, r.A,
                                                          (const i64*)idx_dev, B, s, a, rr, s2, d);
  }
  ++r.launches;
  SACX_CUDA(cudaGetLastError());
  return SACX_OK;
}

int sacx_ring_gather_host(sacx_ring_t h, int32_t agent, const int64_t* idx, int32_t B, float* s, float* a, float* rr, float* s2, float* d) {
  if (!h || !idx || B <= 0) return fail(SACX_ERR_INVALID, "ring_gather_host: bad arguments");
  Ring& r = h->r;
  if (agent < 0 || agent >= r.n_agents) return fail(SACX_ERR_INVALID, "ring_gather: agent out of range");
  const i64 n = r.len(agent);
  if (n < B)
    return fail(SACX_ERR_UNDERFILLED, "Not enough samples in the replay buffer to sample " + std::to_string(B) +
                                          " transitions. Current size: " + std::to_string(n));
  for (int i = 0; i < B; ++i)
    if (idx[i] < 0 || idx[i] >= n) return fail(SACX_ERR_INVALID, "ring_gather_host: logical index out of range");
  const size_t rowf = (size_t)r.W;
  const size_t bytes = (size_t)B * (sizeof(i64) + rowf * sizeof(float));
  int rc = r.ensure_scratch(bytes);
  if (rc) return rc;
  i64* d_idx = (i64*)r.scr_dev;
  float* d_out = (float*)((char*)r.scr_dev + (size_t)B * sizeof(i64));
  float* ds = d_out, *da = ds + (size_t)B * r.O, *dr = da + (size_t)B * r.A, *ds2 = dr + B, *dd = ds2 + (size_t)B * r.O;
  memcpy(r.scr_host, idx, (size_t)B * sizeof(i64));
  SACX_CUDA(cudaMemcpyAsync(d_idx, r.scr_host, (size_t)B * sizeof(i64), cudaMemcpyHostToDevice, r.stream));
  rc = sacx_ring_gather(h, agent, (const int64_t*)d_idx, B, ds, da, dr, ds2, dd);
  if (rc) return rc;
  float* hout = (float*)((char*)r.scr_host + (size_t)B * sizeof(i64));
  SACX_CUDA(cudaMemcpyAsync(hout, d_out, (size_t)B * rowf * sizeof(float), cudaMemcpyDeviceToHost, r.stream));
  SACX_CUDA(cudaStreamSynchronize(r.stream));
  const float* hs = hout, *ha = hs + (size_t)B * r.O, *hr = ha + (size_t)B * r.A, *hs2 = hr + B, *hd = hs2 + (size_t)B * r.O;
  if (s) memcpy(s, hs, (size_t)B * r.O * 4);
  if (a) memcpy(a, ha, (size_t)B * r.A * 4);
  if (rr) memcpy(rr, hr, (size_t)B * 4);
  if (s2) memcpy(s2, hs2, (size_t)B * r.O * 4);
  if (d) memcpy(d, hd, (size_t)B * 4);
  return SACX_OK;
}

// Host helper of the reference-stream index draw (random.sample(range(n), k) on CPython's Mersenne Twister): the binding
// fetches the generator's raw 32-bit words in bulk (random.getrandbits(32 * w)) and this routine applies the stdlib's
// accept/reject rule to them in order -- keep the top `bits` bits of a word, reject values >= n and values already
// selected (Lib/random.py: sample(), set-based branch; _randbelow_with_getrandbits) -- appending to out[have..k).
// Returns the new number of selected positions. Plain host code: no device is touched.
int32_t sacx_index_filter(const uint32_t* words, int32_t n_words, uint64_t n, int32_t bits, int64_t* out, int32_t have, int32_t k) {
  if (!words || !out || n_words < 0 || have < 0 || k < have || bits < 1 || bits > 32) return -1;
  static thread_local std::vector<int64_t> table;
  size_t cap = 64;
  while (cap < (size_t)k * 4) cap <<= 1;
  table.assign(cap, -1);
  auto slot_of = [&](int64_t v) { return (size_t)((uint64_t)v * 0x9E3779B97F4A7C15ull >> 17) & (cap - 1); };
  auto insert = [&](int64_t v) -> bool {          // false when v is already present
    size_t s = slot_of(v);
    while (table[s] >= 0) { if (table[s] == v) return false; s = (s + 1) & (cap - 1); }
    table[s] = v;
    return true;
  };
  for (int32_t i = 0; i < have; ++i) insert(out[i]);
  const int shift = 32 - bits;
  for (int32_t i = 0; i < n_words && have < k; ++i) {
    const uint64_t v = (uint64_t)(words[i] >> shift);
    if (v >= n) continue;
    if (insert((int64_t)v)) out[have++] = (int64_t)v;
  }
  return have;
}

int sacx_ring_sample_indices(sacx_ring_t h, int32_t agent, uint64_t seed, uint64_t counter, int32_t B, int64_t* out_dev) {
  if (!h || !out_dev || B <= 0) return fail(SACX_ERR_INVALID, "ring_sample_indices: bad arguments");
  Ring& r = h->r;
  if (agent < 0 || agent >= r.n_agents) return fail(SACX_ERR_INVALID, "agent out of range");
  if (r.len(agent) < B)
    return fail(SACX_ERR_UNDERFILLED, "Not enough samples in the replay buffer to sample " + std::to_string(B) +
                                          " transitions. Current size: " + std::to_string(r.len(agent)));
  int rc = r.flush();
  if (rc) return rc;
  ring_indices_kernel<<<(B + 255) / 256, 256, 0, r.stream>>>(r.block(agent), r.cap, seed, counter, agent, B, (i64*)out_dev);
  ++r.launches;
  SACX_CUDA(cudaGetLastError());
  return SACX_OK;
}

// ---------------------------------------------------------------------------------------- DonkeyVae observation assembly
struct sacx_obs_s {
  int z = 0, n_cmd = 0, n_hist = 0, n_stack = 0, F = 0, S = 0;
  float* dev = nullptr;          // [hist H | stack S | prev S | act n_cmd | r, d]
  float* hist() { return dev; }
  float* stack() { return dev + n_cmd * n_hist; }
  float* prev() { return stack() + S; }
  float* act() { return prev() + S; }
  float* rd() { return act() + n_cmd; }
};

int sacx_obs_create(int32_t z_size, int32_t n_commands, int32_t n_command_history, int32_t n_stack, sacx_obs_t* out) {
  if (!out || z_size <= 0 || n_commands <= 0 || n_command_history < 0 || n_stack < 1) return fail(SACX_ERR_INVALID, "obs_create: bad arguments");
  sacx_obs_s* h = new sacx_obs_s();
  h->z = z_size; h->n_cmd = n_commands; h->n_hist = n_command_history; h->n_stack = n_stack;
  h->F = z_size + n_commands * n_command_history; h->S = h->F * n_stack;
  if ((size_t)(n_commands * n_command_history + h->S) * 4 > 40000) { delete h; return fail(SACX_ERR_INVALID, "obs_create: observation too wide"); }
  const size_t floats = (size_t)n_commands * n_command_history + 2 * (size_t)h->S + n_commands + 2;
  if (cudaMalloc((void**)&h->dev, floats * 4) != cudaSuccess) { delete h; return fail(SACX_ERR_CUDA, "obs_create: cudaMalloc failed"); }
  cudaMemset(h->dev, 0, floats * 4);
  *out = h;
  return SACX_OK;
}
int sacx_obs_destroy(sacx_obs_t h) {
  if (!h) return SACX_OK;
  if (h->dev) cudaFree(h->dev);
  delete h;
  return SACX_OK;
}
int32_t sacx_obs_dim(sacx_obs_t h) { return h ? h->S : 0; }

static int obs_launch(sacx_obs_t h, const float* latent, const float* action_dev, float a0, float a1, float reward, int done, int reset,
                      cudaStream_t st) {
  const size_t smem = (size_t)(h->n_cmd * h->n_hist + h->S) * 4;
  obs_assemble_kernel<<<1, 256, smem, st>>>(h->hist(), h->stack(), h->prev(), reset ? nullptr : h->act(), reset ? nullptr : h->rd(), latent,
                                            action_dev, a0, a1, reward, done, reset, h->z, h->n_cmd, h->n_hist, h->n_stack);
  SACX_CUDA(cudaGetLastError());
  return SACX_OK;
}

int sacx_obs_reset(sacx_obs_t h, const float* latent_dev, float* obs_out_dev, void* stream) {
  if (!h || !latent_dev) return fail(SACX_ERR_INVALID, "obs_reset: bad arguments");
  int rc = obs_launch(h, latent_dev, nullptr, 0.f, 0.f, 0.f, 0, 1, (cudaStream_t)stream);
  if (rc) return rc;
  if (obs_out_dev) SACX_CUDA(cudaMemcpyAsync(obs_out_dev, h->stack(), (size_t)h->S * 4, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
  return SACX_OK;
}

int sacx_obs_step(sacx_obs_t h, const float* latent_dev, const float* action_dev, const float* action_host, float reward, int32_t done,
                  sacx_ring_t ring, int32_t agent, float* obs_out_dev, void* stream) {
  if (!h || !latent_dev || (!action_dev && !action_host)) return fail(SACX_ERR_INVALID, "obs_step: bad arguments");
  if (!action_dev && h->n_cmd > 2) return fail(SACX_ERR_INVALID, "obs_step: host actions carry at most 2 commands");
  cudaStream_t st = ring ? ring->r.stream : (cudaStream_t)stream;
  if (ring && (ring->r.O != h->S || ring->r.A != h->n_cmd)) return fail(SACX_ERR_INVALID, "obs_step: ring dimensions do not match the assembled observation");
  const float a0 = action_host ? action_host[0] : 0.f, a1 = (action_host && h->n_cmd > 1) ? action_host[1] : 0.f;
  int rc = obs_launch(h, latent_dev, action_dev, a0, a1, reward, done, 0, st);
  if (rc) return rc;
  if (ring) {        // (previous stack, action, reward, new stack, done): straight from device staging into the ring
    rc = sacx_ring_push_n_dev(ring, agent, 1, h->prev(), h->act(), h->rd(), h->stack(), h->rd() + 1);
    if (rc) return rc;
  }
  if (obs_out_dev) SACX_CUDA(cudaMemcpyAsync(obs_out_dev, h->stack(), (size_t)h->S * 4, cudaMemcpyDeviceToDevice, st));
  return SACX_OK;
}

// ---------------------------------------------------------------------------------------- agent API
int sacx_agent_arena_floats(const sacx_config* cfg, int64_t* out) {
  int rc = validate(cfg);
  if (rc) return rc;
  if (!out) return fail(SACX_ERR_INVALID, "null out");
  Engine e;
  e.cfg = *cfg;
  e.build_layout();
  *out = e.stride;
  return SACX_OK;
}

// (error paths of create release whatever was allocated so far through the one destroy routine)
int sacx_agent_create(const sacx_config* cfg, float* arena_dev, sacx_agent_t* out) {
  int rc = validate(cfg);
  if (rc) return rc;
  if (!out) return fail(SACX_ERR_INVALID, "null out");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
    cudaGetLastError();
    return fail(SACX_ERR_CUDA, "no CUDA device: the SAC update engine is CUDA-only (sm_100a) and has no CPU fallback");
  }
  sacx_agent_s* h = new sacx_agent_s();
  Engine& e = h->e;
  e.cfg = *cfg;
  if (e.cfg.dp_world <= 0) { e.cfg.dp_world = 1; e.cfg.dp_rank = 0; }
  { const char* mb = getenv("SACX_TC_MIN_BATCH"); if (mb && atoi(mb) > 0) e.tc_min_batch = atoi(mb); }
  e.tc_min_m = e.cfg.n_agents > 1 ? 128 : e.tc_min_batch;
  { const char* rt = getenv("SACX_RP_TMA"); if (rt && atoi(rt) == 0) e.rp_tma = false; }
  int dev = 0;
  SACX_CUDA(cudaGetDevice(&dev));
  SACX_CUDA(cudaDeviceGetAttribute(&e.n_sms, cudaDevAttrMultiProcessorCount, dev));
  const char* tile_env = getenv("SACX_TILE");
  e.large = (cfg->n_agents > 1) || (cfg->batch_size >= 1024);
  if (tile_env && !strcmp(tile_env, "small")) e.large = false;
  if (tile_env && !strcmp(tile_env, "large")) e.large = true;
  e.build_layout();
  Hyper& hp = e.hp;
  memset(&hp, 0, sizeof hp);
  hp.gamma = (float)cfg->gamma; hp.tau = (float)cfg->tau; hp.one_minus_tau = (float)(1.0 - cfg->tau);
  hp.log_std_min = cfg->log_std_min; hp.log_std_max = cfg->log_std_max; hp.action_scale = cfg->action_scale;
  hp.lr[OPT_PI] = cfg->actor_lr; hp.lr[OPT_Q1] = hp.lr[OPT_Q2] = cfg->critic_lr;
  hp.alpha_lr = cfg->alpha_lr; hp.alpha_init = cfg->alpha;
  hp.target_entropy = -(float)cfg->act_dim;                 // agent.py:43
  hp.auto_alpha = cfg->auto_entropy_tuning;
  hp.obs = cfg->obs_dim; hp.act = cfg->act_dim; hp.B = cfg->batch_size;
  hp.B_global = cfg->batch_size * e.cfg.dp_world; hp.row0_global = cfg->batch_size * e.cfg.dp_rank;
  hp.n_step = cfg->n_step > 0 ? cfg->n_step : 1;
  hp.seed = cfg->seed;
  if ((rc = e.build_plans())) { sacx_agent_destroy(h); return rc; }
  if ((rc = engine_setup_rp(&e))) { sacx_agent_destroy(h); return rc; }
  // launch geometry: one CTA per SM; a single agent spreads over the chip, a population gets one CTA per agent
  const size_t gemm_floats = e.large ? CfgLarge::SMEM_FLOATS : CfgSmall::SMEM_FLOATS;
  e.smem_bytes = (int)(SMEM_OPS * sizeof(Op) + WSM_FLOATS * 4 + gemm_floats * 4);
  const void* fn = e.large ? (const void*)sacx_run_kernel<true> : (const void*)sacx_run_kernel<false>;
  SACX_CUDA(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, e.smem_bytes));
  int per_sm = 0;
  if (e.large) SACX_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, sacx_run_kernel<true>, 256, e.smem_bytes));
  else SACX_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, sacx_run_kernel<false>, 256, e.smem_bytes));
  if (per_sm < 1) { sacx_agent_destroy(h); return fail(SACX_ERR_CUDA, "update kernel does not fit on an SM"); }
  e.max_ctas = e.n_sms;                                      // one CTA per SM (persistent)
  if (cfg->n_agents == 1) {
    e.grid_x = cfg->ctas_per_agent > 0 ? cfg->ctas_per_agent : std::min(e.max_ctas, e.max_phase_tiles());
    e.grid_x = std::max(1, std::min(e.grid_x, e.max_ctas));
    e.grid_y = 1;
  } else {
    e.grid_x = std::max(1, std::min(cfg->ctas_per_agent > 0 ? cfg->ctas_per_agent : 1, e.max_ctas));
    e.grid_y = std::max(1, std::min(cfg->n_agents, e.max_ctas / e.grid_x));
  }
  const size_t total = (size_t)e.stride * 4 * cfg->n_agents;
  if (arena_dev) e.arena = arena_dev;
  else {
    SACX_CUDA(cudaMalloc((void**)&e.arena, total));
    SACX_CUDA(cudaMemset(e.arena, 0, total));
    e.own_arena = true;
  }
  {
    std::string w;
    const bool planned = e.tc_wanted(w);
    if ((rc = engine_setup_tc(&e))) { sacx_agent_destroy(h); return rc; }
    if (planned && !e.tc) {            // the plans were built for the tensor-core path (head GEMMs, tails, projections): rebuild without
      e.tc_forbid = true;
      if ((rc = e.build_plans())) { sacx_agent_destroy(h); return rc; }
      if ((rc = engine_setup_rp(&e))) { sacx_agent_destroy(h); return rc; }
    }
  }
  if ((rc = engine_setup_rp_tma(&e))) { sacx_agent_destroy(h); return rc; }
  SACX_CUDA(cudaMalloc((void**)&e.d_plans, sizeof(Plan) * N_PLANS));
  SACX_CUDA(cudaMemcpy(e.d_plans, e.h_plans.data(), sizeof(Plan) * N_PLANS, cudaMemcpyHostToDevice));
  SACX_CUDA(cudaMalloc((void**)&e.d_barrier, sizeof(unsigned) * 64 * 4096));
  SACX_CUDA(cudaMemset(e.d_barrier, 0, sizeof(unsigned) * 64 * 4096));
  SACX_CUDA(cudaMallocHost((void**)&e.pinned_metrics, sizeof(sacx_metrics)));
  if ((rc = engine_init_scalars(&e))) { sacx_agent_destroy(h); return rc; }
  *out = h;
  return SACX_OK;
}

int sacx_agent_destroy(sacx_agent_t h) {
  if (!h) return SACX_OK;
  Engine& e = h->e;
  if (e.per) { e.per->flush(); e.per->agent = nullptr; }     // the pending write-back reads this arena
  cudaStreamSynchronize(e.stream);
  if (e.own_arena && e.arena) cudaFree(e.arena);
  if (e.d_plans) cudaFree(e.d_plans);
  if (e.d_prog) cudaFree(e.d_prog);
  if (e.d_rp_part) cudaFree(e.d_rp_part);
  if (e.d_rp_maps) cudaFree(e.d_rp_maps);
  if (e.d_tc_scratch) cudaFree(e.d_tc_scratch);
  if (e.d_barrier) cudaFree(e.d_barrier);
  if (e.pinned_metrics) cudaFreeHost(e.pinned_metrics);
  if (e.pinned_io) cudaFreeHost(e.pinned_io);
  if (e.dev_io) cudaFree(e.dev_io);
  for (auto& io : e.slots) {
    if (io.pinned) cudaFreeHost(io.pinned); if (io.dev) cudaFree(io.dev); if (io.done) cudaEventDestroy(io.done); if (io.copied) cudaEventDestroy(io.copied);
  }
  if (e.copy_stream) cudaStreamDestroy(e.copy_stream);
  if (e.pbt_pinned) cudaFreeHost(e.pbt_pinned);
  if (e.pbt_dev) cudaFree(e.pbt_dev);
  if (e.pbt_copied) cudaEventDestroy(e.pbt_copied);
  delete h;
  return SACX_OK;
}

int sacx_agent_set_stream(sacx_agent_t h, void* stream) {
  if (!h) return fail(SACX_ERR_INVALID, "null agent");
  Engine& e = h->e;
  if ((cudaStream_t)stream != e.stream) {       // updates queued on the old stream come first
    cudaEvent_t ev;
    SACX_CUDA(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
    SACX_CUDA(cudaEventRecord(ev, e.stream));
    SACX_CUDA(cudaStreamWaitEvent((cudaStream_t)stream, ev, 0));
    SACX_CUDA(cudaEventDestroy(ev));
  }
  e.stream = (cudaStream_t)stream;
  return SACX_OK;
}
int sacx_agent_attach_ring(sacx_agent_t h, sacx_ring_t r) {
  if (!h) return fail(SACX_ERR_INVALID, "null agent");
  if (r) {
    if (r->r.O != h->e.cfg.obs_dim || r->r.A != h->e.cfg.act_dim) return fail(SACX_ERR_INVALID, "ring/agent dimension mismatch");
    if (r->r.n_agents != h->e.cfg.n_agents) return fail(SACX_ERR_INVALID, "ring/agent population mismatch");
  }
  h->e.ring = r ? &r->r : nullptr;
  return SACX_OK;
}
float* sacx_agent_arena(sacx_agent_t h) { return h ? h->e.arena : nullptr; }
int64_t sacx_agent_stride(sacx_agent_t h) { return h ? h->e.stride : 0; }

int sacx_agent_layout(sacx_agent_t h, sacx_tensor_desc* out, int32_t capacity, int32_t* n_out) {
  if (!h || !n_out) return fail(SACX_ERR_INVALID, "layout: bad arguments");
  const auto& lay = h->e.lay;
  *n_out = (int32_t)lay.size();
  if (out) for (int i = 0; i < (int)lay.size() && i < capacity; ++i) out[i] = lay[i];
  return SACX_OK;
}

int sacx_agent_grid(sacx_agent_t h, int32_t* gx, int32_t* gy, int32_t* smem) {
  if (!h) return fail(SACX_ERR_INVALID, "null agent");
  if (gx) *gx = h->e.rp ? h->e.rp_grid : h->e.grid_x;
  if (gy) *gy = h->e.grid_y;
  if (smem) *smem = h->e.rp ? h->e.rp_smem_bytes : h->e.smem_bytes;
  return SACX_OK;
}

int sacx_agent_path(sacx_agent_t h, char* reason, int32_t capacity) {
  if (!h) return fail(SACX_ERR_INVALID, "null agent");
  if (reason && capacity > 0) snprintf(reason, (size_t)capacity, "%s", h->e.rp ? "" : h->e.rp_why.c_str());
  return h->e.rp ? 1 : 0;
}

int sacx_agent_tc(sacx_agent_t h, char* reason, int32_t capacity, int64_t* tc_launches) {
  if (!h) return fail(SACX_ERR_INVALID, "null agent");
  if (reason && capacity > 0) snprintf(reason, (size_t)capacity, "%s", h->e.tc ? "" : h->e.tc_why.c_str());
  if (tc_launches) *tc_launches = h->e.tc_launches;
  return h->e.tc ? 1 : 0;
}

int sacx_agent_reset_state(sacx_agent_t h) {
  if (!h) return fail(SACX_ERR_INVALID, "null agent");
  Engine& e = h->e;
  for (int ag = 0; ag < e.cfg.n_agents; ++ag) {
    float* base = e.arena + (i64)ag * e.stride;
    SACX_CUDA(cudaMemcpyAsync(base + e.T0, base + e.q1.begin, (size_t)e.n_critic * 4, cudaMemcpyDeviceToDevice, e.stream));
    SACX_CUDA(cudaMemsetAsync(base + e.P0 + e.blk, 0, (size_t)e.blk * 3 * 4, e.stream));
  }
  return engine_init_scalars(&e);
}

int sacx_agent_refresh_alpha(sacx_agent_t h) {
  if (!h) return fail(SACX_ERR_INVALID, "null agent");
  Engine& e = h->e;
  SACX_CUDA(cudaStreamSynchronize(e.stream));
  for (int ag = 0; ag < e.cfg.n_agents; ++ag) {
    AgentScalars s;
    float* p = e.arena + (i64)ag * e.stride + e.scal_off;
    SACX_CUDA(cudaMemcpy(&s, p, sizeof s, cudaMemcpyDeviceToHost));
    if (e.cfg.auto_entropy_tuning) s.alpha = std::exp(s.log_alpha);
    s.alpha_f32 = (float)s.alpha;
    s.metrics[4] = (float)s.alpha; s.metrics[5] = (float)s.log_alpha;
    SACX_CUDA(cudaMemcpy(p, &s, sizeof s, cudaMemcpyHostToDevice));
  }
  return SACX_OK;
}

static int need_ring(Engine& e, bool device_sampling) {
  if (!e.ring) return fail(SACX_ERR_INVALID, "no replay ring attached to the agent");
  for (int ag = 0; ag < e.cfg.n_agents; ++ag)
    if (e.ring->len(ag) < (i64)e.cfg.batch_size * (device_sampling ? e.cfg.dp_world : 1))
      return fail(SACX_ERR_UNDERFILLED, "Not enough samples in the replay buffer to sample " + std::to_string(e.cfg.batch_size) +
                                            " transitions. Current size: " + std::to_string(e.ring->len(ag)));
  int rc = e.ring->flush();
  if (rc) return rc;
  if (e.ring->stream != e.stream) {   // order the ring's writes before the update
    SACX_CUDA(cudaStreamSynchronize(e.ring->stream));
  }
  return SACX_OK;
}

static int do_update(sacx_agent_t h, const int64_t* idx, const float* e1, const float* e2, int n_steps, bool staged) {
  if (!h || n_steps <= 0) return fail(SACX_ERR_INVALID, "update: bad arguments");
  Engine& e = h->e;
  int rc = need_ring(e, idx == nullptr);
  if (rc) return rc;
  RunArgs a;
  memset(&a, 0, sizeof a);
  if (e.per) {
    // prioritized replay: per update, one tree launch (deferred write-back of the previous update + new pushes + sample of
    // this batch and its weights), then the update itself with n_steps = 1; this update's write-back is left pending
    if (idx) return fail(SACX_ERR_INVALID, "update: a prioritized replay tree is attached; it samples the batch (pass idx = NULL)");
    if (staged) return fail(SACX_ERR_INVALID, "sacx_update_staged does not support prioritized replay");
    Per& p = *e.per;
    const i64 nba = (i64)e.cfg.batch_size * e.cfg.act_dim;
    for (int s = 0; s < n_steps; ++s) {
      PerArgs pa = p.base();
      pa.B = e.cfg.batch_size; pa.scal = reinterpret_cast<const AgentScalars*>(e.arena + e.scal_off);
      pa.out_idx = p.d_idx; pa.out_w = p.d_w; pa.out_slots = p.d_slots;
      if ((rc = p.run(pa))) return rc;
      a.idx_ext = p.d_idx; a.w_ext = p.d_w;
      a.eps1_ext = e1 ? e1 + s * nba : nullptr; a.eps2_ext = e2 ? e2 + s * nba : nullptr;
      if ((rc = e.rp ? engine_launch_rp(&e, 1, a) : engine_launch(&e, PLAN_FUSED, 0, -1, 1, a, false))) return rc;
      p.pend_n = e.cfg.batch_size;
      p.pend_q1 = e.arena + e.b_q[0]; p.pend_q2 = e.arena + e.b_q[1]; p.pend_y = e.arena + e.b_y;
    }
    return SACX_OK;
  }
  a.idx_ext = (const i64*)idx; a.eps1_ext = e1; a.eps2_ext = e2;
  if (e.rp && !staged) return engine_launch_rp(&e, n_steps, a);
  return engine_launch(&e, PLAN_FUSED, 0, -1, n_steps, a, staged);
}

int sacx_update(sacx_agent_t h, const int64_t* idx, const float* e1, const float* e2, int32_t n_steps) {
  return do_update(h, idx, e1, e2, n_steps, false);
}
int sacx_update_staged(sacx_agent_t h, const int64_t* idx, const float* e1, const float* e2, int32_t n_steps) {
  return do_update(h, idx, e1, e2, n_steps, true);
}

static int read_metrics(Engine& e, int agent, sacx_metrics* out) {
  AgentScalars s;
  SACX_CUDA(cudaMemcpyAsync(e.pinned_io ? e.pinned_io : (void*)&s, e.arena + (i64)agent * e.stride + e.scal_off, sizeof s,
                            cudaMemcpyDeviceToHost, e.stream));
  SACX_CUDA(cudaStreamSynchronize(e.stream));
  if (e.pinned_io) memcpy(&s, e.pinned_io, sizeof s);
  out->q1_loss = s.metrics[0]; out->q2_loss = s.metrics[1]; out->policy_loss = s.metrics[2]; out->alpha_loss = s.metrics[3];
  out->alpha = s.metrics[4]; out->log_alpha = s.metrics[5]; out->q1_mean = s.metrics[6]; out->q2_mean = s.metrics[7];
  out->logpi_mean = s.metrics[8]; out->y_mean = s.metrics[9];
  out->nonfinite = s.nonfinite; out->reserved = 0; out->updates = s.updates;
  return SACX_OK;
}

static int ensure_io(Engine& e, size_t bytes) {
  bytes = std::max(bytes, sizeof(AgentScalars));
  if (bytes > e.pinned_io_bytes) {
    if (e.pinned_io) cudaFreeHost(e.pinned_io);
    if (e.dev_io) cudaFree(e.dev_io);
    e.pinned_io = e.dev_io = nullptr;
    e.pinned_io_bytes = e.dev_io_bytes = 0;
    SACX_CUDA(cudaMallocHost(&e.pinned_io, bytes));
    SACX_CUDA(cudaMalloc(&e.dev_io, bytes));
    e.pinned_io_bytes = e.dev_io_bytes = bytes;
  }
  return SACX_OK;
}

// Two staging slots (pinned host + device + event) so that the host can prepare update t+1 while update t runs.
static int host_update_submit(Engine& e, int slot, const int64_t* idx, const float* e1, const float* e2, int n_steps) {
  Engine::IoSlot& io = e.slots[slot];
  const size_t nb = (size_t)n_steps * e.cfg.n_agents * e.cfg.batch_size;
  const size_t b_idx = idx ? nb * sizeof(i64) : 0;
  const size_t b_eps = nb * e.cfg.act_dim * sizeof(float);
  const size_t total = b_idx + (e1 ? b_eps : 0) + (e2 ? b_eps : 0) + sizeof(AgentScalars) + 256;
  if (io.busy) { SACX_CUDA(cudaEventSynchronize(io.done)); io.busy = false; }
  if (total > io.bytes) {
    if (io.pinned) cudaFreeHost(io.pinned);
    if (io.dev) cudaFree(io.dev);
    io.pinned = io.dev = nullptr; io.bytes = 0;
    SACX_CUDA(cudaMallocHost(&io.pinned, total));
    SACX_CUDA(cudaMalloc(&io.dev, total));
    io.bytes = total;
  }
  if (!io.done) SACX_CUDA(cudaEventCreateWithFlags(&io.done, cudaEventDisableTiming));
  if (!io.copied) SACX_CUDA(cudaEventCreateWithFlags(&io.copied, cudaEventDisableTiming));
  if (!e.copy_stream) SACX_CUDA(cudaStreamCreateWithFlags(&e.copy_stream, cudaStreamNonBlocking));
  char* hp = (char*)io.pinned;
  char* dp = (char*)io.dev;
  size_t off = 0;
  const i64* d_idx = nullptr; const float* d_e1 = nullptr; const float* d_e2 = nullptr;
  if (idx) { memcpy(hp + off, idx, b_idx); d_idx = (const i64*)(dp + off); off += b_idx; }
  if (e1) { memcpy(hp + off, e1, b_eps); d_e1 = (const float*)(dp + off); off += b_eps; }
  if (e2) { memcpy(hp + off, e2, b_eps); d_e2 = (const float*)(dp + off); off += b_eps; }
  int rc = need_ring(e, idx == nullptr);
  if (rc) return rc;
  io.metrics_off = (off + 255) & ~(size_t)255;
  RunArgs a;
  memset(&a, 0, sizeof a);
  a.idx_ext = d_idx; a.eps1_ext = d_e1; a.eps2_ext = d_e2;
  const bool direct_metrics = e.rp;          // the row-parallel kernel writes the metrics block into the pinned slot itself
  if (direct_metrics) a.metrics_host = reinterpret_cast<float*>(hp + io.metrics_off);
  // The H2D copy goes on its own stream: the slot's device buffer is free (its previous kernel completed: io.done above), so the
  // copy of step t+1 overlaps the kernel of step t instead of sitting between two kernels on one stream (~10 us per step at
  // batch 256); the kernel waits for io.copied.
  if (off) {
    if (cudaMemcpyAsync(dp, hp, off, cudaMemcpyHostToDevice, e.copy_stream) != cudaSuccess) return fail(SACX_ERR_CUDA, "update_host: H2D copy failed");
    if (cudaEventRecord(io.copied, e.copy_stream) != cudaSuccess || cudaStreamWaitEvent(e.stream, io.copied, 0) != cudaSuccess)
      return fail(SACX_ERR_CUDA, "update_host: H2D copy ordering failed");
  }
  rc = e.rp ? engine_launch_rp(&e, n_steps, a) : engine_launch(&e, PLAN_FUSED, 0, -1, n_steps, a, false);
  if (rc) return rc;
  // the step's result travels back right behind the kernel (metrics block of agent 0)
  if (!direct_metrics &&
      cudaMemcpyAsync(hp + io.metrics_off, e.arena + e.scal_off, sizeof(AgentScalars), cudaMemcpyDeviceToHost, e.stream) != cudaSuccess)
    return fail(SACX_ERR_CUDA, "update_host: metrics D2H copy failed");
  SACX_CUDA(cudaEventRecord(io.done, e.stream));
  io.busy = true;
  return SACX_OK;
}

static int host_update_collect(Engine& e, int slot, sacx_metrics* out) {
  Engine::IoSlot& io = e.slots[slot];
  if (!io.pinned) return fail(SACX_ERR_INVALID, "no update was submitted on this slot");
  if (io.busy) { SACX_CUDA(cudaEventSynchronize(io.done)); io.busy = false; }
  if (out) {
    AgentScalars s;
    memcpy(&s, (char*)io.pinned + io.metrics_off, sizeof s);
    out->q1_loss = s.metrics[0]; out->q2_loss = s.metrics[1]; out->policy_loss = s.metrics[2]; out->alpha_loss = s.metrics[3];
    out->alpha = s.metrics[4]; out->log_alpha = s.metrics[5]; out->q1_mean = s.metrics[6]; out->q2_mean = s.metrics[7];
    out->logpi_mean = s.metrics[8]; out->y_mean = s.metrics[9];
    out->nonfinite = s.nonfinite; out->reserved = 0; out->updates = s.updates;
  }
  return SACX_OK;
}

int sacx_update_host(sacx_agent_t h, const int64_t* idx, const float* e1, const float* e2, int32_t n_steps, sacx_metrics* m) {
  if (!h || n_steps <= 0) return fail(SACX_ERR_INVALID, "update_host: bad arguments");
  if (h->e.per) return fail(SACX_ERR_INVALID, "update_host: not available with prioritized replay (use sacx_update)");
  Engine& e = h->e;
  const int slot = (int)(e.host_calls++ & 1);
  int rc = host_update_submit(e, slot, idx, e1, e2, n_steps);
  if (rc) return rc;
  return m ? host_update_collect(e, slot, m) : SACX_OK;     // without metrics the call stays asynchronous
}

int sacx_update_host_pipelined(sacx_agent_t h, const int64_t* idx, const float* e1, const float* e2, int32_t n_steps,
                               sacx_metrics* prev_metrics, int32_t* have_prev) {
  if (!h || n_steps <= 0) return fail(SACX_ERR_INVALID, "update_host_pipelined: bad arguments");
  if (h->e.per) return fail(SACX_ERR_INVALID, "update_host_pipelined: not available with prioritized replay (use sacx_update)");
  Engine& e = h->e;
  const int slot = (int)(e.host_calls++ & 1);
  int rc = host_update_submit(e, slot, idx, e1, e2, n_steps);
  if (rc) return rc;
  const bool prev = e.slots[slot ^ 1].pinned != nullptr && e.pipelined_pending;
  if (have_prev) *have_prev = prev ? 1 : 0;
  if (prev) rc = host_update_collect(e, slot ^ 1, prev_metrics);
  e.pipelined_pending = true;
  return rc;
}

int sacx_update_host_flush(sacx_agent_t h, sacx_metrics* last_metrics) {
  if (!h) return fail(SACX_ERR_INVALID, "null agent");
  Engine& e = h->e;
  if (e.host_calls == 0) return fail(SACX_ERR_INVALID, "no host update was submitted");
  e.pipelined_pending = false;
  return host_update_collect(e, (int)((e.host_calls - 1) & 1), last_metrics);
}

int sacx_sample_batch(sacx_agent_t h, const int64_t* idx) {
  if (!h) return fail(SACX_ERR_INVALID, "null agent");
  int rc = need_ring(h->e, idx == nullptr);
  if (rc) return rc;
  RunArgs a; memset(&a, 0, sizeof a);
  a.idx_ext = (const i64*)idx;
  return engine_launch(&h->e, PLAN_SAMPLE, 0, -1, 1, a, false);
}

int sacx_load_batch(sacx_agent_t h, const float* s, const float* a_, const float* r, const float* s2, const float* d) {
  if (!h) return fail(SACX_ERR_INVALID, "null agent");
  Engine& e = h->e;
  const int B = e.cfg.batch_size;
  load_batch_kernel<<<(B + 7) / 8, 256, 0, e.stream>>>(e.arena, e.x_sa, e.x_s2, e.x_pi, e.b_r, e.b_d, e.ldx, e.cfg.obs_dim,
                                                       e.cfg.act_dim, B, s, a_, r, s2, d);
  ++e.launches;
  SACX_CUDA(cudaGetLastError());
  return SACX_OK;
}

static int copy_out(Engine& e, i64 off, float* dst, int n) {
  if (!dst) return SACX_OK;
  SACX_CUDA(cudaMemcpyAsync(dst, e.arena + off, (size_t)n * 4, cudaMemcpyDeviceToDevice, e.stream));
  return SACX_OK;
}

int sacx_target(sacx_agent_t h, const float* eps1, float* y_out) {
  if (!h) return fail(SACX_ERR_INVALID, "null agent");
  RunArgs a; memset(&a, 0, sizeof a);
  a.eps1_ext = eps1;
  int rc = engine_launch(&h->e, PLAN_TARGET, 0, -1, 1, a, false);
  if (rc) return rc;
  return copy_out(h->e, h->e.b_y, y_out, h->e.cfg.batch_size);
}

static int zero_grads(Engine& e, const NetLayout& a, const NetLayout& b) {
  if (!e.grads_atomic) return SACX_OK;
  for (int ag = 0; ag < e.cfg.n_agents; ++ag)
    SACX_CUDA(cudaMemsetAsync(e.arena + (i64)ag * e.stride + a.begin + 3 * e.blk, 0, (size_t)(b.end - a.begin) * 4, e.stream));
  return SACX_OK;
}

static int critic_run(sacx_agent_t h, const float* y, int plan) {
  if (!h) return fail(SACX_ERR_INVALID, "null agent");
  if (plan == PLAN_CRITIC_GRADS) { int rc = zero_grads(h->e, h->e.q1, h->e.q2); if (rc) return rc; }
  RunArgs a; memset(&a, 0, sizeof a);
  a.y_ext = y;
  return engine_launch(&h->e, plan, 0, -1, 1, a, false);
}
int sacx_critic_step(sacx_agent_t h, const float* y) { return critic_run(h, y, PLAN_CRITIC); }
int sacx_critic_grads(sacx_agent_t h, const float* y) { return critic_run(h, y, PLAN_CRITIC_GRADS); }

static int actor_run(sacx_agent_t h, const float* eps2, float* lp_out, int plan) {
  if (!h) return fail(SACX_ERR_INVALID, "null agent");
  if (plan == PLAN_ACTOR_GRADS) { int rc = zero_grads(h->e, h->e.pi, h->e.pi); if (rc) return rc; }
  RunArgs a; memset(&a, 0, sizeof a);
  a.eps2_ext = eps2;
  int rc = engine_launch(&h->e, plan, 0, -1, 1, a, false);
  if (rc) return rc;
  return copy_out(h->e, h->e.b_lp, lp_out, h->e.cfg.batch_size);
}
int sacx_actor_step(sacx_agent_t h, const float* eps2, float* lp_out) { return actor_run(h, eps2, lp_out, PLAN_ACTOR); }
int sacx_actor_grads(sacx_agent_t h, const float* eps2, float* lp_out) { return actor_run(h, eps2, lp_out, PLAN_ACTOR_GRADS); }

int sacx_alpha_step(sacx_agent_t h, const float* logpi, sacx_metrics* m) {
  if (!h) return fail(SACX_ERR_INVALID, "null agent");
  RunArgs a; memset(&a, 0, sizeof a);
  a.lp_ext = logpi;
  int rc = engine_launch(&h->e, PLAN_ALPHA, 0, -1, 1, a, false);
  if (rc) return rc;
  if (m) { rc = ensure_io(h->e, 0); if (rc) return rc; return read_metrics(h->e, 0, m); }
  return SACX_OK;
}

int sacx_polyak(sacx_agent_t h) {
  if (!h) return fail(SACX_ERR_INVALID, "null agent");
  RunArgs a; memset(&a, 0, sizeof a);
  return engine_launch(&h->e, PLAN_POLYAK, 0, -1, 1, a, false);
}

int sacx_apply_grads(sacx_agent_t h, int32_t which, int32_t polyak) {
  if (!h) return fail(SACX_ERR_INVALID, "null agent");
  RunArgs a; memset(&a, 0, sizeof a);
  int rc = SACX_OK;
  if (which & 1) rc = engine_launch(&h->e, polyak ? PLAN_APPLY_Q_POLYAK : PLAN_APPLY_Q, 0, -1, 1, a, false);
  if (!rc && (which & 2)) rc = engine_launch(&h->e, PLAN_APPLY_PI, 0, -1, 1, a, false);
  if (!rc && (which & 4)) rc = engine_launch(&h->e, PLAN_ALPHA_APPLY, 0, -1, 1, a, false);
  return rc;
}

static NetRef make_ref(const NetLayout& n, i64 shift) {
  NetRef r;
  memset(&r, 0, sizeof r);
  r.n_lin = n.n_lin; r.in_dim = n.dims[0]; r.out_dim = n.dims[n.n_lin]; r.act_h = n.act_h; r.act_o = n.act_o;
  for (int l = 0; l <= n.n_lin; ++l) r.dims[l] = n.dims[l];
  for (int l = 0; l < n.n_lin; ++l) { r.W[l] = n.W[l] + shift; r.b[l] = n.b[l] + shift; }
  return r;
}
static int max_width(const NetLayout& n) {
  int m = 0;
  for (int l = 0; l <= n.n_lin; ++l) m = std::max(m, n.dims[l]);
  return m;
}

int sacx_act(sacx_agent_t h, int32_t agent, const float* s, int32_t n, const float* eps, int32_t deterministic, float* a_out) {
  if (!h || !s || !a_out || n <= 0) return fail(SACX_ERR_INVALID, "act: bad arguments");
  Engine& e = h->e;
  if (agent < 0 || agent >= e.cfg.n_agents) return fail(SACX_ERR_INVALID, "act: agent out of range");
  const int mw = max_width(e.pi);
  act_kernel<<<n, 256, (size_t)2 * mw * 4, e.stream>>>(e.arena, make_ref(e.pi, 0), mw, s, eps, deterministic,
                                                      a_out, e.cfg.act_dim, e.hp.log_std_min, e.hp.log_std_max, e.hp.action_scale,
                                                      e.scal_off, e.act_calls++, agent, e.stride);
  ++e.launches;
  SACX_CUDA(cudaGetLastError());
  return SACX_OK;
}

int sacx_act_population(sacx_agent_t h, const float* s, int32_t n_per_agent, const float* eps, int32_t deterministic, float* a_out) {
  if (!h || !s || !a_out || n_per_agent <= 0) return fail(SACX_ERR_INVALID, "act_population: bad arguments");
  Engine& e = h->e;
  if (e.cfg.n_agents > 65535) return fail(SACX_ERR_INVALID, "act_population: more than 65535 agents");
  const int mw = max_width(e.pi);
  act_kernel<<<dim3(n_per_agent, e.cfg.n_agents), 256, (size_t)2 * mw * 4, e.stream>>>(
      e.arena, make_ref(e.pi, 0), mw, s, eps, deterministic, a_out, e.cfg.act_dim, e.hp.log_std_min, e.hp.log_std_max, e.hp.action_scale,
      e.scal_off, e.act_calls++, 0, e.stride);
  ++e.launches;
  SACX_CUDA(cudaGetLastError());
  return SACX_OK;
}

int sacx_act_host(sacx_agent_t h, int32_t agent, const float* s, int32_t n, const float* eps, int32_t deterministic, float* a_out) {
  if (!h || !s || !a_out || n <= 0) return fail(SACX_ERR_INVALID, "act_host: bad arguments");
  Engine& e = h->e;
  const size_t bs = (size_t)n * e.cfg.obs_dim * 4, be = eps ? (size_t)n * e.cfg.act_dim * 4 : 0, ba = (size_t)n * e.cfg.act_dim * 4;
  int rc = ensure_io(e, bs + be + ba);
  if (rc) return rc;
  char* hp = (char*)e.pinned_io; char* dp = (char*)e.dev_io;
  memcpy(hp, s, bs);
  if (eps) memcpy(hp + bs, eps, be);
  SACX_CUDA(cudaMemcpyAsync(dp, hp, bs + be, cudaMemcpyHostToDevice, e.stream));
  rc = sacx_act(h, agent, (const float*)dp, n, eps ? (const float*)(dp + bs) : nullptr, deterministic, (float*)(dp + bs + be));
  if (rc) return rc;
  SACX_CUDA(cudaMemcpyAsync(hp + bs + be, dp + bs + be, ba, cudaMemcpyDeviceToHost, e.stream));
  SACX_CUDA(cudaStreamSynchronize(e.stream));
  memcpy(a_out, hp + bs + be, ba);
  return SACX_OK;
}

int sacx_q_values(sacx_agent_t h, int32_t agent, const float* s, const float* a_, int32_t n, float* q1o, float* q2o) {
  if (!h || !s || !a_ || !q1o || !q2o || n <= 0) return fail(SACX_ERR_INVALID, "q_values: bad arguments");
  Engine& e = h->e;
  if (agent < 0 || agent >= e.cfg.n_agents) return fail(SACX_ERR_INVALID, "q_values: agent out of range");
  const int mw = max_width(e.q1);
  qvalue_kernel<<<dim3(n, 2), 256, (size_t)2 * mw * 4, e.stream>>>(e.arena + (i64)agent * e.stride, make_ref(e.q1, 0), make_ref(e.q2, 0),
                                                                  mw, e.cfg.obs_dim, e.cfg.act_dim, s, a_, q1o, q2o);
  ++e.launches;
  SACX_CUDA(cudaGetLastError());
  return SACX_OK;
}

int sacx_q_values_host(sacx_agent_t h, int32_t agent, const float* s, const float* a_, int32_t n, float* q1o, float* q2o) {
  if (!h || !s || !a_ || !q1o || !q2o || n <= 0) return fail(SACX_ERR_INVALID, "q_values_host: bad arguments");
  Engine& e = h->e;
  const size_t bs = (size_t)n * e.cfg.obs_dim * 4, ba = (size_t)n * e.cfg.act_dim * 4, bq = (size_t)n * 4;
  int rc = ensure_io(e, bs + ba + 2 * bq);
  if (rc) return rc;
  char* hp = (char*)e.pinned_io; char* dp = (char*)e.dev_io;
  memcpy(hp, s, bs);
  memcpy(hp + bs, a_, ba);
  SACX_CUDA(cudaMemcpyAsync(dp, hp, bs + ba, cudaMemcpyHostToDevice, e.stream));
  rc = sacx_q_values(h, agent, (const float*)dp, (const float*)(dp + bs), n, (float*)(dp + bs + ba), (float*)(dp + bs + ba + bq));
  if (rc) return rc;
  SACX_CUDA(cudaMemcpyAsync(hp + bs + ba, dp + bs + ba, 2 * bq, cudaMemcpyDeviceToHost, e.stream));
  SACX_CUDA(cudaStreamSynchronize(e.stream));
  memcpy(q1o, hp + bs + ba, bq);
  memcpy(q2o, hp + bs + ba + bq, bq);
  return SACX_OK;
}

int sacx_get_metrics(sacx_agent_t h, int32_t agent, sacx_metrics* m) {
  if (!h || !m) return fail(SACX_ERR_INVALID, "get_metrics: bad arguments");
  if (agent < 0 || agent >= h->e.cfg.n_agents) return fail(SACX_ERR_INVALID, "agent out of range");
  int rc = ensure_io(h->e, 0);
  if (rc) return rc;
  return read_metrics(h->e, agent, m);
}

int sacx_debug_profile(sacx_agent_t h, int32_t n_steps, uint64_t* out_host, int64_t capacity, int32_t* n_phases, int32_t* n_ctas) {
  if (!h || !out_host || n_steps <= 0) return fail(SACX_ERR_INVALID, "debug_profile: bad arguments");
  Engine& e = h->e;
  int rc = need_ring(e, true);
  if (rc) return rc;
  const int np = e.rp ? 4 : e.h_plans[PLAN_FUSED].n_phases;
  const int gx = e.rp ? e.rp_grid : e.grid_x;
  const size_t words = (size_t)n_steps * np * gx * 10;
  if ((int64_t)words > capacity) return fail(SACX_ERR_INVALID, "debug_profile: output too small");
  unsigned long long* d = nullptr;
  SACX_CUDA(cudaMalloc((void**)&d, words * 8));
  SACX_CUDA(cudaMemset(d, 0, words * 8));
  RunArgs a; memset(&a, 0, sizeof a);
  a.dbg = d;
  a.dbg2 = d + (size_t)n_steps * np * gx * 2;
  rc = e.rp ? engine_launch_rp(&e, n_steps, a) : engine_launch(&e, PLAN_FUSED, 0, -1, n_steps, a, false);
  if (!rc) {
    cudaError_t ce = cudaStreamSynchronize(e.stream);
    if (ce == cudaSuccess) ce = cudaMemcpy(out_host, d, words * 8, cudaMemcpyDeviceToHost);
    if (ce != cudaSuccess) rc = fail(SACX_ERR_CUDA, cudaGetErrorString(ce));
  }
  cudaFree(d);
  if (n_phases) *n_phases = np;
  if (n_ctas) *n_ctas = gx;
  return rc;
}

int sacx_sync(sacx_agent_t h) {
  if (!h) return fail(SACX_ERR_INVALID, "null agent");
  SACX_CUDA(cudaStreamSynchronize(h->e.stream));
  return SACX_OK;
}

int64_t sacx_launch_count(sacx_agent_t h) { return h ? h->e.launches + (h->e.ring ? h->e.ring->launches : 0) : 0; }

// ---------------------------------------------------------------------------------------- population-based training
int sacx_sizeof_pbt_record(void) { return (int)sizeof(sacx_pbt_record); }

int64_t sacx_pbt_state_floats(sacx_agent_t h) { return h ? pbt_span0(h->e) + pbt_span1(h->e) : 0; }

int sacx_pbt_copy(sacx_agent_t h, const int32_t* src, const int32_t* dst, int32_t n, const sacx_pbt_record* rec) {
  if (!h || n < 0 || (n > 0 && (!src || !dst))) return fail(SACX_ERR_INVALID, "pbt_copy: bad arguments");
  Engine& e = h->e;
  int rc;
  if ((rc = pbt_check_agents(e, src, n, "source")) || (rc = pbt_check_agents(e, dst, n, "destination")) ||
      (rc = pbt_check_destinations(e, dst, n, src)))
    return rc;
  return pbt_launch(e, pbt_arena(e), pbt_arena(e), true, src, dst, n, rec);
}

int sacx_pbt_pack(sacx_agent_t h, const int32_t* agents, int32_t n, float* buf) {
  if (!h || n < 0 || (n > 0 && (!agents || !buf))) return fail(SACX_ERR_INVALID, "pbt_pack: bad arguments");
  if ((uintptr_t)buf & 15) return fail(SACX_ERR_INVALID, "pbt_pack: buffer not 16-byte aligned");
  Engine& e = h->e;
  int rc = pbt_check_agents(e, agents, n, "source");
  if (rc) return rc;
  std::vector<int32_t> slots((size_t)n);
  for (int i = 0; i < n; ++i) slots[i] = i;
  return pbt_launch(e, pbt_arena(e), pbt_buffer(e, buf), false, agents, slots.data(), n, nullptr);
}

int sacx_pbt_unpack(sacx_agent_t h, const float* buf, int32_t n_slots, const int32_t* slots, const int32_t* dst, int32_t n,
                    const sacx_pbt_record* rec) {
  if (!h || n < 0 || n_slots < 0 || (n > 0 && (!buf || !slots || !dst))) return fail(SACX_ERR_INVALID, "pbt_unpack: bad arguments");
  if ((uintptr_t)buf & 15) return fail(SACX_ERR_INVALID, "pbt_unpack: buffer not 16-byte aligned");
  Engine& e = h->e;
  for (int i = 0; i < n; ++i)
    if (slots[i] < 0 || slots[i] >= n_slots)
      return fail(SACX_ERR_INVALID, "pbt_unpack: slot " + std::to_string(slots[i]) + " out of range [0, " + std::to_string(n_slots) + ")");
  int rc;
  if ((rc = pbt_check_agents(e, dst, n, "destination")) || (rc = pbt_check_destinations(e, dst, n, nullptr))) return rc;
  return pbt_launch(e, pbt_buffer(e, buf), pbt_arena(e), true, slots, dst, n, rec);
}

// ---------------------------------------------------------------------------------------- prioritized replay
int sacx_per_create(sacx_ring_t ring, float alpha, float beta0, int64_t beta_steps, float eps, int32_t max_batch, sacx_per_t* out) {
  if (!ring || !out) return fail(SACX_ERR_INVALID, "per_create: null argument");
  if (!(alpha >= 0.f) || !(beta0 >= 0.f && beta0 <= 1.f) || beta_steps < 0 || !(eps > 0.f) || !std::isfinite(alpha) || !std::isfinite(eps) ||
      max_batch <= 0)
    return fail(SACX_ERR_INVALID, "per_create: need alpha >= 0, 0 <= beta0 <= 1, beta_steps >= 0, eps > 0, max_batch > 0");
  Ring& r = ring->r;
  if (r.n_agents != 1) return fail(SACX_ERR_INVALID, "per_create: prioritized replay needs a single-agent ring");
  sacx_per_s* h = new sacx_per_s();
  Per& p = h->p;
  p.ring = &r; p.alpha = alpha; p.beta0 = beta0; p.beta_steps = beta_steps; p.eps = eps; p.max_batch = max_batch;
  p.nodes[0] = r.cap;
  do {
    ++p.depth;
    p.nodes[p.depth] = (p.nodes[p.depth - 1] + PER_FANOUT - 1) / PER_FANOUT;
    p.internal += p.nodes[p.depth];
  } while (p.nodes[p.depth] > 1);
  int rc = SACX_OK;
  auto bad = [&](cudaError_t ce) { if (ce == cudaSuccess) return false; rc = fail(SACX_ERR_CUDA, cudaGetErrorString(ce)); return true; };
  int dev = 0, sms = 0, per_sm = 0;
  PerState st;
  memset(&st, 0, sizeof st);
  const float one = 1.f;
  memcpy(&st.pmax_bits, &one, 4);
  if (bad(cudaGetDevice(&dev)) || bad(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev)) ||
      bad(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, per_refresh_kernel, 256, 0)) ||
      bad(cudaMalloc((void**)&p.d_leaf, (size_t)r.cap * 4)) || bad(cudaMalloc((void**)&p.d_tree, (size_t)p.internal * 8)) ||
      bad(cudaMalloc((void**)&p.d_mark, (size_t)p.internal * 4)) || bad(cudaMalloc((void**)&p.d_win, (size_t)r.cap * 8)) ||
      bad(cudaMalloc((void**)&p.d_st, sizeof(PerState))) || bad(cudaMalloc((void**)&p.d_idx, (size_t)max_batch * 8)) ||
      bad(cudaMalloc((void**)&p.d_w, (size_t)max_batch * 4)) || bad(cudaMalloc((void**)&p.d_slots, (size_t)max_batch * 8)) ||
      bad(cudaMemset(p.d_leaf, 0, (size_t)r.cap * 4)) || bad(cudaMemset(p.d_mark, 0, (size_t)p.internal * 4)) ||
      bad(cudaMemset(p.d_win, 0, (size_t)r.cap * 8)) || bad(cudaMemcpy(p.d_st, &st, sizeof st, cudaMemcpyHostToDevice))) {
    sacx_per_destroy(h);
    return rc;
  }
  p.grid_max = std::max(1, per_sm * sms);
  *out = h;
  return SACX_OK;
}

int sacx_per_destroy(sacx_per_t h) {
  if (!h) return SACX_OK;
  Per& p = h->p;
  if (p.agent) { p.flush(); p.agent->per = nullptr; p.agent = nullptr; }
  cudaStreamSynchronize(p.stream());
  cudaFree(p.d_leaf); cudaFree(p.d_tree); cudaFree(p.d_mark); cudaFree(p.d_win); cudaFree(p.d_st);
  cudaFree(p.d_idx); cudaFree(p.d_w); cudaFree(p.d_slots);
  delete h;
  return SACX_OK;
}

int sacx_per_sample(sacx_per_t h, int32_t B, float beta, const float* u_dev, uint64_t seed, uint64_t counter, int64_t* idx_dev,
                    float* w_dev) {
  if (!h || B <= 0 || !idx_dev || !w_dev) return fail(SACX_ERR_INVALID, "per_sample: bad arguments");
  Per& p = h->p;
  if (B > p.max_batch) return fail(SACX_ERR_INVALID, "per_sample: B exceeds the tree's max_batch");
  if (!(beta >= 0.f && beta <= 1.f)) return fail(SACX_ERR_INVALID, "per_sample: beta must be in [0, 1]");
  if (p.ring->len(0) < 1) return fail(SACX_ERR_UNDERFILLED, "per_sample: the replay buffer is empty");
  PerArgs a = p.base();
  a.B = B; a.beta = beta; a.u_ext = u_dev; a.seed = seed; a.counter = counter; a.agent = 0;
  a.out_idx = (i64*)idx_dev; a.out_w = w_dev; a.out_slots = p.d_slots;
  return p.run(a);
}

int sacx_per_update_priorities(sacx_per_t h, const int64_t* idx_dev, const float* delta_dev, int32_t B) {
  if (!h || !idx_dev || !delta_dev || B <= 0) return fail(SACX_ERR_INVALID, "per_update_priorities: bad arguments");
  Per& p = h->p;
  int rc = p.pend_n ? p.flush() : SACX_OK;
  if (rc) return rc;
  PerArgs a = p.base();
  a.wb_n = B; a.wb_idx = (const i64*)idx_dev; a.wb_delta = delta_dev;
  return p.run(a);
}

int sacx_per_priorities(sacx_per_t h, float* leaves_dev, float* p_max) {
  if (!h) return fail(SACX_ERR_INVALID, "null tree");
  Per& p = h->p;
  int rc = p.flush();
  if (rc) return rc;
  if (leaves_dev) SACX_CUDA(cudaMemcpyAsync(leaves_dev, p.d_leaf, (size_t)p.ring->cap * 4, cudaMemcpyDeviceToDevice, p.stream()));
  if (p_max) {
    PerState st;
    SACX_CUDA(cudaMemcpyAsync(&st, p.d_st, sizeof st, cudaMemcpyDeviceToHost, p.stream()));
    SACX_CUDA(cudaStreamSynchronize(p.stream()));
    memcpy(p_max, &st.pmax_bits, 4);
  }
  return SACX_OK;
}

int sacx_per_load_priorities(sacx_per_t h, const float* leaves_dev, float p_max) {
  if (!h || !leaves_dev || !(p_max > 0.f) || !std::isfinite(p_max)) return fail(SACX_ERR_INVALID, "per_load_priorities: bad arguments");
  Per& p = h->p;
  p.pend_n = 0;                                        // priorities of the run being replaced
  int rc = p.ring->flush();
  if (rc) return rc;
  SACX_CUDA(cudaStreamSynchronize(p.ring->stream));
  const i64 pushes = p.ring->pushes[0], cap = p.ring->cap;
  PerState st;
  memset(&st, 0, sizeof st);
  st.seen = pushes; st.sample_oldest = pushes > cap ? pushes % cap : 0;
  memcpy(&st.pmax_bits, &p_max, 4);
  SACX_CUDA(cudaMemcpyAsync(p.d_leaf, leaves_dev, (size_t)cap * 4, cudaMemcpyDeviceToDevice, p.stream()));
  SACX_CUDA(cudaMemcpyAsync(p.d_st, &st, sizeof st, cudaMemcpyHostToDevice, p.stream()));
  SACX_CUDA(cudaStreamSynchronize(p.stream()));
  p.seen_hint = pushes;
  p.rebuild = true;
  return p.flush();
}

int sacx_agent_attach_per(sacx_agent_t h, sacx_per_t per) {
  if (!h) return fail(SACX_ERR_INVALID, "null agent");
  Engine& e = h->e;
  if (per) {
    Per& p = per->p;
    if (e.cfg.n_agents != 1 || e.cfg.dp_world > 1)
      return fail(SACX_ERR_INVALID, "prioritized replay supports a single agent without data parallelism");
    if (e.ring != p.ring) return fail(SACX_ERR_INVALID, "attach_per: the tree belongs to a different ring than the agent's");
    if (p.max_batch < e.cfg.batch_size) return fail(SACX_ERR_INVALID, "attach_per: the tree's max_batch is below the batch size");
    if (p.agent && p.agent != &e) return fail(SACX_ERR_INVALID, "attach_per: the tree is attached to another agent");
  }
  if (e.per && e.per != (per ? &per->p : nullptr)) {
    int rc = e.per->flush();
    if (rc) return rc;
    e.per->agent = nullptr;
  }
  e.per = per ? &per->p : nullptr;
  if (per) per->p.agent = &e;
  return SACX_OK;
}

}  // extern "C"
