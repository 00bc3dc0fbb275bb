// Host side of the engine: arena layout, plan (op table) construction, launches.
#pragma once
#include <cuda_runtime.h>

#include <algorithm>
#include <cstddef>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#include "sacx_kernels.cuh"
#include "sacx_rowpar.cuh"
#include "sacx_tc.cuh"

namespace sacx {

extern thread_local std::string g_err;
int fail(int code, const std::string& msg);
#define SACX_CUDA(call)                                                                        \
  do {                                                                                         \
    cudaError_t e__ = (call);                                                                  \
    if (e__ != cudaSuccess)                                                                    \
      return fail(SACX_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e__));         \
  } while (0)

inline i64 align4(i64 x) { return (x + 3) & ~(i64)3; }
inline int rup4(int x) { return (x + 3) & ~3; }

struct NetLayout {
  int n_lin = 0, act_h = 0, act_o = 0;
  int dims[SACX_MAX_HIDDEN + 2] = {0};
  i64 W[SACX_MAX_HIDDEN + 1], b[SACX_MAX_HIDDEN + 1];
  i64 begin = 0, end = 0;
  int L() const { return n_lin - 1; }                 // hidden layers
};

struct ActSet {                                         // hidden activations of one forward pass
  i64 h[SACX_MAX_HIDDEN], z[SACX_MAX_HIDDEN];
  int ld[SACX_MAX_HIDDEN];
  i64 aux(int l) const { return z[l] >= 0 ? z[l] : h[l]; }
};

enum PlanId { PLAN_FUSED = 0, PLAN_SAMPLE, PLAN_TARGET, PLAN_CRITIC, PLAN_CRITIC_GRADS, PLAN_ACTOR, PLAN_ACTOR_GRADS,
              PLAN_ALPHA, PLAN_POLYAK, PLAN_APPLY_Q, PLAN_APPLY_Q_POLYAK, PLAN_APPLY_PI, PLAN_FUSED_NOGATHER, PLAN_ALPHA_APPLY, PLAN_RP, N_PLANS };

struct Ring;
struct Per;

struct Engine {
  sacx_config cfg;
  int n_sms = 0, max_ctas = 0;
  bool large = false, grads_atomic = false;
  int grid_x = 1, grid_y = 1, smem_bytes = 0;
  std::vector<sacx_tensor_desc> lay;
  i64 cur = 0, stride = 0;
  NetLayout pi, q1, q2;
  i64 P0 = 0, blk = 0, T0 = 0, scal_off = 0, pi_x = 0;
  i64 n_online = 0, n_critic = 0;
  // batch / scratch
  int ldx = 0;
  i64 x_sa, x_s2, x_pi, b_r, b_d, b_idx, b_eps1, b_eps2, b_lp2, b_lp, b_y, b_tq[2], b_q[2], b_qa[2], b_dout[2], b_loss[2], b_coef[2],
      b_ploss, b_tz, b_se, b_mask, b_headz, b_headz_t, b_headz_a, b_dhead;
  ActSet a_pit, a_pia, a_q[2], a_qt[2];
  i64 d_q[2][SACX_MAX_HIDDEN], d_p[SACX_MAX_HIDDEN];
  float* arena = nullptr;
  bool own_arena = false;
  Plan* d_plans = nullptr;
  std::vector<Plan> h_plans;
  unsigned* d_barrier = nullptr;
  sacx_metrics* pinned_metrics = nullptr;
  void* pinned_io = nullptr;
  size_t pinned_io_bytes = 0;
  void* dev_io = nullptr;
  size_t dev_io_bytes = 0;
  struct IoSlot {
    void* pinned = nullptr; void* dev = nullptr; size_t bytes = 0, metrics_off = 0; cudaEvent_t done = nullptr; bool busy = false;
    cudaEvent_t copied = nullptr;         // the slot's H2D copy (on copy_stream) has landed
  };
  cudaStream_t copy_stream = nullptr;     // host inputs of step t+1 travel here while the kernel of step t runs on `stream`
  IoSlot slots[2];
  unsigned long long host_calls = 0;
  bool pipelined_pending = false;
  cudaStream_t stream = 0;
  Ring* ring = nullptr;
  Per* per = nullptr;                     // prioritized replay tree (sacx_agent_attach_per), or null: uniform sampling
  long long launches = 0;
  unsigned long long act_calls = 0;
  Hyper hp;
  // row-parallel cluster path (sacx_rowpar.cuh): single agent, 2+ hidden layers of width 64/128/256
  bool rp = false;
  RpProgram h_prog;
  RpProgram* d_prog = nullptr;
  float* d_rp_part = nullptr;
  int rp_grid = 0, rp_smem_bytes = 0;
  unsigned long long rp_launch_no = 0;  // parity selects the barrier counter set of a launch
  bool rp_tma = true;              // weight slices by TMA where the layout allows (SACX_RP_TMA=0: cp.async everywhere)
  void* d_rp_maps = nullptr;       // device array of CUtensorMap: one per job, then two (dy, x) per dW op of the tile-parallel phases
  std::string rp_why;
  // tensor-core path (sacx_tc.cuh): single agent at large batch; per plan phase the TC-eligible GEMM ops in groups of <= 4
  struct TcGroup { TcParams p; TcMaps maps; int grid = 0; bool has_red = false; TcRedParams red; int red_blocks = 0; };
  struct TcPhase { std::vector<TcGroup> groups; bool other_ops = false; bool light = true; };   // light: no FFMA GEMM tile left in the phase
  bool tc = false;
  int tc_min_batch = 4096;         // single agent: smallest batch that takes the tensor-core path
  int tc_min_m = 4096;             // smallest GEMM row count per agent (population: 128, one row tile)
  std::string tc_why;
  bool tc_forbid = false;          // tensor-core setup failed: plans are rebuilt without the features that need it
  std::vector<std::vector<TcPhase>> tc_phases;       // [plan][phase]
  float* d_tc_scratch = nullptr;
  size_t tc_scratch_floats = 0;
  long long tc_launches = 0;
  int rows_tsm_floats = 0, rows_smem_bytes = 0, rows_ctas_per_sm = 1;

  // ---------------------------------------------------------------- layout
  i64 alloc(const std::string& name, int rows, int cols, int ld = -1, int dtype = 0) {
    if (ld < 0) ld = cols;
    cur = align4(cur);
    sacx_tensor_desc d;
    memset(&d, 0, sizeof d);
    snprintf(d.name, sizeof d.name, "%s", name.c_str());
    d.offset = cur; d.rows = rows; d.cols = cols; d.ld = ld; d.dtype = dtype;
    lay.push_back(d);
    cur += (i64)rows * ld * (dtype == 0 ? 1 : 2);
    return d.offset;
  }

  void layout_net(NetLayout& n, const std::string& tag, int in, const int32_t* hidden, int nh, int out, int act_h, int act_o) {
    n.n_lin = nh + 1; n.act_h = act_h; n.act_o = act_o;
    n.dims[0] = in;
    for (int i = 0; i < nh; ++i) n.dims[i + 1] = hidden[i];
    n.dims[nh + 1] = out;
    cur = align4(cur);
    n.begin = cur;
    for (int l = 0; l < n.n_lin; ++l) {
      n.W[l] = alloc(tag + ".W" + std::to_string(l), n.dims[l + 1], n.dims[l]);
      n.b[l] = alloc(tag + ".b" + std::to_string(l), 1, n.dims[l + 1]);
    }
    n.end = align4(cur);
    cur = n.end;
  }

  void alias_block(const std::string& prefix, i64 shift, const NetLayout& n, const std::string& tag) {
    for (int l = 0; l < n.n_lin; ++l) {
      for (int wb = 0; wb < 2; ++wb) {
        sacx_tensor_desc d;
        memset(&d, 0, sizeof d);
        snprintf(d.name, sizeof d.name, "%s%s.%c%d", prefix.c_str(), tag.c_str(), wb ? 'b' : 'W', l);
        d.offset = (wb ? n.b[l] : n.W[l]) + shift;
        d.rows = wb ? 1 : n.dims[l + 1];
        d.cols = wb ? n.dims[l + 1] : n.dims[l];
        d.ld = d.cols;
        lay.push_back(d);
      }
    }
  }

  void alloc_actset(ActSet& s, const std::string& tag, const NetLayout& n, bool save_z) {
    const int B = cfg.batch_size;
    for (int l = 0; l < SACX_MAX_HIDDEN; ++l) { s.h[l] = s.z[l] = -1; s.ld[l] = 0; }
    for (int l = 0; l < n.L(); ++l) {
      s.ld[l] = rup4(n.dims[l + 1]);
      s.h[l] = alloc(tag + ".h" + std::to_string(l), B, n.dims[l + 1], s.ld[l]);
      if (save_z && act_needs_z(n.act_h)) s.z[l] = alloc(tag + ".z" + std::to_string(l), B, n.dims[l + 1], s.ld[l]);
    }
  }

  void build_layout() {
    const int O = cfg.obs_dim, A = cfg.act_dim, B = cfg.batch_size;
    cur = 0;
    scal_off = alloc("scalars", 1, (int)((sizeof(AgentScalars) + 3) / 4));
    {  // named views of the scalar block (offsetof keeps the Python side in step with the struct)
      auto sub = [&](const char* name, size_t byte_off, int count, int dtype) {
        sacx_tensor_desc d; memset(&d, 0, sizeof d);
        snprintf(d.name, sizeof d.name, "%s", name);
        d.offset = scal_off + (i64)(byte_off / 4); d.rows = 1; d.cols = d.ld = count; d.dtype = dtype;
        lay.push_back(d);
      };
      sub("scal.log_alpha", offsetof(AgentScalars, log_alpha), 1, 1);
      sub("scal.alpha_m", offsetof(AgentScalars, alpha_m), 1, 1);
      sub("scal.alpha_v", offsetof(AgentScalars, alpha_v), 1, 1);
      sub("scal.alpha", offsetof(AgentScalars, alpha), 1, 1);
      sub("scal.step", offsetof(AgentScalars, step), N_OPT, 2);
      sub("scal.updates", offsetof(AgentScalars, updates), 1, 2);
      sub("scal.alpha_lr", offsetof(AgentScalars, alpha_lr), 1, 1);
      sub("scal.alpha_f32", offsetof(AgentScalars, alpha_f32), 1, 0);
      sub("scal.metrics", offsetof(AgentScalars, metrics), 12, 0);
      sub("scal.nonfinite", offsetof(AgentScalars, nonfinite), 1, 0);
      sub("scal.dp_alpha", offsetof(AgentScalars, dp_mean_t), 2, 0);
      sub("scal.lr", offsetof(AgentScalars, lr), 3, 1);
      sub("scal.gamma", offsetof(AgentScalars, gamma), 1, 0);
      sub("scal.tau", offsetof(AgentScalars, tau), 2, 0);                 // (tau, 1 - tau) as the Polyak update uses them
      sub("scal.rng_agent", offsetof(AgentScalars, rng_agent), 1, 0);     // uint32 bits in an f32 view
      sub("scal.rng_seed", offsetof(AgentScalars, rng_seed), 1, 2);
    }
    cur = align4(cur);
    P0 = cur;
    layout_net(pi, "pi", O, cfg.hidden_pi, cfg.n_hidden_pi, 2 * A, cfg.act_hidden_pi, cfg.act_out_pi);
    // four spare floats behind the policy in every block: in the GRADIENT block they carry this rank's share of the temperature
    // gradient, so the data-parallel exchange #2 is ONE all-reduce of [policy gradients | share] ("block.g.policy_x")
    pi_x = cur;
    cur += 4;
    layout_net(q1, "q1", O + A, cfg.hidden_q, cfg.n_hidden_q, 1, cfg.act_hidden_q, cfg.act_out_q);
    layout_net(q2, "q2", O + A, cfg.hidden_q, cfg.n_hidden_q, 1, cfg.act_hidden_q, cfg.act_out_q);
    blk = align4(cur - P0);
    n_online = cur - P0;
    n_critic = q2.end - q1.begin;
    { sacx_tensor_desc d; memset(&d, 0, sizeof d); snprintf(d.name, sizeof d.name, "block.params"); d.offset = P0; d.rows = 1; d.cols = d.ld = (int)n_online; lay.push_back(d); }
    const char* pre[3] = {"m.", "v.", "g."};
    for (int k = 0; k < 3; ++k) {
      const i64 shift = blk * (k + 1);
      alias_block(pre[k], shift, pi, "pi");
      alias_block(pre[k], shift, q1, "q1");
      alias_block(pre[k], shift, q2, "q2");
      sacx_tensor_desc d; memset(&d, 0, sizeof d);
      snprintf(d.name, sizeof d.name, "block.%c", pre[k][0]); d.offset = P0 + shift; d.rows = 1; d.cols = d.ld = (int)n_online; lay.push_back(d);
    }
    { // contiguous gradient slices for the data-parallel all-reduce
      sacx_tensor_desc d; memset(&d, 0, sizeof d);
      snprintf(d.name, sizeof d.name, "block.g.policy"); d.offset = pi.begin + 3 * blk; d.rows = 1; d.cols = d.ld = (int)(pi.end - pi.begin); lay.push_back(d);
      snprintf(d.name, sizeof d.name, "block.g.policy_x"); d.cols = d.ld = (int)(pi.end - pi.begin) + 4; lay.push_back(d);
      snprintf(d.name, sizeof d.name, "block.g.critics"); d.offset = q1.begin + 3 * blk; d.cols = d.ld = (int)(q2.end - q1.begin); lay.push_back(d);
    }
    cur = P0 + 4 * blk;
    T0 = align4(cur);
    alias_block("", T0 - q1.begin, q1, "q1t");
    alias_block("", T0 - q1.begin, q2, "q2t");
    { sacx_tensor_desc d; memset(&d, 0, sizeof d); snprintf(d.name, sizeof d.name, "block.targets"); d.offset = T0; d.rows = 1; d.cols = d.ld = (int)n_critic; lay.push_back(d); }
    cur = T0 + align4(n_critic);
    // batch buffers
    ldx = rup4(O + A);
    x_sa = alloc("batch.sa", B, O + A, ldx);
    x_s2 = alloc("batch.s2a", B, O + A, ldx);
    x_pi = alloc("batch.spi", B, O + A, ldx);
    b_r = alloc("batch.r", 1, B);
    b_d = alloc("batch.d", 1, B);
    b_idx = alloc("batch.idx", 1, B, B, 2);
    b_eps1 = alloc("batch.eps1", B, A);
    b_eps2 = alloc("batch.eps2", B, A);
    b_lp2 = alloc("out.logpi_next", 1, B);
    b_lp = alloc("out.logpi", 1, B);
    b_y = alloc("out.y", 1, B);
    for (int c = 0; c < 2; ++c) {
      const std::string s = std::to_string(c + 1);
      b_tq[c] = alloc("out.tq" + s, 1, B);
      b_q[c] = alloc("out.q" + s, 1, B);
      b_qa[c] = alloc("out.q" + s + "_pi", 1, B);
      b_dout[c] = alloc("scr.dout" + s, B, 1, 4);        // row stride 4: the dW tile reads it as a 16B-aligned [batch][1] operand
      b_loss[c] = alloc("scr.lossrow" + s, 1, B);
      b_coef[c] = alloc("scr.coef" + s, B, 1, 4);         // actor phase: routed dQ coefficient per row (tensor-core plans)
    }
    b_ploss = alloc("scr.plossrow", 1, B);
    b_tz = alloc("scr.tz", B, A);
    b_se = alloc("scr.se", B, A);
    b_mask = alloc("scr.mask", B, A);
    b_headz = alloc("scr.headz", B, 2 * A);
    b_headz_t = alloc("scr.headz_t", B, 2 * A, rup4(2 * A));      // head pre-activations of pi(s') / pi(s) as the tensor-core head GEMM
    b_headz_a = alloc("scr.headz_a", B, 2 * A, rup4(2 * A));      // writes them: rows padded to 16 bytes (TMA store)
    b_dhead = alloc("scr.dhead", B, 2 * A);
    alloc_actset(a_pit, "act.pit", pi, false);
    alloc_actset(a_pia, "act.pia", pi, true);
    for (int c = 0; c < 2; ++c) {
      alloc_actset(a_q[c], "act.q" + std::to_string(c + 1), c ? q2 : q1, true);
      alloc_actset(a_qt[c], "act.qt" + std::to_string(c + 1), c ? q2 : q1, false);
      for (int l = 0; l < q1.L(); ++l)
        d_q[c][l] = alloc("delta.q" + std::to_string(c + 1) + "." + std::to_string(l), B, q1.dims[l + 1], rup4(q1.dims[l + 1]));
    }
    for (int l = 0; l < pi.L(); ++l) d_p[l] = alloc("delta.pi." + std::to_string(l), B, pi.dims[l + 1], rup4(pi.dims[l + 1]));
    stride = (align4(cur) + 127) & ~(i64)127;   // 512-byte aligned agent blocks
  }

  // ---------------------------------------------------------------- op constructors
  static Op blank(int type) {
    Op o;
    memset(&o, 0, sizeof o);
    o.type = type;
    o.a = o.b = o.c = o.bias = o.aux = o.zout = -1;
    o.p = o.pm = o.pv = o.pt = o.pg = o.pb = o.pbm = o.pbv = o.pbt = o.pbg = -1;
    for (auto& x : o.o) x = -1;
    return o;
  }
  int BMt() const { return large ? CfgLarge::BM : CfgSmall::BM; }
  int BNt() const { return large ? CfgLarge::BN : CfgSmall::BN; }
  void finish_gemm(Op& o) const {
    const int tm = (o.M + BMt() - 1) / BMt();
    o.tiles_n = (o.N + BNt() - 1) / BNt();
    o.ntiles = tm * o.tiles_n;
    o.cfg = large ? 1 : 0;
    // operand orientation follows the epilogue kind (forward: A,B row-major; dA: B k-major; dW: both k-major)
    const bool a_km = (o.epi == EPI_DW), b_km = (o.epi != EPI_FWD);
    const int ao = a_km ? o.a_sk : o.a_sm, bo = b_km ? o.b_sk : o.b_sn;
    o.a_vec = (o.a % 4 == 0) && (ao % 4 == 0);
    o.b_vec = (o.b % 4 == 0) && (bo % 4 == 0);
  }
  Op gemm_fwd(const NetLayout& n, int l, i64 wshift, i64 x, int ld_x, const ActSet& as) const {
    Op o = blank(OP_GEMM);
    o.epi = EPI_FWD; o.act = n.act_h;
    o.M = cfg.batch_size; o.N = n.dims[l + 1]; o.K = n.dims[l];
    o.a = x; o.a_sm = ld_x; o.a_sk = 1;
    o.b = n.W[l] + wshift; o.b_sk = 1; o.b_sn = o.K;
    o.bias = n.b[l] + wshift;
    o.c = as.h[l]; o.ldc = as.ld[l]; o.zout = as.z[l];
    finish_gemm(o);
    return o;
  }
  // delta_{l-1} = (delta_l . W_l) * act'(layer l-1)
  Op gemm_da(const NetLayout& n, int l, i64 dy, int ld_dy, i64 dx, int ld_dx, i64 aux, int ld_aux) const {
    Op o = blank(OP_GEMM);
    o.epi = EPI_DACT; o.act = n.act_h;
    o.M = cfg.batch_size; o.N = n.dims[l]; o.K = n.dims[l + 1];
    o.a = dy; o.a_sm = ld_dy; o.a_sk = 1;
    o.b = n.W[l]; o.b_sk = n.dims[l]; o.b_sn = 1;
    o.c = dx; o.ldc = ld_dx; o.aux = aux; o.ld_aux = ld_aux;
    finish_gemm(o);
    return o;
  }
  // dW_l = delta_l^T . input_l  (+ db_l) with the optimiser step fused into the epilogue
  Op gemm_dw(const NetLayout& n, int l, int opt, int flags, i64 dy, int ld_dy, i64 x, int ld_x, bool is_critic) const {
    Op o = blank(OP_GEMM);
    o.epi = EPI_DW; o.opt = opt; o.flags = flags;
    o.M = n.dims[l + 1]; o.N = n.dims[l]; o.K = cfg.batch_size;
    o.a = dy; o.a_sm = 1; o.a_sk = ld_dy;
    o.b = x; o.b_sk = ld_x; o.b_sn = 1;
    o.p = n.W[l]; o.pm = n.W[l] + blk; o.pv = n.W[l] + 2 * blk; o.pg = n.W[l] + 3 * blk;
    o.pb = n.b[l]; o.pbm = n.b[l] + blk; o.pbv = n.b[l] + 2 * blk; o.pbg = n.b[l] + 3 * blk;
    if (is_critic) { o.pt = n.W[l] - q1.begin + T0; o.pbt = n.b[l] - q1.begin + T0; }
    finish_gemm(o);
    if (flags == DW_STORE_GRAD && o.K >= 2048) {      // gradient-only dW at large batch: split the batch range over CTAs
      const int kc = 512;
      const int ksplit = (o.K + kc - 1) / kc;
      o.i[0] = ksplit; o.i[1] = kc;
      o.ntiles *= ksplit;
      o.flags = DW_STORE_GRAD | DW_ATOMIC;
    }
    return o;
  }
  int row_tiles() const { return (cfg.batch_size + ROWS_PER_TILE - 1) / ROWS_PER_TILE; }

  Op op_gather() const {
    Op o = blank(OP_GATHER);
    o.o[0] = x_sa; o.o[1] = x_s2; o.o[2] = x_pi; o.o[3] = b_r; o.o[4] = b_d; o.o[5] = b_idx;
    o.i[0] = ldx; o.ntiles = row_tiles();
    return o;
  }
  // large batch: critic heads projected in the epilogue of the last hidden layer's tensor-core GEMM, per-row tails, delta stream
  bool tc_rows() const {
    std::string w;
    if (!tc_wanted(w) || getenv_off("SACX_TC_ROWS")) return false;
    const int L = q1.L();
    if (q1.dims[L] > TC_NMAX || (q1.dims[L] & 3)) return false;
    Op t = gemm_fwd(q1, L - 1, 0, L > 1 ? a_q[0].h[L - 2] : x_sa, L > 1 ? a_q[0].ld[L - 2] : ldx, a_q[0]);
    return tc_op_eligible(t);            // the projection needs that GEMM on the tensor-core kernel
  }
  // forward layer l of critic c; the last hidden layer carries the head projection into `head_out` when tc_rows()
  Op gemm_fwd_q(int c, int l, i64 wshift, i64 x, int ld_x, const ActSet& as, i64 head_out) const {
    const NetLayout& n = c ? q2 : q1;
    Op o = gemm_fwd(n, l, wshift, x, ld_x, as);
    if (l == n.L() - 1 && tc_rows()) { o.o[28] = n.W[n.L()] + wshift; o.o[29] = head_out; o.o[30] = n.b[n.L()] + wshift; }
    return o;
  }
  Op op_q_tail(int mode) const {
    Op o = blank(OP_Q_TAIL);
    o.mode = mode; o.act_out = q1.act_o;
    for (int c = 0; c < 2; ++c) {
      o.o[c] = b_tq[c]; o.o[2 + c] = b_q[c]; o.o[4 + c] = b_qa[c];
      o.o[10 + c] = (mode & 4) ? b_coef[c] : b_dout[c]; o.o[12 + c] = b_loss[c];
    }
    o.o[6] = b_r; o.o[7] = b_d; o.o[8] = b_lp2; o.o[9] = b_y; o.o[14] = b_lp; o.o[15] = b_ploss;
    o.ntiles = (cfg.batch_size + TAIL_ROWS - 1) / TAIL_ROWS;
    return o;
  }
  Op op_delta(bool actor) const {
    Op o = blank(OP_DELTA);
    const int L = q1.L();
    o.act = q1.act_h;
    for (int c = 0; c < 2; ++c) {
      o.o[c] = actor ? b_coef[c] : b_dout[c];
      o.o[2 + c] = (c ? q2 : q1).W[L];
      o.o[4 + c] = a_q[c].aux(L - 1);
      o.o[6 + c] = d_q[c][L - 1];
    }
    o.i[0] = a_q[0].ld[L - 1]; o.i[1] = q1.dims[L];
    o.i[2] = (cfg.batch_size + DELTA_ROWS - 1) / DELTA_ROWS;
    o.ntiles = 2 * o.i[2];
    return o;
  }
  // large batch: the policy head as [tensor-core GEMM -> one-thread-per-row tail] instead of the one-warp-per-row head op
  bool tc_heads() const {
    std::string w;
    return tc_wanted(w) && pi.dims[pi.L()] % 4 == 0 && !getenv_off("SACX_TC_HEADS");
  }
  static bool getenv_off(const char* name) { const char* v = getenv(name); return v && atoi(v) == 0; }
  Op gemm_pi_head(bool actor) const {
    const ActSet& as = actor ? a_pia : a_pit;
    const int L = pi.L();
    Op o = blank(OP_GEMM);
    o.epi = EPI_FWD; o.act = SACX_ACT_IDENTITY;            // pre-activations: the tail applies the output activation
    o.M = cfg.batch_size; o.N = 2 * cfg.act_dim; o.K = pi.dims[L];
    o.a = as.h[L - 1]; o.a_sm = as.ld[L - 1]; o.a_sk = 1;
    o.b = pi.W[L]; o.b_sk = 1; o.b_sn = o.K;
    o.bias = pi.b[L];
    o.c = actor ? b_headz_a : b_headz_t; o.ldc = rup4(2 * cfg.act_dim); o.zout = -1;
    finish_gemm(o);
    return o;
  }
  Op op_pi_tail(bool actor) const {
    Op o = blank(OP_PI_TAIL);
    o.mode = actor ? 2 : 1; o.act_out = pi.act_o;
    o.o[0] = actor ? b_headz_a : b_headz_t; o.i[3] = rup4(2 * cfg.act_dim);
    o.o[3] = actor ? x_pi : x_s2; o.i[2] = ldx;
    o.o[4] = actor ? b_lp : b_lp2;
    o.o[5] = actor ? b_eps2 : b_eps1;
    if (actor) { o.o[6] = b_tz; o.o[7] = b_se; o.o[8] = b_mask; o.o[9] = b_headz; }      // o[9]: compact copy for the head backward
    o.ntiles = (cfg.batch_size + TAIL_ROWS - 1) / TAIL_ROWS;
    return o;
  }
  Op op_pi_head(bool actor) const {
    Op o = blank(OP_PI_HEAD);
    const ActSet& as = actor ? a_pia : a_pit;
    const int L = pi.L();
    o.mode = actor ? 2 : 1; o.act_out = pi.act_o;
    o.o[0] = as.h[L - 1]; o.i[0] = as.ld[L - 1]; o.i[1] = pi.dims[L];
    o.o[1] = pi.W[L]; o.o[2] = pi.b[L];
    o.o[3] = actor ? x_pi : x_s2; o.i[2] = ldx;
    o.o[4] = actor ? b_lp : b_lp2;
    o.o[5] = actor ? b_eps2 : b_eps1;
    if (actor) { o.o[6] = b_tz; o.o[7] = b_se; o.o[8] = b_mask; o.o[9] = b_headz; }
    o.ntiles = row_tiles();
    return o;
  }
  // mode: 1 target y, 2 critic delta, 3 both chained on the same row (fused plan)
  Op op_q_row(int mode) const {
    Op o = blank(OP_Q_ROW);
    const int L = q1.L();
    o.mode = mode; o.act = q1.act_h; o.act_out = q1.act_o;
    for (int c = 0; c < 2; ++c) {
      const NetLayout& n = c ? q2 : q1;
      if (mode & 1) {
        o.o[c] = a_qt[c].h[L - 1];
        o.o[2 + c] = n.W[L] - q1.begin + T0;
        o.o[4 + c] = n.b[L] - q1.begin + T0;
        o.o[10 + c] = b_tq[c];
      }
      if (mode & 2) {
        o.o[12 + c] = a_q[c].h[L - 1]; o.o[14 + c] = a_q[c].aux(L - 1);
        o.o[16 + c] = n.W[L]; o.o[18 + c] = n.b[L];
        o.o[20 + c] = b_q[c]; o.o[22 + c] = b_dout[c]; o.o[24 + c] = d_q[c][L - 1]; o.o[26 + c] = b_loss[c];
      }
    }
    o.i[0] = a_q[0].ld[L - 1]; o.i[1] = q1.dims[L];
    o.o[6] = b_r; o.o[7] = b_d; o.o[8] = b_lp2; o.o[9] = b_y;
    o.ntiles = row_tiles();
    return o;
  }
  Op op_actor_q() const {
    Op o = blank(OP_ACTOR_Q);
    const int L = q1.L();
    o.act = q1.act_h; o.act_out = q1.act_o;
    for (int c = 0; c < 2; ++c) {
      const NetLayout& n = c ? q2 : q1;
      o.o[c] = a_q[c].h[L - 1]; o.o[2 + c] = a_q[c].aux(L - 1);
      o.o[4 + c] = n.W[L]; o.o[6 + c] = n.b[L];
      o.o[9 + c] = b_qa[c]; o.o[13 + c] = d_q[c][L - 1];
    }
    o.o[8] = b_lp; o.o[15] = b_ploss;
    o.i[0] = a_q[0].ld[L - 1]; o.i[1] = q1.dims[L];
    o.ntiles = row_tiles();
    return o;
  }
  Op op_actor_bwd() const {
    Op o = blank(OP_ACTOR_BWD);
    const int L = pi.L();
    o.act = pi.act_h; o.act_out = pi.act_o;
    for (int c = 0; c < 2; ++c) {
      o.o[c] = d_q[c][0];
      o.o[2 + c] = (c ? q2 : q1).W[0];
    }
    o.i[0] = rup4(q1.dims[1]); o.i[1] = q1.dims[1]; o.i[2] = q1.dims[0];
    o.o[4] = b_tz; o.o[5] = b_se; o.o[6] = b_mask; o.o[7] = b_headz; o.o[8] = b_dhead;
    o.o[9] = pi.W[L]; o.o[11] = a_pia.aux(L - 1); o.o[12] = d_p[L - 1];
    o.i[3] = a_pia.ld[L - 1]; o.i[4] = pi.dims[L];
    o.ntiles = row_tiles();
    return o;
  }
  Op op_prologue(int mask) const { Op o = blank(OP_PROLOGUE); o.mode = mask; o.ntiles = 1; return o; }
  Op op_final(int mode) const {
    Op o = blank(OP_FINAL);
    o.mode = mode; o.ntiles = 1;
    o.o[0] = b_loss[0]; o.o[1] = b_loss[1]; o.o[2] = b_ploss; o.o[3] = b_lp; o.o[4] = b_q[0]; o.o[5] = b_q[1]; o.o[6] = b_y;
    o.o[7] = pi_x + 3 * blk;                    // temperature-gradient share next to the policy gradients (data parallel)
    return o;
  }
  Op op_polyak() const {
    Op o = blank(OP_POLYAK);
    o.o[0] = q1.begin; o.o[1] = T0; o.o[2] = n_critic;
    o.ntiles = (int)((n_critic + FLAT_TILE - 1) / FLAT_TILE);
    return o;
  }
  Op op_adam_flat(const NetLayout& n, int opt, bool polyak) const {
    Op o = blank(OP_ADAM_FLAT);
    const i64 cnt = n.end - n.begin;
    o.opt = opt;
    o.o[0] = n.begin; o.o[1] = n.begin + blk; o.o[2] = n.begin + 2 * blk; o.o[3] = n.begin + 3 * blk; o.o[4] = cnt;
    o.o[5] = polyak ? n.begin - q1.begin + T0 : -1;
    o.ntiles = (int)((cnt + FLAT_TILE - 1) / FLAT_TILE);
    return o;
  }

  // ---------------------------------------------------------------- plan construction
  struct PB {
    Plan p;
    bool overflow = false;
    PB() { memset(&p, 0, sizeof p); }
    void phase() {
      if (p.n_phases >= MAX_PHASES) { overflow = true; return; }
      p.phases[p.n_phases] = Phase{p.n_ops, 0, 0, 0};
      p.n_phases++;
    }
    void add(const Op& o) {
      if (p.n_ops >= MAX_OPS || p.n_phases == 0) { overflow = true; return; }
      Phase& ph = p.phases[p.n_phases - 1];
      Op& d = p.ops[p.n_ops++];
      d = o;
      d.tile0 = ph.ntiles;
      ph.ntiles += d.ntiles;
      ph.nops++;
    }
  };

  // backward stages of one MLP given delta of the last hidden layer (row op) and dout = delta of the output
  // layer. Stage k: DA producing delta_{L-2-k}; DW of layer L-k; DW of layer 0 joins the last stage.
  int bwd_stages(const NetLayout& n) const { return std::max(1, n.L()); }
  void emit_bwd_stage(PB& pb, int k, const NetLayout& n, const ActSet& as, const i64* delta, i64 dout, int ld_dout,
                      i64 x, int ld_x, int opt, int flags, bool is_critic, bool with_dw) const {
    const int L = n.L();
    auto dl = [&](int l) { return delta[l]; };
    auto ldd = [&](int l) { return rup4(n.dims[l + 1]); };
    if (L - 2 - k >= 0) {   // DA: delta_{l-1} from delta_l with l = L-1-k
      const int l = L - 1 - k;
      pb.add(gemm_da(n, l, dl(l), ldd(l), dl(l - 1), ldd(l - 1), as.aux(l - 1), as.ld[l - 1]));
    }
    if (!with_dw) return;
    const int lw = L - k;     // layer whose weights get their gradient in this stage
    if (lw >= 1) {
      const i64 dy = (lw == L) ? dout : dl(lw);
      const int ldy = (lw == L) ? ld_dout : ldd(lw);
      pb.add(gemm_dw(n, lw, opt, flags, dy, ldy, as.h[lw - 1], as.ld[lw - 1], is_critic));
    }
    if (k == bwd_stages(n) - 1)   // layer 0 joins the last stage
      pb.add(gemm_dw(n, 0, opt, flags, L >= 1 ? dl(0) : dout, L >= 1 ? ldd(0) : ld_dout, x, ld_x, is_critic));
  }

  // the head of pi(s') / pi(s): one phase (row op) or two (GEMM, then tail)
  void emit_pi_head(PB& pb, bool actor) const {
    if (tc_heads()) { pb.phase(); pb.add(gemm_pi_head(actor)); pb.phase(); pb.add(op_pi_tail(actor)); }
    else { pb.phase(); pb.add(op_pi_head(actor)); }
  }
  void emit_target(PB& pb) const {
    for (int l = 0; l < pi.L(); ++l) { pb.phase(); pb.add(gemm_fwd(pi, l, 0, l ? a_pit.h[l - 1] : x_s2, l ? a_pit.ld[l - 1] : ldx, a_pit)); }
    emit_pi_head(pb, false);
    for (int l = 0; l < q1.L(); ++l) {
      pb.phase();
      for (int c = 0; c < 2; ++c)
        pb.add(gemm_fwd_q(c, l, T0 - q1.begin, l ? a_qt[c].h[l - 1] : x_s2, l ? a_qt[c].ld[l - 1] : ldx, a_qt[c], b_tq[c]));
    }
    pb.phase(); pb.add(tc_rows() ? op_q_tail(1) : op_q_row(1));
  }
  void emit_critic(PB& pb, int flags) const {
    for (int l = 0; l < q1.L(); ++l) {
      pb.phase();
      if (l == 0 && (flags & DW_ADAM)) pb.add(op_prologue((1 << OPT_Q1) | (1 << OPT_Q2)));
      for (int c = 0; c < 2; ++c) pb.add(gemm_fwd_q(c, l, 0, l ? a_q[c].h[l - 1] : x_sa, l ? a_q[c].ld[l - 1] : ldx, a_q[c], b_q[c]));
    }
    if (tc_rows()) { pb.phase(); pb.add(op_q_tail(2)); pb.phase(); pb.add(op_delta(false)); }
    else { pb.phase(); pb.add(op_q_row(2)); }
    for (int k = 0; k < bwd_stages(q1); ++k) {
      pb.phase();
      for (int c = 0; c < 2; ++c)
        emit_bwd_stage(pb, k, c ? q2 : q1, a_q[c], d_q[c], b_dout[c], 4, x_sa, ldx, c ? OPT_Q2 : OPT_Q1, flags, true, true);
      if (k == 0) pb.add(op_final(1));
    }
  }
  void emit_actor(PB& pb, int flags) const {
    for (int l = 0; l < pi.L(); ++l) {
      pb.phase();
      if (l == 0 && (flags & DW_ADAM)) pb.add(op_prologue(1 << OPT_PI));
      pb.add(gemm_fwd(pi, l, 0, l ? a_pia.h[l - 1] : x_pi, l ? a_pia.ld[l - 1] : ldx, a_pia));
    }
    emit_pi_head(pb, true);
    emit_actor_tail(pb, flags, (flags & DW_ADAM) ? 2 : (2 | 16));
  }
  // critics on (s, a~pi) -> routed dQ -> dQ/da -> head backward -> policy backward (+Adam)
  void emit_actor_tail(PB& pb, int flags, int final_mode) const {
    for (int l = 0; l < q1.L(); ++l) {
      pb.phase();
      for (int c = 0; c < 2; ++c) pb.add(gemm_fwd_q(c, l, 0, l ? a_q[c].h[l - 1] : x_pi, l ? a_q[c].ld[l - 1] : ldx, a_q[c], b_qa[c]));
    }
    if (tc_rows()) { pb.phase(); pb.add(op_q_tail(4)); pb.phase(); pb.add(op_delta(true)); }
    else { pb.phase(); pb.add(op_actor_q()); }
    for (int k = 0; k + 1 < q1.L(); ++k) {
      pb.phase();
      for (int c = 0; c < 2; ++c)
        emit_bwd_stage(pb, k, c ? q2 : q1, a_q[c], d_q[c], -1, 1, x_pi, ldx, 0, 0, true, false);
    }
    pb.phase(); pb.add(op_actor_bwd());
    for (int k = 0; k < bwd_stages(pi); ++k) {
      pb.phase();
      emit_bwd_stage(pb, k, pi, a_pia, d_p, b_dhead, 2 * cfg.act_dim, x_pi, ldx, OPT_PI, flags, false, true);
      if (k == 0 && final_mode) pb.add(op_final(final_mode));
    }
  }
  void emit_fused(PB& pb, bool gather) const {
    const int AD = DW_ADAM;
    pb.phase();
    pb.add(op_prologue(7));
    if (gather) pb.add(op_gather());
    // Forward work off the critical chain (critics on (s,a)) rides along with later phases so that no phase
    // needs two waves of tiles: pi(s'), pi(s) layer by layer; then heads + Q(s,a) layer 0; then the target critics
    // layer by layer with Q(s,a)'s deeper layers next to them.
    for (int l = 0; l < pi.L(); ++l) {
      pb.phase();
      pb.add(gemm_fwd(pi, l, 0, l ? a_pit.h[l - 1] : x_s2, l ? a_pit.ld[l - 1] : ldx, a_pit));
      pb.add(gemm_fwd(pi, l, 0, l ? a_pia.h[l - 1] : x_pi, l ? a_pia.ld[l - 1] : ldx, a_pia));
    }
    // tile order matters: tiles wrap round the 148 CTAs, so the second-wave tiles (Q2 layer 0) land on the CTAs
    // that ran Q1 layer 0 (two short GEMM tiles) and not behind a head tile
    pb.phase();
    pb.add(gemm_fwd_q(0, 0, 0, x_sa, ldx, a_q[0], b_q[0]));
    if (tc_heads()) { pb.add(gemm_pi_head(false)); pb.add(gemm_pi_head(true)); }
    else { pb.add(op_pi_head(false)); pb.add(op_pi_head(true)); }
    pb.add(gemm_fwd_q(1, 0, 0, x_sa, ldx, a_q[1], b_q[1]));
    if (tc_heads()) { pb.phase(); pb.add(op_pi_tail(false)); pb.add(op_pi_tail(true)); }
    for (int l = 0; l < q1.L(); ++l) {
      pb.phase();
      for (int c = 0; c < 2; ++c)
        pb.add(gemm_fwd_q(c, l, T0 - q1.begin, l ? a_qt[c].h[l - 1] : x_s2, l ? a_qt[c].ld[l - 1] : ldx, a_qt[c], b_tq[c]));
      if (l + 1 < q1.L())
        for (int c = 0; c < 2; ++c) pb.add(gemm_fwd_q(c, l + 1, 0, a_q[c].h[l], a_q[c].ld[l], a_q[c], b_q[c]));
    }
    if (tc_rows()) { pb.phase(); pb.add(op_q_tail(3)); pb.phase(); pb.add(op_delta(false)); }
    else { pb.phase(); pb.add(op_q_row(3)); }      // target y and critic delta chained on the same row: one phase
    for (int k = 0; k < bwd_stages(q1); ++k) {   // critic Adam with the Polyak update fused behind it (K10)
      pb.phase();
      for (int c = 0; c < 2; ++c)
        emit_bwd_stage(pb, k, c ? q2 : q1, a_q[c], d_q[c], b_dout[c], 4, x_sa, ldx, c ? OPT_Q2 : OPT_Q1, AD | DW_POLYAK, true, true);
    }
    emit_actor_tail(pb, AD, 1 | 2 | 4 | 8);
  }

  // ---- row-parallel program (sacx_rowpar.cuh) -----------------------------------------------------------------------
  bool rowpar_eligible(std::string& why) const {
    const char* env = getenv("SACX_ROWPAR");
    if (env && atoi(env) == 0) { why = "disabled by SACX_ROWPAR=0"; return false; }
    if (cfg.n_agents != 1) { why = "population mode"; return false; }
    if (cfg.dp_world > 1) { why = "data-parallel mode"; return false; }
    { std::string w; if (tc_wanted(w)) { why = "large batch runs the tensor-core path"; return false; } }
    // measured (Donkey latent shape, batch 1024): 4 row blocks per group cost more than the 64x64 FFMA tiles save in
    // barriers -- 1932 vs 2358 updates/s; SACX_ROWPAR=1 still forces this kernel
    if (cfg.batch_size > 512 && !(env && atoi(env) == 1)) { why = "batch above 512: the tile-parallel kernel is faster"; return false; }
    if (pi.L() < 2 || q1.L() < 2) { why = "fewer than two hidden layers"; return false; }
    if (act_needs_z(pi.act_h) || act_needs_z(q1.act_h)) { why = "hidden activation needs saved pre-activations"; return false; }
    if (cfg.act_dim > RP_MAXA) { why = "action dimension above 8"; return false; }
    if (2 * cfg.obs_dim + cfg.act_dim + 2 > 256) { why = "observation wider than 123"; return false; }
    for (const NetLayout* n : {&pi, &q1})
      for (int l = 1; l <= n->L(); ++l)
        if (n->dims[l] != 64 && n->dims[l] != 128 && n->dims[l] != 256) { why = "hidden width not 64/128/256"; return false; }
    if (2 * (q1.L() + 1) + (pi.L() + 1) + 1 > RP_MAX_DW_OPS) { why = "network too deep"; return false; }
    return true;
  }

  bool build_rowpar(PB& pb) {
    RpProgram& P = h_prog;
    memset(&P, 0, sizeof P);
    const int O = cfg.obs_dim, A = cfg.act_dim, Lq = q1.L(), Lp = pi.L();
    bool overflow = false;
    // wmax: floats of the widest weight slice (sizes the slots); red: floats of the k-group reduction buffer.
    // wcap: a pair with two slices runs as one job only if both fit in a slot sized for single slices (set by a first pass)
    int wmax = 0, red = 0, wcap = 0;
    auto step = [&](int row_op) {
      if (P.n_steps_a + P.n_steps_c >= RP_MAX_STEPS) { overflow = true; return; }
      RpStep& st = P.steps[P.n_steps_a + P.n_steps_c];
      st.row_op = row_op; st.job0 = P.n_jobs; st.njobs = 0; st.load0 = P.n_loads; st.nloads = 0;
    };
    auto cur = [&]() -> RpStep& { return P.steps[P.n_steps_a + P.n_steps_c]; };
    // TMA-staged slice (sacx_rowpar.cuh): 32 columns per CTA, rows the tensor map can address
    auto tma_ok = [&](const RpJob& j, i64 w) { return rp_tma && j.N / RP_CS == 32 && (j.w_ld % 4) == 0 && (w % 4) == 0 && j.K <= 256; };
    auto slice_floats = [&](const RpJob& j, bool tma) {
      const int NS = j.N / RP_CS;
      if (tma) return j.bkm ? j.K * 32 : ((j.K + 31) / 32) * 1024;
      return j.bkm ? j.K * NS : NS * (j.Kp + 4);
    };
    // two slices of a pair: a TMA-staged second slice starts at a 1 KB granule (swizzled tiles) behind the first, placed so that
    // the cp.async layout fits as well (the slices fall back to it when a tensor map cannot be encoded); a cp.async-only slice
    // needs 16-byte alignment only
    auto pair_w2_off = [&](const RpJob& j, bool tma) {
      if (!tma) return (slice_floats(j, false) + 3) & ~3;
      return (std::max(slice_floats(j, true), slice_floats(j, false)) + 255) & ~255;
    };
    auto add_job = [&](const RpJob& j) {
      if (P.n_jobs >= RP_MAX_JOBS) { overflow = true; return; }
      const int NS = j.N / RP_CS;
      RpJob jj = j;
      const bool sep = j.pair && j.w2 != j.w;
      jj.tma = (tma_ok(j, j.w) && (!sep || tma_ok(j, j.w2))) ? 1 : 0;
      jj.map = 2 * P.n_jobs; jj.map2 = 2 * P.n_jobs + 1;      // tensor maps of the two halves' slices
      jj.w2_off = sep ? pair_w2_off(j, jj.tma) : 0;
      P.jobs[P.n_jobs++] = jj; cur().njobs++;
      wmax = std::max(wmax, jj.w2_off + (sep ? jj.w2_off : slice_floats(j, jj.tma)));
      red = std::max(red, (1 + j.pair) * (64 / NS) * RP_RB * (NS + 8));      // k-groups (8 warps x 8 columns / NS) x [16][NS + 8]
    };
    // two independent forward jobs of the same shape as one pair job (fewer fixed per-job costs: waits, barriers, issue,
    // reduction and epilogue). Either the weight slice is shared (pi(s') / pi(s): W, bias and head weights are the policy's), or
    // each half has its own slice and bias and no projection (the critics' first layers: never the last hidden layer).
    // Pairing shortens the job sequence, and rp_run_steps issues job j + 2's operands when job j starts. A backward job's
    // aux operand (the saved activations of layer l - 1) must therefore come from a job at least three positions earlier.
    // That holds because the last hidden layer, whose backward job follows right after, carries the head projection and
    // so never pairs with its twin: its two single jobs keep that distance for the layer in front of it.
    auto add_pair = [&](const RpJob& a, const RpJob& b) {
      const bool shared = a.w == b.w && a.bias == b.bias && a.proj_w == b.proj_w;
      bool ok = wcap > 0 && !a.bkm && !b.bkm && a.K == b.K && a.N == b.N && a.act == b.act && a.w_ld == b.w_ld &&
                a.out_ld == b.out_ld && a.proj_J == b.proj_J && (shared || a.proj_J == 0);
      if (ok && !shared) {
        const bool tma = tma_ok(a, a.w) && tma_ok(a, b.w);
        ok = 2 * pair_w2_off(a, tma) <= wcap && (!tma || 2 * ((a.K + 31) / 32) <= 8);      // (one TMA tile per warp)
      }
      if (!ok) { add_job(a); add_job(b); return; }
      RpJob j = a;
      j.pair = 1; j.a_src2 = b.a_src; j.out2 = b.out; j.proj_slot2 = b.proj_slot; j.w2 = b.w; j.bias2 = b.bias;
      add_job(j);
    };
    auto add_load = [&](i64 off, int ld, int K, int abuf) {
      if (P.n_loads >= RP_MAX_LOADS) { overflow = true; return; }
      P.loads[P.n_loads++] = RpLoad{off, ld, K, abuf, 0}; cur().nloads++;
    };
    auto fwd = [&](const NetLayout& n, int l, i64 wshift, int a_src, const ActSet& as, int slot) {
      RpJob j; memset(&j, 0, sizeof j);
      j.bkm = 0; j.a_src = a_src; j.K = n.dims[l]; j.Kp = (j.K + 7) & ~7; j.N = n.dims[l + 1]; j.act = n.act_h;
      j.ns_log2 = j.N == 256 ? 5 : (j.N == 128 ? 4 : 3);
      j.w = n.W[l] + wshift; j.w_ld = j.K; j.bias = n.b[l] + wshift; j.out = as.h[l]; j.out_ld = as.ld[l]; j.aux = -1; j.proj_w = -1;
      if (l == n.L() - 1) {
        j.proj_J = n.dims[n.L() + 1]; j.proj_slot = slot; j.proj_w = n.W[n.L()] + wshift; j.proj_sj = n.dims[n.L()]; j.proj_sn = 1;
      }
      return j;
    };
    // delta_l (full rows in a_src) -> delta_{l-1} slice, through W_l
    auto bwd = [&](const NetLayout& n, int l, int a_src, const ActSet& as, const i64* delta, int da_slot) {
      RpJob j; memset(&j, 0, sizeof j);
      j.bkm = 1; j.a_src = a_src; j.K = n.dims[l + 1]; j.Kp = j.K; j.N = n.dims[l]; j.act = n.act_h;
      j.ns_log2 = j.N == 256 ? 5 : (j.N == 128 ? 4 : 3);
      j.w = n.W[l]; j.w_ld = n.dims[l]; j.bias = -1; j.aux = as.h[l - 1]; j.aux_ld = as.ld[l - 1];
      j.out = delta[l - 1]; j.out_ld = rup4(n.dims[l]); j.proj_w = -1;
      if (da_slot >= 0) { j.proj_J = A; j.proj_slot = da_slot; j.proj_w = n.W[0] + O; j.proj_sj = 1; j.proj_sn = n.dims[0]; }
      return j;
    };
    const i64 tsh = T0 - q1.begin;
    auto emit = [&]() {
      // ---------------- phase A: pi(s'), pi(s), Q(s,a) forward; target critics; Bellman target; critics' backward
      step(RPR_GATHER);
      add_pair(fwd(pi, 0, 0, RPS_XS2, a_pit, RPP_PI_T), fwd(pi, 0, 0, RPS_XSA, a_pia, RPP_PI_A));
      add_pair(fwd(q1, 0, 0, RPS_XSA, a_q[0], RPP_Q1), fwd(q2, 0, 0, RPS_XSA, a_q[1], RPP_Q2));
      P.n_steps_a++;
      for (int l = 1; l < std::max(Lp, Lq); ++l) {
        step(RPR_NONE);
        if (l < Lp) {
          add_load(a_pit.h[l - 1], a_pit.ld[l - 1], pi.dims[l], 0);
          add_load(a_pia.h[l - 1], a_pia.ld[l - 1], pi.dims[l], 1);
          add_pair(fwd(pi, l, 0, 0, a_pit, RPP_PI_T), fwd(pi, l, 0, 1, a_pia, RPP_PI_A));
        }
        if (l < Lq) {
          for (int c = 0; c < 2; ++c) add_load(a_q[c].h[l - 1], a_q[c].ld[l - 1], q1.dims[l], 2 + c);
          add_pair(fwd(q1, l, 0, 2, a_q[0], RPP_Q1), fwd(q2, l, 0, 3, a_q[1], RPP_Q2));
        }
        P.n_steps_a++;
      }
      step(RPR_PI_HEADS);
      add_pair(fwd(q1, 0, tsh, RPS_XS2, a_qt[0], RPP_QT1), fwd(q2, 0, tsh, RPS_XS2, a_qt[1], RPP_QT2));
      P.n_steps_a++;
      for (int l = 1; l < Lq; ++l) {
        step(RPR_NONE);
        for (int c = 0; c < 2; ++c) add_load(a_qt[c].h[l - 1], a_qt[c].ld[l - 1], q1.dims[l], c);
        add_pair(fwd(q1, l, tsh, 0, a_qt[0], RPP_QT1), fwd(q2, l, tsh, 1, a_qt[1], RPP_QT2));
        P.n_steps_a++;
      }
      step(RPR_TARGET_CRITIC);
      for (int c = 0; c < 2; ++c) {
        add_load(a_q[c].h[Lq - 1], a_q[c].ld[Lq - 1], q1.dims[Lq], 2 + c);
        add_job(bwd(c ? q2 : q1, Lq - 1, 2 + c, a_q[c], d_q[c], -1));
      }
      P.n_steps_a++;
      for (int l = Lq - 2; l >= 1; --l) {
        step(RPR_NONE);
        for (int c = 0; c < 2; ++c) {
          add_load(d_q[c][l], rup4(q1.dims[l + 1]), q1.dims[l + 1], c);
          add_job(bwd(c ? q2 : q1, l, c, a_q[c], d_q[c], -1));
        }
        P.n_steps_a++;
      }
      // ---------------- phase C: critics on (s, a~pi), routed dQ back to the action, policy backward
      step(RPR_RELOAD);
      add_pair(fwd(q1, 0, 0, RPS_XPI, a_q[0], RPP_Q1), fwd(q2, 0, 0, RPS_XPI, a_q[1], RPP_Q2));
      P.n_steps_c++;
      for (int l = 1; l < Lq; ++l) {
        step(RPR_NONE);
        for (int c = 0; c < 2; ++c) add_load(a_q[c].h[l - 1], a_q[c].ld[l - 1], q1.dims[l], c);
        add_pair(fwd(q1, l, 0, 0, a_q[0], RPP_Q1), fwd(q2, l, 0, 1, a_q[1], RPP_Q2));
        P.n_steps_c++;
      }
      step(RPR_ACTOR_Q);
      for (int c = 0; c < 2; ++c) {
        add_load(a_q[c].h[Lq - 1], a_q[c].ld[Lq - 1], q1.dims[Lq], 2 + c);
        add_job(bwd(c ? q2 : q1, Lq - 1, 2 + c, a_q[c], d_q[c], Lq - 1 == 1 ? RPP_DA1 + c : -1));
      }
      P.n_steps_c++;
      for (int l = Lq - 2; l >= 1; --l) {
        step(RPR_NONE);
        for (int c = 0; c < 2; ++c) {
          add_load(d_q[c][l], rup4(q1.dims[l + 1]), q1.dims[l + 1], c);
          add_job(bwd(c ? q2 : q1, l, c, a_q[c], d_q[c], l == 1 ? RPP_DA1 + c : -1));
        }
        P.n_steps_c++;
      }
      step(RPR_PI_BWD);
      add_load(a_pia.h[Lp - 1], a_pia.ld[Lp - 1], pi.dims[Lp], 0);
      add_job(bwd(pi, Lp - 1, 0, a_pia, d_p, -1));
      P.n_steps_c++;
      for (int l = Lp - 2; l >= 1; --l) {
        step(RPR_NONE);
        add_load(d_p[l], rup4(pi.dims[l + 1]), pi.dims[l + 1], 1);
        add_job(bwd(pi, l, 1, a_pia, d_p, -1));
        P.n_steps_c++;
      }
    };
    // first pass with single jobs only: the widest single slice sizes the slots, and a pair with two slices runs as one job
    // only if they fit in one of those slots
    emit();
    wcap = wmax;
    P.n_steps_a = P.n_steps_c = P.n_jobs = P.n_loads = 0;
    wmax = red = 0; overflow = false;
    emit();
    if (overflow) { rp_why = "program tables too small"; return false; }
    // ---------------- geometry, row-op operands
    P.O = O; P.A = A; P.Hq = q1.dims[Lq]; P.Hpi = pi.dims[Lp]; P.ld_hq = rup4(P.Hq); P.ld_hpi = rup4(P.Hpi);
    P.act_q = q1.act_h; P.act_oq = q1.act_o; P.act_pi = pi.act_h; P.act_opi = pi.act_o;
    P.ab_q[0] = 2; P.ab_q[1] = 3; P.ab_pi = 0;
    P.x_sa = x_sa; P.x_s2 = x_s2; P.x_pi = x_pi; P.b_r = b_r; P.b_d = b_d; P.b_idx = b_idx; P.b_eps1 = b_eps1; P.b_eps2 = b_eps2;
    P.b_lp2 = b_lp2; P.b_lp = b_lp; P.b_y = b_y; P.b_ploss = b_ploss; P.b_tz = b_tz; P.b_se = b_se; P.b_mask = b_mask;
    P.b_headz = b_headz; P.b_dhead = b_dhead;
    for (int c = 0; c < 2; ++c) {
      const NetLayout& n = c ? q2 : q1;
      P.b_tq[c] = b_tq[c]; P.b_q[c] = b_q[c]; P.b_qa[c] = b_qa[c]; P.b_dout[c] = b_dout[c]; P.b_loss[c] = b_loss[c];
      P.q_bL[c] = n.b[Lq]; P.q_WL[c] = n.W[Lq]; P.qt_bL[c] = n.b[Lq] + tsh; P.dq_last[c] = d_q[c][Lq - 1];
    }
    P.pi_bL = pi.b[Lp]; P.pi_WL = pi.W[Lp]; P.dp_last = d_p[Lp - 1];
    // ---------------- shared-memory layout (floats)
    int hmax = 0;
    for (int l = 1; l <= Lp; ++l) hmax = std::max(hmax, pi.dims[l]);
    for (int l = 1; l <= Lq; ++l) hmax = std::max(hmax, q1.dims[l]);
    P.lda = hmax + 4; P.abuf_floats = RP_RB * P.lda;
    P.ldx = ((O + A + 7) & ~7) + 4;
    P.gldx = ldx;
    P.wslot_floats = ((wmax + 255) & ~255) + 1024;   // (1 KB granules: swizzled TMA tiles) + epilogue operand [16][32] + projection weights [16][32]
    int off = 0;
    P.sm_abuf = off; off += RP_NABUF * P.abuf_floats;
    P.sm_xbuf = off; off += 3 * RP_RB * P.ldx;
    off = (off + 255) & ~255;
    P.sm_wslot = off; off += RP_NWSLOT * P.wslot_floats;
    P.sm_red = off; off += red;
    P.sm_otile = off; P.sm_pw = off;
    off = std::max(off, WSM_FLOATS + CfgSmall::SMEM_FLOATS);
    off = std::max(off, RP_DW_SMEM);      // the dW tiles alias the same region
    P.sm_total = off;
    // partial-sum scratch of one group (global memory): [slot][rank][16][J]
    const int J[RPP_N] = {2 * A, 2 * A, 1, 1, 1, 1, A, A};
    int poff = 0;
    for (int i = 0; i < RPP_N; ++i) { P.part_off[i] = poff; poff += RP_CS * RP_RB * J[i]; }
    P.part_stride = (poff + 31) & ~31;
    // ---------------- the two tile-parallel phases: dW + Adam (+ Polyak) of the critics, then of the policy
    const bool keep_large = large;
    large = false;
    const int AD = DW_ADAM;
    pb.phase();
    for (int l = Lq - 1; l >= 1; --l)
      for (int c = 0; c < 2; ++c)
        pb.add(gemm_dw(c ? q2 : q1, l, c ? OPT_Q2 : OPT_Q1, AD | DW_POLYAK, d_q[c][l], rup4(q1.dims[l + 1]), a_q[c].h[l - 1], a_q[c].ld[l - 1], true));
    for (int c = 0; c < 2; ++c) {
      pb.add(gemm_dw(c ? q2 : q1, 0, c ? OPT_Q2 : OPT_Q1, AD | DW_POLYAK, d_q[c][0], rup4(q1.dims[1]), x_sa, ldx, true));
      pb.add(gemm_dw(c ? q2 : q1, Lq, c ? OPT_Q2 : OPT_Q1, AD | DW_POLYAK, b_dout[c], 4, a_q[c].h[Lq - 1], a_q[c].ld[Lq - 1], true));
    }
    pb.phase();
    for (int l = Lp - 1; l >= 1; --l) pb.add(gemm_dw(pi, l, OPT_PI, AD, d_p[l], rup4(pi.dims[l + 1]), a_pia.h[l - 1], a_pia.ld[l - 1], false));
    pb.add(gemm_dw(pi, 0, OPT_PI, AD, d_p[0], rup4(pi.dims[1]), x_pi, ldx, false));
    pb.add(gemm_dw(pi, Lp, OPT_PI, AD, b_dhead, 2 * A, a_pia.h[Lp - 1], a_pia.ld[Lp - 1], false));
    pb.add(op_final(1 | 2 | 4 | 8));
    large = keep_large;
    if (pb.overflow || pb.p.n_ops > RP_MAX_DW_OPS) { rp_why = "too many dW ops"; return false; }
    return true;
  }

  int build_plans() {
    h_plans.assign(N_PLANS, Plan());
    auto put = [&](int id, PB& pb) -> int {
      if (pb.overflow) return fail(SACX_ERR_INVALID, "network too deep for the op table (MAX_OPS/MAX_PHASES)");
      h_plans[id] = pb.p;
      return SACX_OK;
    };
    int rc;
    { PB pb; emit_fused(pb, true); if ((rc = put(PLAN_FUSED, pb))) return rc; }
    { PB pb; emit_fused(pb, false); if ((rc = put(PLAN_FUSED_NOGATHER, pb))) return rc; }
    { PB pb; pb.phase(); pb.add(op_gather()); if ((rc = put(PLAN_SAMPLE, pb))) return rc; }
    { PB pb; emit_target(pb); if ((rc = put(PLAN_TARGET, pb))) return rc; }
    { PB pb; emit_critic(pb, DW_ADAM); if ((rc = put(PLAN_CRITIC, pb))) return rc; }
    { PB pb; emit_critic(pb, DW_STORE_GRAD); if ((rc = put(PLAN_CRITIC_GRADS, pb))) return rc; }
    { PB pb; emit_actor(pb, DW_ADAM); if ((rc = put(PLAN_ACTOR, pb))) return rc; }
    { PB pb; emit_actor(pb, DW_STORE_GRAD); if ((rc = put(PLAN_ACTOR_GRADS, pb))) return rc; }
    grads_atomic = false;
    for (int id : {PLAN_CRITIC_GRADS, PLAN_ACTOR_GRADS})
      for (int i = 0; i < h_plans[id].n_ops; ++i)
        if (h_plans[id].ops[i].type == OP_GEMM && (h_plans[id].ops[i].flags & DW_ATOMIC)) grads_atomic = true;
    { PB pb; pb.phase(); pb.add(op_final(4)); if ((rc = put(PLAN_ALPHA, pb))) return rc; }
    { PB pb; pb.phase(); pb.add(op_final(32 | 8)); if ((rc = put(PLAN_ALPHA_APPLY, pb))) return rc; }
    { PB pb; pb.phase(); pb.add(op_polyak()); pb.add(op_final(8)); if ((rc = put(PLAN_POLYAK, pb))) return rc; }
    for (int pol = 0; pol < 2; ++pol) {
      PB pb;
      pb.phase(); pb.add(op_prologue((1 << OPT_Q1) | (1 << OPT_Q2)));
      pb.phase(); pb.add(op_adam_flat(q1, OPT_Q1, pol)); pb.add(op_adam_flat(q2, OPT_Q2, pol));
      if ((rc = put(pol ? PLAN_APPLY_Q_POLYAK : PLAN_APPLY_Q, pb))) return rc;
    }
    { PB pb; pb.phase(); pb.add(op_prologue(1 << OPT_PI)); pb.phase(); pb.add(op_adam_flat(pi, OPT_PI, false));
      if ((rc = put(PLAN_APPLY_PI, pb))) return rc; }
    rp = rowpar_eligible(rp_why);
    if (rp) { PB pb; rp = build_rowpar(pb); if (rp) h_plans[PLAN_RP] = pb.p; }
    return SACX_OK;
  }

  // ---- tensor-core path ------------------------------------------------------------------------------------------------
  bool tc_op_eligible(const Op& o) const {
    if (o.type != OP_GEMM || o.zout >= 0) return false;
    auto al = [](i64 x) { return x >= 0 && (x & 3) == 0; };
    if (o.N > TC_NMAX) return false;
    if (o.epi == EPI_DACT && (o.N < 16 || (o.N & 3))) return false;
    if (o.epi == EPI_FWD && o.N < 1) return false;                        // narrow heads: UMMA N = 16, weight rows beyond N read as zero
    // dW: any width (B operand rows are 16B-aligned batch rows)
    if (o.epi == EPI_FWD)
      return o.M >= tc_min_m && o.a_sk == 1 && o.b_sk == 1 && !(o.a_sm & 3) && !(o.b_sn & 3) && !(o.ldc & 3) && al(o.a) && al(o.b) &&
             al(o.c) && al(o.bias) && o.K >= 4;
    if (o.epi == EPI_DACT)
      return o.M >= tc_min_m && o.a_sk == 1 && o.b_sn == 1 && !(o.a_sm & 3) && !(o.b_sk & 3) && !(o.ldc & 3) && !(o.ld_aux & 3) &&
             al(o.a) && al(o.b) && al(o.c) && al(o.aux) && !(o.K & 3);
    if (o.epi == EPI_DW)
      return o.K >= tc_min_m && o.M >= 1 && o.a_sm == 1 && o.b_sn == 1 && !(o.a_sk & 3) && !(o.b_sk & 3) && al(o.a) &&
             al(o.b) && o.p >= 0;
    return false;
  }
  bool tc_wanted(std::string& why) const {
    const char* env = getenv("SACX_TC");
    if (env && atoi(env) == 0) { why = "disabled by SACX_TC=0"; return false; }
    if (tc_forbid) { why = "tensor-core setup failed"; return false; }
    if (cfg.n_agents == 1 && cfg.batch_size < tc_min_batch) { why = "batch below the tensor-core threshold"; return false; }
    if (cfg.n_agents > 1) {      // population: every agent contributes >= one 128-row tile; enough agents to fill the chip
      const char* pe = getenv("SACX_TC_POP");
      if (pe && atoi(pe) == 0) { why = "disabled by SACX_TC_POP=0"; return false; }
      if (cfg.n_agents > 65535) { why = "more than 65535 agents (grid.z of the dW reduce kernel)"; return false; }
      if (cfg.batch_size < 128 || (long long)cfg.n_agents * cfg.batch_size < 4LL * tc_min_batch) {
        why = "population too small for the tensor-core path"; return false;
      }
    }
    if (act_needs_z(pi.act_h) || act_needs_z(q1.act_h)) { why = "hidden activation needs saved pre-activations"; return false; }
    return true;
  }

  int max_phase_tiles() const {
    int m = 1;
    for (const Plan& p : h_plans)
      for (int i = 0; i < p.n_phases; ++i) m = std::max(m, p.phases[i].ntiles);
    return m;
  }
};

}  // namespace sacx
