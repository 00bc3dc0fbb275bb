// Shared host/device types of the fused SAC update engine: the op table ("plan") that the
// persistent kernel interprets, per-agent scalar state, and launch arguments.
#pragma once
#include <stdint.h>

namespace sacx {

typedef long long i64;

enum OpType : int {
  OP_NONE = 0,
  OP_GATHER,      // ring rows -> batch buffers (a2/a3: replay_buffer.py:32-39, agent.py:166-193)
  OP_GEMM,        // tiled FP32 GEMM with fused epilogue (a4 forward, backward dA, backward dW+Adam)
  OP_PI_HEAD,     // policy output layer + tanh-Gaussian rsample/log_prob (a5: models.py:73-87)
  OP_Q_ROW,       // critic output layers: soft Bellman target y (a6, mode&1) and/or MSE delta + delta of the last hidden layer (a7, mode&2)
  OP_ACTOR_Q,     // critics' heads on (s, a~pi): min, policy loss rows, routed dQ (a8)
  OP_ACTOR_BWD,   // dQ/da through layer 0, head backward, policy delta of last hidden (a8)
  OP_PROLOGUE,    // per-update scalars: Adam step/bias corrections (a11)
  OP_FINAL,       // loss means, temperature step (a9), counters
  OP_POLYAK,      // standalone soft target update (a10)
  OP_ADAM_FLAT,   // Adam over a packed gradient block (data-parallel apply)
  OP_LOAD_EXT,    // copy external y / logpi into arena buffers
  OP_PI_TAIL,     // large batch: rsample / tanh squash / log_prob from head pre-activations a tensor-core GEMM produced (one thread per row)
  OP_Q_TAIL,      // large batch: Bellman target / critic loss gradient / actor routing from head values the GEMM epilogue projected (one thread per row)
  OP_DELTA,       // large batch: delta of the critics' last hidden layer, coef[b] * W_L[k] * act'(h[b][k]) (element-wise stream)
};

enum Epi : int { EPI_FWD = 1, EPI_DACT = 2, EPI_DW = 3 };
enum DwFlags : int { DW_STORE_GRAD = 1, DW_ADAM = 2, DW_POLYAK = 4, DW_ATOMIC = 8 };
enum OptId : int { OPT_PI = 0, OPT_Q1 = 1, OPT_Q2 = 2, OPT_ALPHA = 3, N_OPT = 4 };

// One schedulable operation. All `long long` fields are float32-word offsets from the agent's
// arena base (or -1 when unused).
struct Op {
  int type, mode, act, act_out;
  int tile0, ntiles, tiles_n, cfg;
  // GEMM: C[M,N] = sum_k A(m,k) * B(k,n);  A(m,k) = a[m*a_sm + k*a_sk], B(k,n) = b[k*b_sk + n*b_sn]
  int M, N, K, epi;
  int a_sm, a_sk, b_sk, b_sn;
  int ldc, ld_aux, a_vec, b_vec;
  i64 a, b, c, bias, aux, zout;
  // EPI_DW: parameter / Adam / target / gradient blocks for the weight (ld = K_in) and its bias
  i64 p, pm, pv, pt, pg;
  i64 pb, pbm, pbv, pbt, pbg;
  int opt, flags;
  // row ops: generic slots (documented at each op's builder)
  i64 o[32];
  int i[8];
  float f[4];
};

struct Phase {
  int op0, nops, ntiles, pad;
};

constexpr int MAX_OPS = 112;
constexpr int MAX_PHASES = 48;

struct Plan {
  int n_phases, n_ops, pad0, pad1;
  Phase phases[MAX_PHASES];
  Op ops[MAX_OPS];
};

// Per-agent scalar state (lives in the arena at `scal_off`, 8-byte aligned).
struct AgentScalars {
  double log_alpha, alpha_m, alpha_v, alpha;         // F6: float64 temperature state
  i64 step[N_OPT];                                   // Adam step counters (pi, q1, q2, alpha)
  i64 updates;                                       // completed updates (device RNG counter)
  double alpha_lr;                                   // per-agent temperature learning rate (population of trials); 0: Hyper.alpha_lr
  float alpha_f32;                                   // alpha as used by target/actor (F5)
  float adam_step_size[3];                           // lr / (1 - beta1^t)      per optimiser
  float adam_bc2_sqrt[3];                            // sqrt(1 - beta2^t)
  float pad;
  float metrics[12];                                 // q1_loss q2_loss policy_loss alpha_loss alpha log_alpha q1_mean q2_mean logpi_mean y_mean
  int nonfinite;
  float dp_mean_t, dp_mean_lt;                       // data parallel: this rank's share of mean(logpi + H), mean(log_alpha (logpi + H))
  int pad2[1];
  // per-agent hyper-parameters (a population of Optuna trials: hparam_search/scripts/run_search.py:24-39 is generic over any
  // section/param of the YAML). Initialised from the config by sacx_agent_reset_state / create; overwritten per agent through the layout.
  double lr[3];                                      // actor / critic / critic learning rates; 0: Hyper.lr
  float gamma, tau, one_minus_tau;                   // sac.gamma, sac.tau, (float)(1.0 - tau)
  unsigned rng_agent;                                // second key word of the device RNG streams: the GLOBAL agent id
  unsigned long long rng_seed;                       // first key of the device index / normal / rollout-noise streams (train.seed or the agent's own seed)
};

struct RingMeta {          // one per agent, at the head of the agent's ring block
  i64 pushes;
  i64 reserved[3];
};

struct Hyper {
  float gamma, tau, one_minus_tau, log_std_min, log_std_max, action_scale;
  double lr[3];
  double alpha_lr, alpha_init;
  float target_entropy;
  int auto_alpha;
  int obs, act, B, B_global, row0_global;            // data-parallel: this rank's rows are [row0, row0+B)
  int n_step;                                        // buffer.n_step in 1..16: returns folded into the gathered batch
  unsigned long long seed;
};

struct RunArgs {
  float* arena;
  i64 agent_stride;          // float words
  float* ring;               // ring arena base (may be null when no gather op runs)
  i64 ring_stride;           // float words per agent ring block
  i64 ring_capacity;
  // ring field offsets (float words from the agent's ring block)
  i64 ring_s, ring_a, ring_r, ring_s2, ring_d;   // field offsets inside a record (+ ring header): element i of field f of slot k = ring[f + k * ring_rs + i]
  i64 ring_rs;               // floats per packed record [s | s2 | a | r | d | pad]
  const i64* idx_ext;        // [n_steps, n_agents, B] or null
  const float* eps1_ext;     // [n_steps, n_agents, B, A] or null
  const float* eps2_ext;
  const float* y_ext;        // staged critic step: external y [B] or null
  const float* lp_ext;       // staged alpha step: external logpi [B] or null
  const float* w_ext;        // per-row weights of the critic loss [B] (prioritized replay; launches of one update only) or null
  int n_steps, n_agents;
  int phase_begin, phase_end;
  int ctas_per_agent;
  unsigned* barrier;         // [agent_slots] monotonic counters (zero when the launch starts)
  unsigned* barrier_next;    // row-parallel kernel: the counter set of the NEXT launch, zeroed by this one (no memset per launch)
  float* metrics_host;       // row-parallel kernel: pinned host copy of the scalar block, written by the kernel itself, or null
  i64 scal_off;
  unsigned long long* dbg;   // optional [n_steps][n_phases][gridDim.x][2] clock64 at barrier arrive / release
  unsigned long long* dbg2;  // optional [n_steps][n_phases][gridDim.x][8] intra-tile timestamps of the CTA's last GEMM tile
  int tc_skip;               // 1: GEMM ops marked for the tensor-core path (op.cfg & 2) are run by sacx_tc_kernel, skip them here
  float* rp_part;            // row-parallel kernel: partial-sum scratch [groups][part_stride]
  const void* rp_maps;       // row-parallel kernel: device array of CUtensorMap (128 B each) for the TMA-staged weight slices, or null
  Hyper hp;
};

}  // namespace sacx
