/*
 * sacx.h -- C ABI of the B200-native SAC update engine (libsacx.so, sm_100a).
 *
 * The reference (ignaschuemer7/soft-actor-critic) has no FFI: its boundary for the
 * hot path is the Python class surface of sac/agent.py and sac/replay_buffer.py.
 * Every entry point below replaces one of those methods; the Python package `sac`
 * shipped in this repo is the binding a maintainer would add (ctypes, see
 * INTEGRATION.md).  Plain pointers and sizes only; no torch types cross this line.
 *
 * Pointer convention: `*_dev` = CUDA device pointer, `*_host` = host pointer
 * (pinned preferred).  All float data is IEEE fp32 unless stated; indices int64.
 * All functions return SACX_OK (0) or a negative status; the message of the last
 * failure on the calling thread is available from sacx_last_error().
 * Work is enqueued on the handle's stream (sacx_*_set_stream); calls with a
 * `_host` output synchronise that stream before returning.
 */
#ifndef SACX_H_
#define SACX_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SACX_VERSION 100

/* status codes -> Python exceptions raised by the shim */
#define SACX_OK               0
#define SACX_ERR_INVALID     -1  /* ValueError: bad argument / unsupported shape                    */
#define SACX_ERR_UNDERFILLED -2  /* ValueError: fewer stored transitions than batch_size            */
                                 /*   (reference: sac/replay_buffer.py:34-38)                       */
#define SACX_ERR_CUDA        -3  /* RuntimeError: CUDA runtime failure (no device, launch error)    */
#define SACX_ERR_ACTIVATION  -4  /* KeyError: unknown activation (reference: sac/models.py:138-139) */
#define SACX_ERR_NONFINITE   -5  /* ValueError: NaN/Inf policy head (torch Normal validate_args)    */
#define SACX_ERR_EMPTY_HIDDEN -6 /* ValueError: hidden_sizes empty (reference: sac/models.py:135-136) */

#define SACX_MAX_HIDDEN 8        /* hidden layers per network                                       */
#define SACX_MAX_ACT    32       /* action dimension                                                */

/* activation ids: reference sac/models.py:104-112 (_ACTIVATIONS) */
enum sacx_activation {
  SACX_ACT_IDENTITY = 0, SACX_ACT_RELU = 1, SACX_ACT_TANH = 2, SACX_ACT_ELU = 3,
  SACX_ACT_LEAKY_RELU = 4, SACX_ACT_GELU = 5, SACX_ACT_SELU = 6
};
/* name -> id, SACX_ERR_ACTIVATION when unknown */
int sacx_activation_id(const char* name);

/* Mirrors the YAML config consumed by SAC.__init__ (reference: sac/agent.py:22-115,
 * configs/example_config_env.yaml): sections sac / q_net / policy_net / buffer / train. */
typedef struct sacx_config {
  int32_t obs_dim, act_dim;
  int32_t n_hidden_pi;  int32_t hidden_pi[SACX_MAX_HIDDEN];   /* policy_net.hidden_sizes       */
  int32_t n_hidden_q;   int32_t hidden_q[SACX_MAX_HIDDEN];    /* q_net.hidden_sizes            */
  int32_t act_hidden_pi, act_out_pi;                          /* policy_net.*_act              */
  int32_t act_hidden_q,  act_out_q;                           /* q_net.*_act                   */
  int32_t batch_size;                                         /* train.batch_size              */
  int32_t auto_entropy_tuning;                                /* sac.auto_entropy_tuning       */
  int32_t n_agents;                                           /* population size (1 = reference semantics) */
  int32_t ctas_per_agent;                                     /* 0 = auto                      */
  float   log_std_min, log_std_max, action_scale;             /* policy_net.*                  */
  float   reserved_f;
  double  gamma, tau;                                         /* sac.gamma, sac.tau (python doubles in the reference) */
  double  alpha;                                              /* sac.alpha (initial / fixed)   */
  double  actor_lr, critic_lr, alpha_lr;                      /* sac.*_lr                      */
  uint64_t seed;                                              /* device RNG key (train.seed)   */
  int32_t dp_world, dp_rank;                                  /* large-batch data parallel: batch_size is per rank */
  int32_t agent_id_base;                                      /* population sharded over ranks: global id of local agent 0 (keys the device RNG streams) */
  int32_t n_step;                                             /* buffer.n_step: 1..16, 0 = 1 (one-step returns). Every
                                                               * update folds R = sum_{i<m} gamma^i r[j+i] (cut at a terminal, at
                                                               * n and at the newest record) into the gathered row; assumes a ring
                                                               * holds one environment's transitions in time order */
} sacx_config;

typedef struct sacx_ring_s*  sacx_ring_t;    /* replaces sac.replay_buffer.ReplayBuffer        */
typedef struct sacx_agent_s* sacx_agent_t;   /* replaces the update half of sac.agent.SAC      */

/* device-side metrics of the most recent update (reference returns only alpha's dict,
 * sac/agent.py:278; losses are exposed here for parity tests) */
typedef struct sacx_metrics {
  float q1_loss, q2_loss, policy_loss, alpha_loss;
  float alpha, log_alpha, q1_mean, q2_mean;
  float logpi_mean, y_mean;
  int32_t nonfinite;      /* != 0: a policy head produced NaN/Inf                              */
  int32_t reserved;
  int64_t updates;        /* completed updates since create                                    */
} sacx_metrics;

/* one named tensor inside the agent arena (float32 words from the arena base of agent 0;
 * agent k adds k * agent_stride).  dtype: 0 = f32, 1 = f64 (offset is still in f32 words), 2 = i64 */
typedef struct sacx_tensor_desc {
  char    name[40];
  int64_t offset;
  int32_t rows, cols, ld, dtype;
} sacx_tensor_desc;

const char* sacx_last_error(void);
int         sacx_version(void);
int         sacx_device_count(void);
/* struct sizes seen by the library, for bindings to verify their mirror of the structs above */
int         sacx_sizeof_config(void);
int         sacx_sizeof_metrics(void);
int         sacx_sizeof_tensor_desc(void);

/* ---------------------------------------------------------------- replay ring
 * Device-resident ring of packed records [s (O) | s2 (O) | a (A) | r | d | pad] (2O + A + 2 floats rounded up to a multiple
 * of 4) behind a 32-byte header per agent: a sampled transition is one contiguous read.  Push number p
 * lands in slot p % capacity, so logical deque position j (0 = oldest survivor,
 * reference deque(maxlen): sac/replay_buffer.py:19,30) is slot (max(p-N,0)+j) % N.   */
int64_t sacx_ring_bytes(int32_t obs_dim, int32_t act_dim, int64_t capacity, int32_t n_agents);
/* dev_mem NULL -> the library allocates.  replaces ReplayBuffer.__init__ (replay_buffer.py:12-19) */
int sacx_ring_create(int32_t obs_dim, int32_t act_dim, int64_t capacity, int32_t n_agents,
                     void* dev_mem, sacx_ring_t* out);
int sacx_ring_destroy(sacx_ring_t r);
int sacx_ring_set_stream(sacx_ring_t r, void* cuda_stream);
/* replaces ReplayBuffer.push (replay_buffer.py:21-30): appends to a pinned host staging block;
 * the block is flushed to the device ring by one H2D copy + one scatter kernel when full,
 * on sacx_ring_flush, and before any gather / update that reads the ring. */
int sacx_ring_push_host(sacx_ring_t r, int32_t agent, const float* s, const float* a, float reward,
                        const float* s2, float done);
int sacx_ring_push_n_host(sacx_ring_t r, int32_t agent, int64_t n, const float* s, const float* a,
                          const float* reward, const float* s2, const float* done);
/* device producer (SURVEY section 8f-4): rows already on the device */
int sacx_ring_push_n_dev(sacx_ring_t r, int32_t agent, int64_t n, const float* s_dev, const float* a_dev,
                         const float* reward_dev, const float* s2_dev, const float* done_dev);
int sacx_ring_flush(sacx_ring_t r);
/* replaces ReplayBuffer.__len__ (replay_buffer.py:41-42) */
int64_t sacx_ring_len(sacx_ring_t r, int32_t agent);
int64_t sacx_ring_pushes(sacx_ring_t r, int32_t agent);
/* exact resume (no reference counterpart: the reference cannot resume a run, SURVEY 8f-3): after a saved ring image has
 * been copied back into the ring's device block, re-read the per-agent push counters from the ring headers */
int sacx_ring_resync(sacx_ring_t r);
/* replaces ReplayBuffer.sample + SAC.sample_batch (replay_buffer.py:32-39, agent.py:166-193) for a
 * caller-supplied LOGICAL index stream (== random.sample(range(len), B)).  Outputs nullable.
 * SACX_ERR_UNDERFILLED when len < B; SACX_ERR_INVALID when an index is out of range (host variant). */
int sacx_ring_gather(sacx_ring_t r, int32_t agent, const int64_t* logical_idx_dev, int32_t B,
                     float* s_dev, float* a_dev, float* r_dev, float* s2_dev, float* d_dev);
int sacx_ring_gather_host(sacx_ring_t r, int32_t agent, const int64_t* logical_idx_host, int32_t B,
                          float* s_host, float* a_host, float* r_host, float* s2_host, float* d_host);
/* host helper of ReplayBuffer.sample's index stream (replay_buffer.py:39 -> random.sample -> _randbelow_with_getrandbits): applies
 * the stdlib's accept/reject rule, in order, to `n_words` raw 32-bit Mersenne-Twister words fetched in bulk by the binding;
 * appends to out[have..k), returns the new count (-1: bad arguments). No device involved. */
int32_t sacx_index_filter(const uint32_t* words_host, int32_t n_words, uint64_t n, int32_t bits, int64_t* out_host, int32_t have, int32_t k);
/* device index generation used by the throughput mode: B distinct logical positions in [0, n)
 * from a keyed Feistel bijection (exactly without replacement; not the MT19937 stream) */
int sacx_ring_sample_indices(sacx_ring_t r, int32_t agent, uint64_t seed, uint64_t counter, int32_t B,
                             int64_t* logical_idx_dev);

/* ---------------------------------------------------------------- DonkeyVae producer: device-side observation assembly
 * (SURVEY section 8f-4). Replaces the NumPy bookkeeping of DonkeyCarEnv/donkey_gym/envs/vae_env.py:175-210 (postprocessing_step:
 * command-history roll, [latent | history] frame, frame stack with zeroing at episode end) and :253-266 (reset) for a latent
 * that already lives on the device (DonkeyCarEnv/ae/autoencoder.py:64-89 encodes on cuda), and stores the transition
 * (previous stack, action, reward, new stack, done) into the replay ring without a host bounce.
 * Observation width = n_stack * (z_size + n_commands * n_command_history): 3 * (32 + 2 * 20) = 216 in the shipped setup. */
typedef struct sacx_obs_s* sacx_obs_t;
int sacx_obs_create(int32_t z_size, int32_t n_commands, int32_t n_command_history, int32_t n_stack, sacx_obs_t* out);
int sacx_obs_destroy(sacx_obs_t h);
int32_t sacx_obs_dim(sacx_obs_t h);
/* env.reset(): history and stack zeroed, newest frame = [latent | 0]. obs_out_dev (nullable) receives the stacked observation. */
int sacx_obs_reset(sacx_obs_t h, const float* latent_dev, float* obs_out_dev, void* cuda_stream);
/* env.step() post-processing. The action comes from the device (action_dev) or the host (action_host, <= 2 commands); with a
 * ring the transition is pushed on the ring's stream (ring dims must be (sacx_obs_dim, n_commands)), else cuda_stream is used. */
int sacx_obs_step(sacx_obs_t h, const float* latent_dev, const float* action_dev /* nullable */, const float* action_host /* nullable */,
                  float reward, int32_t done, sacx_ring_t ring /* nullable */, int32_t agent, float* obs_out_dev /* nullable */,
                  void* cuda_stream);

/* ---------------------------------------------------------------- agent
 * One arena of float32 words per agent holds parameters (nn.Linear layout [out,in]), target
 * parameters, Adam moments, gradients, temperature scalars (f64), batch and activation scratch.
 * replaces SAC.__init__'s network/optimiser construction (agent.py:34-55); initial weights are
 * written by the caller through the layout (same torch init calls as the reference, F10).     */
int sacx_agent_arena_floats(const sacx_config* cfg, int64_t* floats_per_agent);
int sacx_agent_create(const sacx_config* cfg, float* arena_dev /* nullable */, sacx_agent_t* out);
int sacx_agent_destroy(sacx_agent_t h);
int sacx_agent_set_stream(sacx_agent_t h, void* cuda_stream);
int sacx_agent_attach_ring(sacx_agent_t h, sacx_ring_t r);
float*  sacx_agent_arena(sacx_agent_t h);
int64_t sacx_agent_stride(sacx_agent_t h);          /* float32 words between consecutive agents */
int sacx_agent_layout(sacx_agent_t h, sacx_tensor_desc* out, int32_t capacity, int32_t* n_out);
/* after the caller overwrote online parameters: copy critics to targets (deepcopy, agent.py:88-89),
 * zero Adam state and (re)initialise the temperature scalars from cfg */
int sacx_agent_reset_state(sacx_agent_t h);
/* re-derive alpha (f32/f64) from log_alpha after a checkpoint load (agent.py:549-554) */
int sacx_agent_refresh_alpha(sacx_agent_t h);
int sacx_agent_grid(sacx_agent_t h, int32_t* ctas_per_agent, int32_t* agent_slots, int32_t* smem_bytes);
/* which kernel executes sacx_update: 1 = row-parallel kernel (software groups of 8 CTAs own 16-row blocks, 3xTF32 tensor-core
 * tiles), 0 = tile-parallel persistent kernel (any shape). reason (may be NULL) receives a short text when 0. */
int sacx_agent_path(sacx_agent_t h, char* reason, int32_t capacity);
/* 1 when the MLP GEMMs of this agent run on the tcgen05 tensor-core path (single agent, batch >= SACX_TC_MIN_BATCH,
 * default 4096: 3xTF32 tiles with TMEM accumulators, TMA-staged operands; sacx_tc.cuh), 0 otherwise (reason, may be NULL,
 * says why). tc_launches (may be NULL) receives the number of tensor-core kernel launches so far. */
int sacx_agent_tc(sacx_agent_t h, char* reason, int32_t capacity, int64_t* tc_launches);
/* counter of the rollout-noise stream (sacx_act with eps == NULL); set_to >= 0 overwrites it (exact-resume snapshot) */
int64_t sacx_agent_act_counter(sacx_agent_t h, int64_t set_to);

/* replaces SAC.training_step (agent.py:302-327), n_steps consecutive updates in ONE launch of the
 * persistent fused kernel: gather -> target -> critic Adam x2 -> actor Adam -> alpha -> Polyak.
 *   idx_dev  : [n_steps, n_agents, B] logical indices, or NULL -> device Feistel sampling
 *   eps1_dev : [n_steps, n_agents, B, A] N(0,1) for pi(s'), or NULL -> device Philox
 *   eps2_dev : [n_steps, n_agents, B, A] N(0,1) for pi(s),  or NULL -> device Philox       */
int sacx_update(sacx_agent_t h, const int64_t* idx_dev, const float* eps1_dev, const float* eps2_dev,
                int32_t n_steps);
/* same through HOST buffers (the e2e path): H2D of idx/eps, update, D2H of the metrics, sync */
int sacx_update_host(sacx_agent_t h, const int64_t* idx_host, const float* eps1_host,
                     const float* eps2_host, int32_t n_steps, sacx_metrics* metrics_host);
/* software-pipelined form of sacx_update_host: submits this update (H2D, kernel, metrics D2H) and returns the
 * metrics of the PREVIOUS submission, so the host prepares update t+1 while update t runs.  *have_prev = 0 on the
 * first call.  sacx_update_host_flush waits for the last submission and returns its metrics. */
int sacx_update_host_pipelined(sacx_agent_t h, const int64_t* idx_host, const float* eps1_host, const float* eps2_host,
                               int32_t n_steps, sacx_metrics* prev_metrics_host, int32_t* have_prev);
int sacx_update_host_flush(sacx_agent_t h, sacx_metrics* last_metrics_host);
/* multi-kernel variant of the same update (one launch per phase); used as a cross-check and
 * as the fallback schedule when a cooperative launch is unavailable */
int sacx_update_staged(sacx_agent_t h, const int64_t* idx_dev, const float* eps1_dev,
                       const float* eps2_dev, int32_t n_steps);

/* Per-phase entry points mirroring the reference's methods one to one (agent 0 only). */
/* SAC.sample_batch with the engine's ring: fills the batch buffers, agent.py:166-193 */
int sacx_sample_batch(sacx_agent_t h, const int64_t* idx_dev /* nullable */);
/* load an external batch (device pointers, B = cfg.batch_size rows) into the batch buffers */
int sacx_load_batch(sacx_agent_t h, const float* s_dev, const float* a_dev, const float* r_dev,
                    const float* s2_dev, const float* d_dev);
/* SAC.compute_target_q_values, agent.py:195-211 */
int sacx_target(sacx_agent_t h, const float* eps1_dev /* nullable */, float* y_out_dev /* nullable */);
/* SAC.update_q_networks, agent.py:213-236.  y_dev NULL -> use the y produced by sacx_target */
int sacx_critic_step(sacx_agent_t h, const float* y_dev);
/* SAC.update_policy_network, agent.py:238-260 */
int sacx_actor_step(sacx_agent_t h, const float* eps2_dev /* nullable */, float* logpi_out_dev /* nullable */);
/* SAC.update_entropy_temperature, agent.py:263-280.  logpi_dev NULL -> the actor step's log_pi */
int sacx_alpha_step(sacx_agent_t h, const float* logpi_dev, sacx_metrics* metrics_host /* nullable */);
/* SAC.soft_update_target_networks, agent.py:282-300 */
int sacx_polyak(sacx_agent_t h);
/* gradient-only variants (no optimiser step): fill the gradient block of the arena.  Used by the
 * large-batch data-parallel mode (all-reduce between grads and apply) and by the parity tests. */
int sacx_critic_grads(sacx_agent_t h, const float* y_dev);
int sacx_actor_grads(sacx_agent_t h, const float* eps2_dev, float* logpi_out_dev);
/* Adam on the gradient block: which = 1 critics (+Polyak if polyak != 0), 2 policy, 4 temperature (from the
 * gradient share left in the scalar block by sacx_actor_grads, summed over ranks by the caller) */
int sacx_apply_grads(sacx_agent_t h, int32_t which, int32_t polyak);

/* SAC.select_action (agent.py:149-156) / PolicyNetwork.deterministic_action (models.py:89-92) */
int sacx_act(sacx_agent_t h, int32_t agent, const float* s_dev, int32_t n, const float* eps_dev /* nullable */,
             int32_t deterministic, float* a_dev);
/* vectorised rollouts of a population (SURVEY 8f-1): the action of every agent's policy on its own n_per_agent states in
 * ONE launch. s_dev [n_agents, n_per_agent, obs], eps_dev [n_agents, n_per_agent, act] or NULL (device Philox),
 * a_out_dev [n_agents, n_per_agent, act]; same arithmetic as sacx_act (agent.py:149-156 per agent). */
int sacx_act_population(sacx_agent_t h, const float* s_dev, int32_t n_per_agent, const float* eps_dev /* nullable */,
                        int32_t deterministic, float* a_out_dev);
int sacx_act_host(sacx_agent_t h, int32_t agent, const float* s_host, int32_t n, const float* eps_host /* nullable */,
                  int32_t deterministic, float* a_host);
/* the two critic forwards of SAC._log_q_values (agent.py:493-500) */
int sacx_q_values(sacx_agent_t h, int32_t agent, const float* s_dev, const float* a_dev, int32_t n,
                  float* q1_dev, float* q2_dev);
int sacx_q_values_host(sacx_agent_t h, int32_t agent, const float* s_host, const float* a_host, int32_t n,
                       float* q1_host, float* q2_host);

int sacx_get_metrics(sacx_agent_t h, int32_t agent, sacx_metrics* metrics_host);   /* syncs */
int sacx_sync(sacx_agent_t h);
/* profiling aid: run n_steps fused updates (device RNG) recording, for every CTA and phase, clock64 at barrier
 * arrival and release: out_host[n_steps][n_phases][n_ctas][2] */
int sacx_debug_profile(sacx_agent_t h, int32_t n_steps, uint64_t* out_host, int64_t capacity, int32_t* n_phases, int32_t* n_ctas);
/* number of kernels this handle has launched since create (bench.py's gpu_launches) */
int64_t sacx_launch_count(sacx_agent_t h);

/* ---------------------------------------------------------------- prioritized experience replay (Schaul et al., 2016)
 * A sum/min tree of fan-out 32 over the slots of a single-agent ring; the handle owns its device memory.
 *   priority of a written row  p = (|delta| + eps)^alpha; transitions pushed since the tree last looked get p_max (the
 *                              largest priority ever assigned, initially 1), applied lazily from the ring header's push count
 *   sampling                   stratified proportional: row k draws u = (k + U_k) / B * sum(p) and takes the first slot whose
 *                              inclusive prefix sum exceeds u (duplicates allowed; never an empty slot)
 *   importance weight          w = (p / p_min)^(-beta), p_min over the stored transitions, so w in (0, 1]
 * Every call is one cooperative kernel on the attached agent's stream (else the ring's); no call synchronises except
 * sacx_per_priorities with p_max != NULL and sacx_per_load_priorities. Tree nodes are recomputed from their children in a fixed
 * order (no atomic accumulation): results are bit-reproducible. */
typedef struct sacx_per_s* sacx_per_t;
/* max_batch: the largest B of sacx_per_sample and of an attached agent's batch. SACX_ERR_INVALID for alpha < 0, beta0 outside [0, 1],
 * beta_steps < 0, eps <= 0 or a ring with n_agents > 1. */
int sacx_per_create(sacx_ring_t ring, float alpha, float beta0, int64_t beta_steps, float eps, int32_t max_batch, sacx_per_t* out);
int sacx_per_destroy(sacx_per_t per);
/* B logical indices (idx_dev, the idx_dev format of sacx_update: position in the deque, 0 = oldest) and weights w_dev at exponent
 * beta. u_dev [B] in [0, 1) or NULL -> device Philox keyed by (seed, agent 0, counter, k), a stream of its own. */
int sacx_per_sample(sacx_per_t per, int32_t B, float beta, const float* u_dev /* nullable */, uint64_t seed, uint64_t counter,
                    int64_t* idx_dev, float* w_dev);
/* new priorities (|delta_dev[k]| + eps)^alpha for logical indices of the most recent sample; out-of-range indices are ignored,
 * a slot named twice takes the row with the highest k, slots overwritten by pushes since keep p_max */
int sacx_per_update_priorities(sacx_per_t per, const int64_t* idx_dev, const float* delta_dev, int32_t B);
/* leaves_dev [capacity] (by ring slot, 0 = empty; nullable) and p_max (nullable; synchronises) after applying pending writes */
int sacx_per_priorities(sacx_per_t per, float* leaves_dev, float* p_max);
/* exact resume: replace the leaves (by ring slot) and p_max, rebuild the tree; the ring image must be loaded first */
int sacx_per_load_priorities(sacx_per_t per, const float* leaves_dev, float p_max);
/* With a tree attached (NULL detaches), sacx_update(h, NULL, eps1, eps2, n) runs n x (tree launch: write-back of the previous
 * update's rows from its q1 / q2 / y, delta = (|q1 - y| + |q2 - y|) / 2, new pushes, sample of this batch with beta(t) = min(1,
 * beta0 + (1 - beta0) t / beta_steps) at the agent's update counter t -> fused update with critic loss (1/B) sum w (q - y)^2,
 * n_steps = 1); the last write-back is applied by the next tree launch or by any other launch on the agent. The actor and
 * temperature losses stay unweighted. SACX_ERR_INVALID: n_agents > 1, dp_world > 1, a tree of another ring, max_batch below
 * batch_size. With a tree attached, sacx_update with idx_dev != NULL, sacx_update_host*, and sacx_update_staged are refused; the
 * per-phase entry points (sacx_critic_step, ...) stay unweighted. */
int sacx_agent_attach_per(sacx_agent_t h, sacx_per_t per);

/* ---------------------------------------------------------------- population-based training (Jaderberg et al., 2017)
 * Learner-state copy between agents of a population ("exploit"), optionally followed by new hyper-parameters ("explore").
 * Copied: online parameters, Adam m and v, target critics, and from the scalar block log_alpha, alpha_m, alpha_v, alpha,
 * alpha_f32, the Adam step counters and bias corrections, the learning rates, gamma, tau, 1 - tau. Kept from the destination:
 * the update counter and the RNG keys (its device streams stay its own), metrics, the non-finite flag, the data-parallel
 * shares, and its replay ring. Each call is one kernel on the agent's stream (behind any queued update); nothing synchronises.
 * Validated before any device work (SACX_ERR_INVALID): agent ids and slots in range, no repeated destination, no destination
 * that is also a source of the same call (every copy reads the state from before the call; a source may feed several
 * destinations), record values positive and finite (tau in (0, 1]), no temperature record with auto_entropy_tuning. */
#define SACX_PBT_ALPHA      1    /* log_alpha, alpha, alpha_f32 (fixed temperature only)  */
#define SACX_PBT_ALPHA_LR   2
#define SACX_PBT_ACTOR_LR   4    /* lr[0]                                                 */
#define SACX_PBT_CRITIC_LR  8    /* lr[1] and lr[2]                                       */
#define SACX_PBT_TAU       16    /* tau and one_minus_tau                                 */
#define SACX_PBT_GAMMA     32
/* new hyper-parameters of one destination, as the final field values (the caller applies the config's roundings) */
typedef struct sacx_pbt_record {
  uint32_t set;                  /* SACX_PBT_* bits of the fields written; 0 = no record */
  uint32_t reserved;
  double   log_alpha, alpha;
  double   alpha_lr, actor_lr, critic_lr;
  float    alpha_f32, gamma, tau, one_minus_tau;
} sacx_pbt_record;
int     sacx_sizeof_pbt_record(void);
/* float32 words of one packed learner state (a slot of the pack / unpack buffers; 16-byte multiple) */
int64_t sacx_pbt_state_floats(sacx_agent_t h);
/* agent dst[i] <- agent src[i] (local ids), then records[i] (records nullable) */
int sacx_pbt_copy(sacx_agent_t h, const int32_t* src_host, const int32_t* dst_host, int32_t n_pairs,
                  const sacx_pbt_record* records_host /* nullable */);
/* slot k of buf_dev [n, sacx_pbt_state_floats] <- agent agents[k] */
int sacx_pbt_pack(sacx_agent_t h, const int32_t* agents_host, int32_t n, float* buf_dev);
/* agent dst[i] <- slot slots[i] of buf_dev [n_slots, sacx_pbt_state_floats], then records[i] (records nullable) */
int sacx_pbt_unpack(sacx_agent_t h, const float* buf_dev, int32_t n_slots, const int32_t* slots_host, const int32_t* dst_host,
                    int32_t n, const sacx_pbt_record* records_host /* nullable */);

#ifdef __cplusplus
}
#endif
#endif /* SACX_H_ */
