/*
 * saceo.h - C ABI of the B200-native SAC-EO gradient-update hot path.
 *
 * The reference (noc-lab/sac-expert) is pure Python on TensorFlow-2 eager and has no FFI or
 * plugin layer; its de-facto operator API for this path is a set of Python methods.  Each
 * entry point below names the reference call site(s) it replaces (paths relative to the
 * reference checkout, file:line).  The Python mirror classes in sac_expert_b200/sac_eo/ bind
 * these through ctypes (sac_expert_b200/lib.py); INTEGRATION.md shows the stub a reference
 * maintainer would add.
 *
 * Conventions
 *   - every function returns 0 on success or a negative SACEO_E_* code, never throws;
 *     saceo_last_error() returns a thread-local human-readable message for the last failure.
 *   - all pointers inside saceo_tables are DEVICE pointers owned by the caller (PyTorch only
 *     supplies tensor.data_ptr()); the library owns its context and workspace and never frees
 *     caller memory.
 *   - calls are stream-ordered on the cudaStream_t passed as `stream` (void* to keep this
 *     header free of CUDA includes) and non-blocking, except the *_host variants, which are
 *     documented to synchronise.
 *   - one context per (process, device); contexts are not re-entrant.
 *   - there is NO CPU fallback: create() fails if no sm_100 device is present.
 *
 * Population model: `n_agents` independent agents (seeds x hyper-parameters) share one set of
 * static dimensions; every table is [n_agents, ...] with the strides saceo_query_layout()
 * reports.  n_agents = 1 reproduces the reference's single-agent behaviour.
 *
 * Flat parameter layout per network (Keras get_weights() order, each tensor row-major,
 * sac_eo/common/nn_utils.py:86-138,162-182; actor: sac_eo/actors/continuous_actors.py:201-209):
 *     [ W0 (in x h1) | b0 (h1) | W1 (h1 x h2) | b1 (h2) | W2 (h2 x out) | b2 (out) | logstd (A)* ]
 *     (*) only for a state-independent-std actor.  W is [in, out], y = x @ W + b.
 */
#ifndef SACEO_H_
#define SACEO_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SACEO_ABI_VERSION 1

enum {
  SACEO_OK = 0,
  SACEO_E_INVALID = -1,   /* bad argument / unsupported configuration */
  SACEO_E_CUDA = -2,      /* CUDA runtime error (message in saceo_last_error) */
  SACEO_E_NODEVICE = -3,  /* no sm_100-class GPU: the library refuses to run */
  SACEO_E_UNBOUND = -4,   /* tables not bound yet */
  SACEO_E_NOMEM = -5
};

enum { SACEO_ACT_RELU = 0, SACEO_ACT_TANH = 1, SACEO_ACT_ELU = 2 };

/* GEMM engine for the hidden x hidden per-agent contractions. */
enum {
  SACEO_GEMM_FP32_SIMT = 0,   /* CUDA-core fp32 FMA (exact fp32 products) */
  SACEO_GEMM_TCGEN05_BF16X3 = 1 /* tcgen05.mma kind::f16 on 16-bit hi/lo operand planes (fp16 planes in forward passes,
                                   bf16 planes for gradients), 3 MMAs per product, fp32 accumulation in TMEM */
};

/* Static dimensions - what the reference passes through its kwargs dicts
 * (sac_eo/common/train_parser.py: --actor_layers/--critic_layers/--model_layers,
 *  --*_activations, --actor_per_state_std, --separate_reward_nn, --delta_clip_pred,
 *  --num_models, --sac_batch_size, --expert_buffer_size/--expert_batch_size,
 *  --target_update_int, --actor_std_mult). */
typedef struct saceo_config {
  int32_t abi_version;        /* = SACEO_ABI_VERSION */
  int32_t device;             /* CUDA device ordinal */
  int32_t n_agents;
  int32_t S, A;               /* observation / action dims */
  int32_t actor_hidden[2], critic_hidden[2], model_hidden[2];
  int32_t actor_act[2], critic_act[2], model_act[2];   /* SACEO_ACT_* per hidden layer */
  int32_t per_state_std;      /* actor outputs 2A (mean, logstd) instead of A */
  int32_t separate_reward_nn; /* model outputs S instead of S+1 */
  int32_t num_models;         /* 0 = plain SAC (SAC.py), 1 / 2 = SAC-EO branches (SAC_expert.py:271,299) */
  float   delta_clip_pred;    /* 0 = off (base_world_model.py:80-82) */
  int32_t B;                  /* sac_batch_size */
  int32_t E;                  /* expert rows per update; must be even when num_models == 2 */
  int32_t target_update_int;  /* Polyak gate: num_timesteps % target_update_int == 0 (SAC_expert.py:475) */
  int32_t replay_capacity;    /* rows per agent in the device replay table */
  int32_t fvp_rows;           /* N states for the Fisher-vector product (0 = CG unused) */
  float   std_mult;           /* --actor_std_mult, only used by the GaussianActor._forward (CG) path */
  int32_t gemm_mode;          /* SACEO_GEMM_* */
  int32_t use_graph;          /* capture one update into a CUDA graph and replay it */
  int32_t reserved[8];        /* tuning switches, 0 = default: [0] tcgen05 tile variant (0: 128x256 tile, 1: 128x128 2 CTAs/SM,
                                 2: force the register-staged kernel); [1] != 0 disables the fused 3-layer forward kernel;
                                 [2] != 0 disables the fused backward-chain kernel;
                                 [5] != 0 disables the warp-specialised TMA-fed fused kernels and their weight planes
                                 (round-1 fused kernels are used instead); [6] != 0 keeps the whole update on one stream (no
                                 concurrent actor-phase branch); [3], [4], [7] must be 0 (SACEO_E_INVALID otherwise) */
} saceo_config;

/* Strides/offsets (in 4-byte words unless stated) derived from a config. */
typedef struct saceo_layout {
  int64_t na, nc, nm;                 /* parameter counts actor / one critic / one model */
  int64_t na_stride, nc_stride, nm_stride;   /* padded per-agent (per-net) strides */
  int32_t Ao, model_out;
  /* device replay row (AoS, 16-byte aligned): [ s(S) | a(A) | sp(S) | r | pad | d (f64, 2 words) | pad ] */
  int32_t row_words, off_s, off_a, off_sp, off_r, off_d;
  /* per-agent normaliser record */
  int32_t norm_stride, off_s_mean, off_s_std, off_a_mean, off_a_std, off_ret_std,
          off_m_s_mean, off_m_s_std, off_m_a_mean, off_m_a_std, off_m_d_mean, off_m_d_std,
          off_act_limit;
  int32_t hyper_stride;               /* = 8: gamma,tau,lr_q,lr_pi,lr_alpha,eps,target_entropy,damp */
  int32_t n_losses;                   /* = 8: L_q1,L_q2,L_pi,mse,p_loss,alpha_loss,alpha,eps */
  int64_t workspace_bytes;            /* what create() will cudaMalloc */
} saceo_layout;

/* Device tables, all caller-owned.  Shapes use the strides of saceo_layout.
 * They replace the reference's tf.Variable / optimizer-slot / NumPy state:
 *   actor*       SquashedGaussianActor._nn (+logstd)        continuous_actors.py:46-57
 *   q*, qt       QCritic._nn x2 live, x2 targets            critics/init_critic.py:27-35
 *   model        MSEModel/GaussianModel._nn x2 (frozen)     models/init_world_models.py:5-29
 *   alpha*       self.alpha (raw, log-initialised)          SAC_expert.py:106
 *   *_m,*_v,adam_t   tf.keras.optimizers.Adam slots x4      SAC_expert.py:108-115
 *   norm         RunningNormalizers stats                   common/normalizer.py:126-190
 *   replay*      TrajectoryBuffer arrays                    common/buffers.py:28-39
 *   expert_*     expert_reg[0], expert_reg[2]               SAC_expert.py:423 */
typedef struct saceo_tables {
  float *actor, *actor_m, *actor_v;          /* [n_agents, na_stride] */
  float *q, *q_m, *q_v;                      /* [n_agents, 2, nc_stride] */
  float *qt;                                 /* [n_agents, 2, nc_stride] */
  const float *model;                        /* [n_agents, 2, nm_stride] (unused if num_models == 0) */
  float *alpha, *alpha_m, *alpha_v;          /* [n_agents] */
  int32_t *adam_t;                           /* [n_agents, 4]: q1, q2, actor, alpha step counts */
  const float *norm;                         /* [n_agents, norm_stride] */
  const float *hyper;                        /* [n_agents, hyper_stride] */
  float *replay;                             /* [n_agents, replay_capacity, row_words]; written by saceo_replay_append */
  int32_t *replay_size;                      /* [n_agents] rows currently valid */
  int32_t *replay_start;                     /* [n_agents] physical row of logical index 0 (ring), may be NULL (then
                                                saceo_replay_append is unavailable) */
  float *expert_s, *expert_sp;               /* [n_agents, E, S]; saceo_update_host* overwrite them with expert_host */
  const float *fvp_states;                   /* [n_agents, fvp_rows, S] or NULL */
} saceo_tables;

typedef struct saceo_ctx saceo_ctx;

/* Layout helper (pure host arithmetic; callable without a GPU). */
int saceo_query_layout(const saceo_config *cfg, saceo_layout *out);

/* Lifetime.  create() allocates the workspace on cfg->device and fails with
 * SACEO_E_NODEVICE when there is no compute-capability-10.x GPU. */
int saceo_create(const saceo_config *cfg, saceo_ctx **out);
int saceo_destroy(saceo_ctx *ctx);
int saceo_bind(saceo_ctx *ctx, const saceo_tables *tables);

/* The tcgen05 engine keeps fp16 hi/lo operand images ("weight planes") of the actor / q / qt tables in its workspace;
 * every kernel of the library that updates a parameter (Adam, Polyak, the trust-region step) keeps them current.  A
 * caller that writes into those tables itself (set_weights, checkpoint restore, torch ops on the tensors) must call
 * this afterwards; the images are rebuilt before the next use.  saceo_bind() implies it.  Replaces nothing in the
 * reference (tf.Variable.assign has no such side state); it is the cost of never converting a weight inside a pass. */
int saceo_weights_changed(saceo_ctx *ctx);

/* TrajectoryBuffer.get_offmodel_info / get_model_info (common/buffers.py:107-144): for the SAME
 * int64 indices (device, [n_agents, B], logical row numbers) writes exact copies of the rows:
 * out_s [n,B,S] f32, out_a [n,B,A] f32, out_sp [n,B,S] f32, out_r [n,B] f32, out_d [n,B] f64.
 * Any out_* may be NULL.  Bit-exact. */
int saceo_gather(saceo_ctx *ctx, const int64_t *idx, float *out_s, float *out_a, float *out_sp,
                 float *out_r, double *out_d, void *stream);

/* TrajectoryBuffer.add (common/buffers.py:41-71) for EVERY agent in one call - the per-step triple add of the
 * environment loop (algs/SAC_expert.py:793-801) without its O(N) np.concatenate: rows (device, 16-byte aligned,
 * [n_agents, k, row_words] in the AoS row layout of saceo_layout) are appended behind each agent's newest row; a full
 * ring overwrites its oldest rows, i.e. keeps the last replay_capacity rows like the reference's tail truncation
 * (:60-66).  replay_size / replay_start are updated on the device (stream-ordered, no host sync). */
int saceo_replay_append(saceo_ctx *ctx, const float *rows, int32_t k, void *stream);

/* Inject the random draws of the next update(s) (parity mode), device pointers, any may be NULL:
 * idx [n,B] int64 (np.random.randint, buffers.py:135); noise [n, 3B+E, A] f32 in reference draw
 * order u1 | u2 | u3,u4 (expert rows, permuted order) | u5 (np.random.normal,
 * continuous_actors.py:297,350); expert_perm [n,E] int32 = concatenated array_split sections of
 * the shuffled arange (SAC_expert.py:301-303). */
int saceo_set_draws(saceo_ctx *ctx, const int64_t *idx, const float *noise,
                    const int32_t *expert_perm, void *stream);

/* SAC_exp._update / SAC._update (SAC_expert.py:463-477, SAC.py:236-250) for every agent,
 * n_steps times.  use_device_rng = 1: idx/noise/permutation are drawn in-kernel (Philox4x32-10
 * keyed by seed, agent, step) before each step; 2: only noise and permutation are drawn in-kernel, the
 * minibatch indices already in the context (set_draws / update_host) are kept; 0: the draws last injected
 * with saceo_set_draws() are consumed (n_steps should then be 1).  num_timesteps gates the Polyak
 * update of step i on (num_timesteps + i) % target_update_int == 0.  losses_out (device,
 * [n_agents, n_losses], may be NULL) receives the values of the LAST step. */
int saceo_update(saceo_ctx *ctx, int32_t n_steps, int64_t num_timesteps, int32_t use_device_rng,
                 uint64_t seed, float *losses_out, void *stream);

/* Same, through HOST buffers (the call the Python `_update` makes per step): copies idx_host
 * [n,B] int64 (may be NULL => device RNG) and expert_host [2, n, E, S] f32 (all sE rows, then all s'E rows; may be
 * NULL => keep the bound tables; otherwise the rows are copied INTO the bound expert_s / expert_sp tables, exactly as if
 * the caller had refreshed them before the update) host->device, runs one update, copies losses [n, n_losses] back into
 * losses_host and synchronises the stream. */
int saceo_update_host(saceo_ctx *ctx, int64_t num_timesteps, uint64_t seed, const int64_t *idx_host,
                      const float *expert_host, float *losses_host, void *stream);

/* Same without the final synchronisation: the copies and the update are only enqueued on `stream`.  The host
 * buffers (pinned) must stay untouched until the stream reaches this point (record an event after the call);
 * with two sets of host buffers the caller prepares step t+1 (np.random.randint, env stepping) while the device
 * runs step t.  The device-side staging is single-buffered and stream-ordered, so calls may be queued back to back. */
int saceo_update_host_async(saceo_ctx *ctx, int64_t num_timesteps, uint64_t seed, const int64_t *idx_host,
                      const float *expert_host, float *losses_host, void *stream);

/* Behaviour cloning from expert observations - BC._update_actor (sac_eo/algs/BC.py:309-363): the expert-observation
 * term ALONE (counterfactual actions through the frozen models, MSE to the expert next states, i.e. the epsilon = 1
 * slice of the SAC-EO actor step) and one Adam step of self.actor_optimizer (BC.py:113).  Critics, temperature,
 * targets and their step counters are untouched.  Draws as in saceo_update: use_device_rng != 0 draws the expert
 * noise / shuffle in-kernel, 0 consumes the noise block [u1|u2|uE|u5] and perm of saceo_set_draws (only uE is used).
 * losses_out (device, [n_agents, n_losses], nullable): slots 3 and 4 hold BC_MSE_loss. */
int saceo_bc_update(saceo_ctx *ctx, int32_t n_steps, int32_t use_device_rng, uint64_t seed, float *losses_out,
                    void *stream);

/* Measurement aid: ONE update launched kernel by kernel (no CUDA graph) with a CUDA event after every launch.
 * names_out [max_n][32] and us_out [max_n] receive the kernel name and the device time between consecutive events
 * (so a launch gap is charged to the kernel that follows it); *n_out = launches recorded.  Synchronises the stream.
 * Same arguments as saceo_update otherwise; the step is a real update (state advances). */
int saceo_profile_step(saceo_ctx *ctx, int64_t num_timesteps, int32_t use_device_rng, uint64_t seed,
                       char *names_out, float *us_out, int32_t max_n, int32_t *n_out, void *stream);

/* Phase-split form of one update for the optional single-agent data-parallel mode (gradients are
 * all-reduced by the caller between *_grads and *_apply; torch.distributed/NCCL does the
 * collective).  phase: 0 = TD target + critic grads, 1 = critic Adam(+Polyak), 2 = actor grads,
 * 3 = actor Adam, 4 = alpha grad, 5 = alpha Adam + clamp.  grad buffers: saceo_debug_ptr(). */
int saceo_update_phase(saceo_ctx *ctx, int32_t phase, int64_t num_timesteps, void *stream);

/* actor.sample(s, deterministic) for the population (SAC_expert.py:779; samplers.py:31):
 * obs [n_agents, rows, S] -> act_out [n_agents, rows, A] (device).  noise [n_agents, rows, A] or
 * NULL (=> deterministic mean action).  Also returns neglogp [n_agents, rows] if non-NULL
 * (= actor.evaluate, continuous_actors.py:327-379). */
int saceo_actor_forward(saceo_ctx *ctx, const float *obs, int32_t rows, const float *noise,
                        float *act_out, float *neglogp_out, void *stream);

/* critic._forward / critic.value (critics.py:84-103): which = 0 live, 1 target.
 * q_out [n_agents, 2, rows] = normalised-space output; scale_ret != 0 multiplies by max(ret_std,1e-8). */
int saceo_critic_forward(saceo_ctx *ctx, int32_t which, const float *obs, const float *act,
                         int32_t rows, int32_t scale_ret, float *q_out, void *stream);

/* model.sample(s, a, deterministic=True) (continuous_models.py:244-254): sp_out [n_agents, 2, rows, S]. */
int saceo_model_eval(saceo_ctx *ctx, const float *obs, const float *act, int32_t rows,
                     float *sp_out, void *stream);

/* ---- dynamics-model fitting (SURVEY.md 8f rank 1) -------------------------------------------------
 * MBRLOnPolicyAlg._apply_model_grads (sac_eo/algs/mbrl_onpolicy_alg.py:301-319) as driven by
 * SAC_exp._update_models (sac_eo/algs/SAC_expert.py:480-556), loss MSEModel.get_loss
 * (sac_eo/models/continuous_models.py:280-302) on BaseWorldModel._forward(clip=False)
 * (sac_eo/models/base_world_model.py:65-87).  Replaces self.model_optimizer (one tf.keras Adam over the
 * tensors of ALL models, mbrl_onpolicy_alg.py:48-49) and tf.clip_by_global_norm (:315-317).
 * GaussianModel.get_loss (continuous_models.py:101-131) is used instead when the logstd tables are given.
 * With separate_reward_nn the reward prediction comes from the reward network bound in saceo_fit_tables (the model
 * network then predicts the S delta columns only).  fit_hyper per agent (8 floats):
 *   [0] model_lr  [1] reward_loss_coef  [2] delta_clip_loss (0 = off)  [3] reward_clip_loss (0 = off)
 *   [4] model_max_grad_norm (0 = None)  [5] r_rms mean  [6] r_rms std  [7] scale_model_loss (0/1, Gaussian only) */
#define SACEO_FIT_HYPER 8
typedef struct saceo_fit_tables {
  float *model;                /* [n_agents, 2, nm_stride] trainable; normally the table bound as saceo_tables.model */
  float *model_m, *model_v;    /* Adam slots, same shape */
  int32_t *model_t;            /* [n_agents] step count of the joint optimiser */
  const float *fit_hyper;      /* [n_agents, SACEO_FIT_HYPER] */
  /* GaussianModel only (all three NULL => MSEModel loss): the trainable logstd variable [n_agents, 2, S]
   * (continuous_models.py:24-27, initial value log(std_mult)) and its Adam slots; part of the same joint optimiser */
  float *model_logstd, *model_logstd_m, *model_logstd_v;
  /* separate_reward_nn only (base_world_model.py:34-38, continuous_models.py:216-219): the reward network of every model,
   * input S+A, two hidden layers reward_hidden with activations reward_act (SACEO_ACT_*), one output, flat Keras layout
   * [W0|b0|W1|b1|W2|b2], [n_agents, 2, reward_stride] (reward_stride % 32 == 0), and its Adam slots.  Its tensors join
   * the same joint optimiser and the same global-norm clip (model.trainable = model_trainable + reward_trainable). */
  float *reward, *reward_m, *reward_v;
  int32_t reward_hidden[2], reward_act[2];
  int64_t reward_stride;
} saceo_fit_tables;

/* Binds the fit tables and allocates the fitting workspace for minibatches of model_batch rows
 * (--model_batch_size, 200).  use_grad_clip != 0 enables the global-norm pass (agents whose
 * model_max_grad_norm is 0 are still left unclipped).  Requires saceo_bind (replay + normalisers). */
int saceo_fit_bind(saceo_ctx *ctx, const saceo_fit_tables *t, int32_t model_batch, int32_t use_grad_clip);

/* n_steps joint gradient steps.  idx: device int64 [n_steps, n_agents, num_models, model_batch] logical
 * replay rows - the columns of the reference's per-model shuffled index matrix (SAC_expert.py:524-545).
 * losses_out (device, nullable): [n_steps, n_agents, num_models] minibatch loss of each model before the step. */
int saceo_model_fit(saceo_ctx *ctx, int32_t n_steps, const int64_t *idx, float *losses_out, void *stream);

/* TRPO._make_F closure (model_free/trpo.py:200-227): Fx = d/dtheta((d/dtheta mean KL) . x) + damp x
 * on the bound fvp_states, x and Fx [n_agents, na_stride] device. */
int saceo_fvp(saceo_ctx *ctx, const float *x, float damp, float *Fx, void *stream);

/* cg(F, b, cg_iters, residual_tol) (common/update_utils.py:4-24) followed by vFv = x.F(x)
 * (trpo.py:185): b, x_out [n_agents, na_stride], vFv_out [n_agents] device. */
int saceo_cg_solve(saceo_ctx *ctx, const float *b, int32_t iters, float tol, float damp,
                   float *x_out, float *vFv_out, void *stream);

/* TRPO.update surrogate gradient (algs/model_free/trpo.py:36-63) on the rows bound as fvp_states (all fvp_rows of
 * them), GaussianActor parameterisation (actors/continuous_actors.py:74-100,137-148):
 *   loss = mean(-exp(nlp_old - neglogp(s,a)) adv) - alpha (mean entropy(s) - ent_targ)
 * act [n,N,A], adv [n,N] (already centred / scaled by the caller, trpo.py:41-48), nlp_old [n,N] or NULL (= current
 * neglogp, ratio 1), alpha [n] or NULL (0); grad_out [n, na_stride] = d loss / d theta ("neg_pg", flat layout);
 * stats_out [n,8] or NULL = {mean(ratio adv), 0, 0.5 mean|ratio-1|, mean entropy, 0...}.  The temperature gradient
 * is -(stats[3] - ent_targ) (host scalar).  All device pointers. */
int saceo_trpo_grad(saceo_ctx *ctx, const float *act, const float *adv, const float *nlp_old, const float *alpha,
                    float *grad_out, float *stats_out, void *stream);

/* PPO._apply_actor_grad gradient (algs/model_free/ppo.py:132-147, expert_reg = None) on the rows bound as fvp_states:
 *   loss = mean(max(-ratio adv, -clip(ratio, 1-eps_clip, 1+eps_clip) adv)) - alpha (mean entropy - ent_targ)
 * followed by tf.clip_by_global_norm(neg_pg, max_grad_norm) (:226-231; max_grad_norm <= 0: no clipping).
 * Arguments as saceo_trpo_grad (nlp_old required); stats_out [n,8] additionally carries [4] = global norm before and
 * [5] = after clipping. */
int saceo_ppo_grad(saceo_ctx *ctx, const float *act, const float *adv, const float *nlp_old, const float *alpha,
                   float eps_clip, float max_grad_norm, float *grad_out, float *stats_out, void *stream);

/* Expert-observation gradient of the on-policy classes: the second tape of TRPO.update's two-model branch
 * (algs/model_free/trpo.py:113-149) and the MSE half of PPO._apply_actor_grad's expert branch (ppo.py:176-213, models[0]):
 * counterfactual actions a = GaussianActor.sample(sE) = mean + exp(logstd) u (actors/continuous_actors.py:103-123, the
 * _forward parameterisation with cfg.std_mult; clip_actions != 0: actor.tf_clip to +-act_limit, :128-129), next-state
 * prediction through the frozen model(s) (models/continuous_models.py:244-254), MSE = mean_i 0.5 sum_j (s'E - pred)^2
 * over the rows of one model (n_models = 2: the two halves of the shuffled expert rows through models 0 and 1, the two
 * means added; n_models = 1: all E rows through model 0).  Expert rows = tables.expert_s / expert_sp; the shuffle
 * (expert_perm) and the noise (rows [2B, 2B+E) of the noise block = the u3 | u4 slots) are the draws last injected with
 * saceo_set_draws.  grad_out [n, na_stride] (device, 16-byte aligned) = d MSE / d(actor trainable), UNWEIGHTED;
 * stats_out [n, 8] (may be NULL): [0] = MSE. */
int saceo_onpolicy_expert_grad(saceo_ctx *ctx, int32_t n_models, int32_t clip_actions, float *grad_out, float *stats_out,
                               void *stream);

/* grad_final = (1 - eps) neg_pg + eps mse_grad (trpo.py:150-158; ppo.py:213 after the tape) per agent, eps [n] (device);
 * out [n, na_stride] may alias neg_pg.  stats_out [n, 8] (may be NULL): [6] = norm_pg, [7] = norm_MSE as the reference
 * logs them (sums of per-tensor L2 norms, trpo.py:160-163), [4] / [5] = global norm of the result before / after
 * tf.clip_by_global_norm(max_grad_norm) (ppo.py:226-231; max_grad_norm <= 0: no clipping). */
int saceo_grad_blend(saceo_ctx *ctx, const float *neg_pg, const float *mse_grad, const float *eps, float max_grad_norm,
                     float *out, float *stats_out, void *stream);

/* actor_optimizer.apply_gradients(zip(neg_pg, actor.trainable)) (ppo.py:234): one Keras-Adam step of the ACTOR
 * optimiser (tables.actor / actor_m / actor_v, adam_t[.,2], learning rate hyper[3]) with grad [n, na_stride]
 * (device, 16-byte aligned).  No other optimiser advances. */
int saceo_actor_adam(saceo_ctx *ctx, const float *grad, void *stream);

/* Quantities of the back-tracking line search TRPO._backtrack (trpo.py:229-317) at the CURRENT actor parameters:
 * nlp_out [n,N] = actor.neglogp(s,a) (:137-143); kl_info_out [n,N,A,2] = actor.get_kl_info(s) (:186-192);
 * stats_out [n,8] = {surr = mean(ratio adv), mean actor.kl(s, kl_ref) (forward, :165-184; 0 if kl_ref NULL),
 * tv = 0.5 mean|ratio-1|, mean actor.entropy(s) (:145-148), 0...}; ratio = exp(nlp_old - neglogp), 1 if nlp_old NULL.
 * Any of act, adv, nlp_old, kl_ref and the outputs may be NULL. */
int saceo_trpo_eval(saceo_ctx *ctx, const float *act, const float *adv, const float *nlp_old, const float *kl_ref,
                    float *nlp_out, float *kl_info_out, float *stats_out, void *stream);

/* actor.set_weights(theta_ref); actor.set_weights(scale * dir, from_flat=True, increment=True)
 * (continuous_actors.py:211-233, incl. the log(1e-3) floor of the state-independent logstd variable):
 * tables.actor[agent] = theta_ref[agent] + scale[agent] * dir[agent]; theta_ref, dir [n, na_stride], scale [n]. */
int saceo_actor_step(saceo_ctx *ctx, const float *theta_ref, const float *dir, const float *scale, void *stream);

/* ---- policy acting for any depth (expert policies) ------------------------------------------------
 * An expert is only ever rolled out, never trained: SAC_exp._collect_expert_data (sac_eo/algs/SAC_expert.py:156-209)
 * calls expert.sample(s, deterministic=True) through trajectory_sampler (common/samplers.py:31).  The reference loads
 * that expert with --expert_file (train.py:65-83); it is a GaussianActor (actors/continuous_actors.py:9-234) or a
 * SquashedGaussianActor (:237-415) of any depth.  These entry points act for a set of n_policies independent policies
 * in one launch, in exact fp32 on CUDA cores, without a context and without the two-hidden-layer training engine. */
#define SACEO_POLICY_MAX_HIDDEN 8
typedef struct saceo_policy_config {
  int32_t abi_version, device, n_policies, S, A;
  int32_t n_hidden, hidden[SACEO_POLICY_MAX_HIDDEN], act[SACEO_POLICY_MAX_HIDDEN];   /* widths 1..1024, SACEO_ACT_* */
  int32_t squash, per_state_std;   /* head; per_state_std: output 2A, else A outputs + logstd variable [A] */
  float   std_mult;                /* GaussianActor only */
} saceo_policy_config;

/* Host arithmetic, no GPU: parameter count, per-policy stride (padded to 32 words), normaliser record stride.  Any
 * output pointer may be NULL. */
int saceo_policy_layout(const saceo_policy_config *cfg, int64_t *n_params, int64_t *param_stride, int32_t *norm_stride);

/* expert.sample(s, deterministic) for every policy of the set: GaussianActor._forward + .sample (squash = 0,
 * continuous_actors.py:74-123) or SquashedGaussianActor.sample (squash = 1, :270-306), observations normalised with the
 * policy's own statistics (normalizer.py:26-41).
 * params [P, param_stride] flat Keras order [W0|b0|...|Wn|bn|(logstd)]; norm [P, norm_stride] = s_mean | s_std | act_limit;
 * obs [P, rows, S]; noise [P, rows, A] or NULL (deterministic); act_out [P, rows, A].  All device pointers on cfg->device.
 * Stream-ordered, no context; one kernel launch.  Policy i's actions are bit-identical whatever the other policies are. */
int saceo_policy_act(const saceo_policy_config *cfg, const float *params, const float *norm, const float *obs,
                     int32_t rows, const float *noise, float *act_out, void *stream);

/* Test / inspection surface: device pointer of a named workspace buffer (e.g. "g_q", "g_actor",
 * "y", "losses", "idx", "noise") and its size in bytes; NULL if unknown. */
void *saceo_debug_ptr(saceo_ctx *ctx, const char *name, int64_t *bytes_out);

/* Number of kernels launched by this context so far (bench.py's gpu_launches). */
int64_t saceo_launch_count(const saceo_ctx *ctx);

/* Standalone batched GEMM self-test surface used by tests/: C[z] = op(A[z]) . op(B[z]) with the
 * engine selected by gemm_mode; all device pointers, row-major. */
int saceo_test_gemm(int32_t gemm_mode, int32_t batch, int32_t M, int32_t N, int32_t K,
                    int32_t transA, int32_t transB, const float *A, const float *Bm, float *C,
                    void *stream);

const char *saceo_last_error(void);
int saceo_abi_version(void);

#ifdef __cplusplus
}
#endif
#endif /* SACEO_H_ */
