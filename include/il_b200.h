/*
 * il_b200.h — C ABI of the B200-native (sm_100a) hot path of Kaixhin/imitation-learning.
 *
 * The reference has no FFI: its hot path sits behind Python signatures (SURVEY.md §8b). Each entry point
 * below is what a binding for that path would call; the comment on each cites the reference interface it
 * replaces (paths relative to the reference tree). INTEGRATION.md shows the ctypes stubs.
 *
 * Conventions
 *  - Plain pointers and sizes only; every pointer is a DEVICE pointer unless stated otherwise. fp32 data,
 *    row-major. All tensors carry a leading REPLICA axis R: replica r is one reference-equivalent run
 *    (own actor / critic / target / log_alpha / optimiser state / discriminator / replay ring / env);
 *    R = 1 is exactly the reference's shapes.
 *  - No allocation, no host synchronisation, CUDA-graph capturable: callers pass workspaces (sizes from the
 *    *_workspace_bytes queries) and a cudaStream_t (as void*).
 *  - Return value: 0 on success, non-zero on error (message via il_last_error()). There is NO CPU fallback.
 *  - All randomness is an explicit input (noise / index tensors). il_fill_normal / il_fill_uniform /
 *    il_replay_sample_indices generate them on the device (Philox4x32-10) when the caller does not inject.
 */
#ifndef IL_B200_H
#define IL_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define IL_MAX_LAYERS 6

enum { IL_ACT_RELU = 0, IL_ACT_TANH = 1, IL_ACT_SIGMOID = 2 };          /* models.py:17 ACTIVATION_FUNCTIONS */
enum { IL_REWARD_AIRL = 0, IL_REWARD_GAIL = 1, IL_REWARD_FAIRL = 2 };    /* models.py:179-180 */
enum { IL_LOSS_BCE = 0, IL_LOSS_MIXUP = 1, IL_LOSS_PUGAIL = 2 };         /* training.py:94-114 */
enum { IL_GEMM_FP32 = 0, IL_GEMM_TF32X3 = 1, IL_GEMM_TF32 = 2 };         /* arithmetic of the dense HxH layers */

typedef struct il_handle il_handle;

/* G independent MLPs (`_create_fcnn`, models.py:48-69) in one flat buffer: per net, per layer l:
 * W_l [dims[l+1], dims[l]] row-major then b_l [dims[l+1]]; every tensor starts on a 4-float boundary
 * (il_mlp_param_offsets). Net g starts at params + g * stride. A TwinCritic is two consecutive nets. */
typedef struct il_mlp {
  float*  params;
  int64_t stride;
  int32_t n_layers;                 /* Linear layers = reference depth + 1 */
  int32_t activation;               /* IL_ACT_* */
  int32_t dims[IL_MAX_LAYERS + 1];
  int32_t _pad;
} il_mlp;

/* torch.optim.Adam / AdamW (decoupled decay) state over one flat parameter buffer (train.py:66,84).
 * Per-replica hyperparameters: lr_r / weight_decay_r (nullable [R] device arrays; NULL = the scalar for every replica) give replica r
 * its own value, with the scalar path's arithmetic in double, so a replica equals a scalar run with its values bit for bit. Replica r
 * owns floats [r * replica_floats, (r + 1) * replica_floats) of the buffer: il_adam_step / il_adam_step_polyak need replica_floats
 * (a multiple of 4) when an array is set; the fused updates take it from their own layout. One call with per-replica values covers at
 * most 4096 replicas (the AdamW kernels keep a 16-byte entry per replica in shared memory); more is an error. */
typedef struct il_adam {
  float*   m;                       /* exp_avg, same shape as the parameter buffer */
  float*   v;                       /* exp_avg_sq */
  int64_t* step;                    /* device scalar, incremented by every update */
  double lr, beta1, beta2, eps, weight_decay;  /* Python floats in the reference; kept in double like torch does */
  const double* lr_r;               /* [R] or NULL */
  const double* weight_decay_r;     /* [R] or NULL */
  int64_t replica_floats;           /* floats per replica (2 x stride for the twin critic) */
} il_adam;

/* Packed transitions [R, B, row]: row = [state S | action A | reward | next_state S | terminal | timeout |
 * weight | step | pad to 4 floats]  (the 8 fields of memory.py:17 as one 128 B row for hopper). */
typedef struct il_batch {
  float*  rows;
  int64_t replica_stride;           /* floats between replicas (0 = one batch shared by all replicas) */
  int32_t B, S, A, row;
} il_batch;

/* Replay ring per replica (memory.py:13-23): rows [R, size, row]; idx/full/num_trajectories per replica. */
typedef struct il_replay {
  float*   rows;
  int64_t  replica_stride;          /* 0 = one memory shared by all replicas (expert buffer) */
  int32_t* idx;                     /* [R] next write position (memory.py:15) */
  int32_t* full;                    /* [R] ring wrapped (memory.py:43) */
  int32_t* num_trajectories;        /* [R] (memory.py:44) */
  int32_t  size, S, A, row;
  int32_t  absorbing;               /* memory.py:16 */
  int32_t  shared;                  /* 1: idx/full/num_trajectories have one entry used by all replicas */
} il_replay;

/* ---- library ----------------------------------------------------------------------------------------- */
int         il_create(int device, il_handle** out);
int         il_destroy(il_handle* h);
const char* il_last_error(void);
int         il_version(void);
int         il_set_gemm_mode(il_handle* h, int mode);              /* IL_GEMM_* for the dense hidden layers */
int64_t     il_launch_count(il_handle* h);                         /* kernels launched by this library so far */
/* Kernel-selection toggles for A/B measurements and tests (defaults from the IL_* environment variables at il_create):
 * "tc_fuse_l1" (first MLP layer inside the tcgen05 producers), "gail_tiled", "tc_pairs", "thin_hoist". */
int         il_set_option(il_handle* h, const char* name, int value);
int         il_struct_sizes(int32_t* out15);                       /* sizeof il_mlp, il_adam, il_batch, il_replay, il_sac_args, il_gail, il_gail_update_args, il_pwil, il_env, il_bc_args, il_eval_args, il_gailx, il_gailx_update_args, il_red, il_red_update_args */
int         il_mlp_param_offsets(const int32_t* dims, int n_layers, int64_t* w_off, int64_t* b_off, int64_t* total);
int         il_row_layout(int S, int A, int32_t* offsets8, int32_t* row_len); /* state, action, reward, next_state, terminal, timeout, weight, step */

/* Measurement aid for bench.py: between begin/end (eager launches, no graph capture) every dense hidden-layer GEMM launch
 * is bracketed by CUDA events on its own stream; end() synchronises and returns the summed device time, the summed
 * algorithmic FLOPs (2 M N K G per launch) and the number of launches; il_profile_bytes then returns the summed
 * algorithmic HBM bytes of those launches (each distinct operand element read once, each output element written once). */
int il_profile_begin(il_handle* h);
int il_profile_end(il_handle* h, double* total_ms, double* total_flops, int64_t* launches);
int il_profile_bytes(il_handle* h, double* total_bytes);

/* Test / diagnostics entry: one grouped GEMM C[g] = A[g] B[g] with the fused epilogues (bias, activation act >= 0,
 * activation-derivative mask, bias-gradient column sums), dispatched exactly like the MLP programs dispatch it
 * (fp32 FFMA engine, or the tcgen05 engine for eligible dense shapes when the gemm mode is tf32x3 / tf32).
 * a_kmajor: A stored [M, K] (else [K, M]); b_kmajor: B stored [N, K] (else [K, N]). */
int il_debug_gemm(il_handle* h, int M, int N, int K, int G, const float* A, int64_t a_gs, int lda, int a_kmajor,
                  const float* B, int64_t b_gs, int ldb, int b_kmajor, float* C, int64_t c_gs, int ldc,
                  const float* bias, int64_t bias_gs, int act, const float* mask, int64_t mask_gs, int ldmask, int mask_act,
                  float* colsum, int64_t colsum_gs, void* stream);

/* ---- random inputs (replace torch / numpy global RNG draws when noise is not injected) ---------------- */
int il_fill_normal(il_handle* h, float* out, int64_t n, uint64_t seed, uint64_t stream_id, const uint64_t* counter, void* stream);
int il_fill_uniform(il_handle* h, float* out, int64_t n, uint64_t seed, uint64_t stream_id, const uint64_t* counter, void* stream);
int il_counter_add(il_handle* h, uint64_t* counter, uint64_t inc, void* stream);

/* ---- replica state copy (population-based training, sweep.py) ------------------------------------------ */
/* For every buffer b and every replica r with src_of[r] != r: copy bytes[b] bytes from base[b] + src_of[r] * stride_bytes[b] to
 * base[b] + r * stride_bytes[b]. src_of is a device [R] int32 map; it may change between replays of a captured call (identity entries
 * cost one read of the map). Host arrays of nbufs <= IL_REPLICA_COPY_MAX_BUFS entries; every base, stride and length 4-byte aligned,
 * bytes <= stride (16-byte aligned buffers take the vector path).
 * Precondition (the caller guarantees it; documented, not checked on the device): every source is its own source, i.e.
 * src_of[src_of[r]] == src_of[r], so no replica is both read and written. */
#define IL_REPLICA_COPY_MAX_BUFS 64
int il_replica_copy(il_handle* h, int nbufs, void* const* base, const int64_t* stride_bytes, const int64_t* bytes, int R, const int32_t* src_of,
                    void* stream);

/* ---- SoftActor (models.py:84-102) --------------------------------------------------------------------- */
/* forward + tanh-Gaussian head for n states per replica. eps == NULL: greedy (tanh(mean), models.py:101-102).
 * eps != NULL: action = tanh(mean + std*eps) and log_prob via the cached pre-tanh value (train.py:152,
 * training.py:20-22,34-36). given_action != NULL: log_prob of that action (models.py:97-99, atanh path).
 * Outputs may be NULL. workspace: il_actor_workspace_bytes. */
int64_t il_actor_workspace_bytes(const il_mlp* actor, int R, int n);
int il_actor_forward(il_handle* h, const il_mlp* actor, int R, int n,
                     const float* states, int64_t states_rs, int ld_states,
                     const float* eps, const float* given_action,
                     float* action, float* log_prob, float* mean, float* log_std,
                     void* workspace, int64_t workspace_bytes, void* stream);

/* ---- TwinCritic (models.py:123-141) -------------------------------------------------------------------- */
int64_t il_critic_workspace_bytes(const il_mlp* critic, int R, int n);
int il_critic_forward(il_handle* h, const il_mlp* twin, int R, int n, int S,
                      const float* states, int64_t states_rs, int ld_states,
                      const float* actions, int64_t actions_rs, int ld_actions,
                      float* q1, float* q2, void* workspace, int64_t workspace_bytes, void* stream);

/* update_target_network (models.py:79-81): target = tau*target + (1-tau)*online over n floats. */
int il_polyak(il_handle* h, float* target, const float* online, int64_t n, float polyak_factor, void* stream);

/* ---- sac_update (training.py:14-54) -------------------------------------------------------------------- */
typedef struct il_sac_args {
  il_mlp  actor, critic, target;    /* critic/target: 2R nets (twin), stride = per-net stride */
  il_adam actor_opt, critic_opt, alpha_opt;
  float*  log_alpha;                /* [R] */
  il_batch batch;                   /* transitions (rewards already relabelled by the caller, train.py:194) */
  const float* absorbing;           /* [R, B] or NULL = states[:, -1] of the batch when batch has absorbing bit */
  int32_t absorbing_from_state;     /* 1: take absorbing = state[S-1] (memory.py:62); 0 with absorbing == NULL: zeros */
  int32_t R;
  const float* eps_next;            /* [R, B, A] noise for training.py:21 */
  const float* eps_new;             /* [R, B, A] noise for training.py:35 */
  float discount, entropy_target, polyak_factor;
  float _pad0;
  float* out_log_probs;             /* [R, B] new_log_probs (training.py:54) */
  float* out_q_values;              /* [R, B] min(values_1, values_2) (training.py:54) */
  float* out_losses;                /* [R, 3] value, policy, temperature loss (may be NULL) */
  void*   workspace;
  int64_t workspace_bytes;
  const float* discount_r;          /* [R] per-replica discount / entropy_target / polyak_factor, or NULL = the scalar */
  const float* entropy_target_r;
  const float* polyak_r;
} il_sac_args;
int64_t il_sac_workspace_bytes(const il_sac_args* a);
int il_sac_update(il_handle* h, const il_sac_args* a, void* stream);

/* ---- behavioural_cloning_update (training.py:57-64): maximum-likelihood step of the actor on expert (state, action) rows */
typedef struct il_bc_args {
  il_mlp   actor;
  il_adam  opt;                     /* train.py:95 pretraining optimiser or the actor optimiser (train.py:201) */
  il_batch batch;                   /* expert transitions; uses states, actions, weights */
  int32_t  R;
  int32_t  _pad;
  float*   out_loss;                /* [R] mean(weight * -log_prob) (may be NULL) */
  void*    workspace;               /* il_bc_workspace_bytes */
  int64_t  workspace_bytes;
} il_bc_args;
int64_t il_bc_workspace_bytes(const il_bc_args* a);
int il_bc_update(il_handle* h, const il_bc_args* a, void* stream);

/* ---- networks with dropout (models.py:48-69 with input_dropout / dropout > 0): DRIL's policy ensemble and RED's predictor -----------
 * Dropout masks are explicit inputs, pre-scaled {0, 1/(1-p)}: mask_in [R, n, dims[0]] for the input, mask_hid[l] [R, n, dims[l+1]] for hidden
 * layer l (applied BEFORE the activation, models.py:54-61); NULL = no dropout at that site. il_fill_dropout_mask draws them (Philox). */
int il_fill_dropout_mask(il_handle* h, float* out, int64_t n, float p, uint64_t seed, uint64_t stream_id, const uint64_t* counter, void* stream);
int64_t il_actor_dropout_workspace_bytes(const il_mlp* actor, int R, int n);
/* SoftActor.log_prob(state, action) (models.py:97-99) of a dropout policy; rows of states / given_action are repeated `repeat` times
 * (torch.repeat_interleave of the 5-member MC-dropout ensemble, models.py:105): n = repeat * source rows. */
int il_actor_log_prob_dropout(il_handle* h, const il_mlp* actor, int R, int n, int repeat, const float* states, int64_t states_rs, int ld_states, const float* given_action,
                              const float* mask_in, const float* const* mask_hid, float* log_prob, void* workspace, int64_t workspace_bytes, void* stream);
/* behavioural_cloning_update (training.py:57-64) of a dropout policy (train.py:120); workspace: il_actor_dropout_workspace_bytes(actor, R, B). */
int il_bc_update_dropout(il_handle* h, const il_bc_args* a, const float* mask_in, const float* const* mask_hid, void* stream);
/* DRIL reward (models.py:104-120): reward = +1 where the unbiased variance over the ensemble of exp(log_prob[r, b * ensemble + e]) is <= q, else -1;
 * variance (optional [R, B]) receives the raw uncertainty (set_uncertainty_threshold takes its quantile). reward may be NULL. */
int il_dril_reward(il_handle* h, const float* log_prob, int R, int B, int ensemble, const float* q, int q_shared, float* reward, int64_t reward_rs, int reward_ld, float* variance,
                   void* stream);

/* ---- REDDiscriminator (models.py:252-284) and target_estimation_update (training.py:68-75) ------------------------------------------ */
typedef struct il_red {
  il_mlp  predictor;                /* R nets din -> hidden^depth -> din (EmbeddingNetwork, models.py:252-259); trained */
  il_mlp  target;                   /* R nets, frozen random embedding (models.py:266-268) */
  float*  sigma;                    /* [R] sigma_1 (models.py:269,277-280) */
  int32_t state_only, _pad;
} il_red;
typedef struct il_red_update_args {
  il_red   disc;
  il_adam  opt;                     /* AdamW over the predictor parameters (the frozen target has no gradient: train.py:84 skips it) */
  il_batch batch;                   /* expert transitions: states, actions, weights */
  int32_t  R, _pad;
  const float* mask_in;             /* predictor dropout masks (NULL = none) */
  const float* mask_hid[IL_MAX_LAYERS];
  float*   out_loss;                /* [R] (may be NULL) */
  void*    workspace;               /* il_red_workspace_bytes */
  int64_t  workspace_bytes;
} il_red_update_args;
int64_t il_red_workspace_bytes(const il_red* disc, int R, int B);
int il_red_update(il_handle* h, const il_red_update_args* a, void* stream);
/* set_sigma (models.py:277-280): sigma[r] = 1 / median over the B x B pairs of mean((prediction_i - target_j)^2) — in train mode in the reference, hence the masks */
int il_red_sigma(il_handle* h, const il_red* disc, int R, const il_batch* batch, const float* mask_in, const float* const* mask_hid, void* workspace, int64_t workspace_bytes, void* stream);
/* predict_reward (models.py:282-284), eval mode */
int il_red_reward(il_handle* h, const il_red* disc, int R, const il_batch* batch, float* reward, int64_t reward_rs, int reward_ld, void* workspace, int64_t workspace_bytes, void* stream);

/* AdamW step over a flat buffer (used by the fused updates; exposed for tests): torch _single_tensor_adam. */
int il_adam_step(il_handle* h, float* params, const float* grads, const il_adam* opt, int64_t n, void* stream);
/* The same step with update_target_network fused (training.py:33 + models.py:78-81): target = polyak * target + (1 - polyak) * params_new. */
int il_adam_step_polyak(il_handle* h, float* params, const float* grads, const il_adam* opt, int64_t n, float* target, float polyak_factor, void* stream);

/* ---- ReplayMemory (memory.py:12-68) --------------------------------------------------------------------- */
/* append (memory.py:40-44) of one transition per replica, with the train.py:157-162 flags: `terminal`
 * (early termination, stored), `timeout`; wrap != 0 applies wrap_for_absorbing_states (memory.py:65-68) to
 * replicas whose terminal flag is set. active[r] == 0 skips replica r (may be NULL). */
int il_replay_append(il_handle* h, const il_replay* mem, int R, const float* step, const float* state, const float* action,
                     const float* reward, const float* next_state, const float* terminal, const float* timeout,
                     const int32_t* active, int wrap, void* stream);
/* transfer_transitions (memory.py:46-48): appends every row of `src` (a single-store memory, e.g. the shared expert buffer) in
 * order to the ring of every replica of `dst` (weights reset to 1 by append, memory.py:41); used by train.py:133,141,143. */
int il_replay_transfer(il_handle* h, const il_replay* dst, int R, const il_replay* src, void* stream);
/* wrap_for_absorbing_states (memory.py:65-68) on the last appended row of every replica with mask != 0 (NULL = all). */
int il_replay_wrap_absorbing(il_handle* h, const il_replay* mem, int R, const int32_t* mask, void* stream);
/* _sample_idx x n (memory.py:51-59): uniform over valid rows, never the newest row. uniform != NULL: [R, n]
 * U[0,1) draws supplied by the caller (e.g. numpy on the host, like the reference) instead of device Philox. */
int il_replay_sample_indices(il_handle* h, const il_replay* mem, int R, int n, int32_t* idx_out, const float* uniform,
                             uint64_t seed, uint64_t stream_id, const uint64_t* counter, void* stream);
/* sample's gather (memory.py:60-62): out.rows[r, i, :] = mem.rows[r, idx[r, i], :] */
int il_replay_gather(il_handle* h, const il_replay* mem, int R, const int32_t* idx, const il_batch* out, void* stream);
/* mix_expert_agent_transitions (models.py:287-290): first B/2 rows <- expert rows (all fields). */
int il_mix_expert_rows(il_handle* h, const il_batch* batch, const il_batch* expert, int R, void* stream);

/* RewardRelabeller.resample_and_relabel (models.py:297-318): AdRIL (update_freq > 0) / SQIL (update_freq == 0) batch construction and reward
 * labels. balanced != 0: the batch becomes the expert batch on calls where *sample_expert_flag != 0 and stays the policy batch otherwise; the
 * flag (device scalar, initially 1) is toggled by the call. Otherwise the first B / 2 rows become expert rows. step = step_f[r] + step_offset. */
int il_adril_relabel(il_handle* h, const il_batch* batch, const il_batch* expert, int R, int balanced, int update_freq, int32_t* sample_expert_flag,
                     const float* step_f, float step_offset, const int32_t* num_trajectories, int trajectories_shared, int num_expert_trajectories, void* stream);

/* ---- GAILDiscriminator (models.py:152-180), depth-1 `g` network, optional spectral norm ------------------- */
typedef struct il_gail {
  il_mlp  g;                        /* R nets, n_layers == 2 (hidden_size x 1), `original` weights */
  float*  u;                        /* [R, u_stride] spectral-norm left vectors: layer0 [H], layer1 [1] (NULL = no SN) */
  float*  v;                        /* [R, v_stride] right vectors: layer0 [d], layer1 [H] */
  int32_t u_stride, v_stride;
  int32_t state_only;               /* imitation.state_only (models.py:156) */
  int32_t reward_function;          /* IL_REWARD_* */
} il_gail;
typedef struct il_gail_update_args {
  il_gail  disc;
  il_adam  opt;                     /* AdamW(imitation.learning_rate, imitation.weight_decay) train.py:84 */
  il_batch policy, expert;          /* transitions / expert_transitions (train.py:173) */
  const float* eps_gp;              /* [R, B] U(0,1) (training.py:118); required when grad_penalty > 0 */
  const float* eps_mix;             /* [R, B] Beta(a,a) draws (training.py:106); required for IL_LOSS_MIXUP */
  int32_t R;
  int32_t loss_function;            /* IL_LOSS_* */
  int32_t training;                 /* discriminator.train() (train.py:178): run the power iterations; 0 = eval-mode forwards */
  int32_t _pad;
  float grad_penalty, entropy_bonus, pos_class_prior, nonnegative_margin;
  float* out_losses;                /* [R, 2] bce/mixup loss, gp loss (may be NULL) */
  void*   workspace;                /* il_gail_workspace_bytes */
  int64_t workspace_bytes;
  const float* grad_penalty_r;      /* [R] per-replica grad_penalty / entropy_bonus, or NULL = the scalar. grad_penalty_r needs eps_gp; */
  const float* entropy_bonus_r;     /* the gradient-penalty pass runs for the replicas whose grad_penalty is > 0 */
} il_gail_update_args;
int64_t il_gail_workspace_bytes(const il_gail_update_args* a);
/* adversarial_imitation_update (training.py:85-134) incl. the train()/eval() power-iteration semantics. */
int il_gail_update(il_handle* h, const il_gail_update_args* a, void* stream);
/* forward logits (models.py:164-175, eval mode) and predict_reward (models.py:177-180); reward/logits may be NULL. */
int il_gail_reward(il_handle* h, const il_gail* disc, int R, const il_batch* batch, float* reward, int64_t reward_rs, int reward_ld,
                   float* logits, void* stream);

/* ---- general GAILDiscriminator (models.py:152-180): reward shaping (linear g + MLP h), subtract_log_policy, any depth / activation ----
 * g and h live in ONE flat [R, stride] parameter buffer (g at offset 0, h behind it; both il_mlp.stride == that stride), so one AdamW state
 * covers discriminator.parameters() (train.py:84). Spectral-norm vectors: per net, u = [u_0 | u_1 | ...] (layer l: dims[l+1] floats),
 * v = [v_0 | v_1 | ...] (layer l: dims[l] floats). */
typedef struct il_gailx {
  il_mlp  g;                        /* without shaping: the MLP of models.py:162; with shaping: nn.Linear (n_layers == 1), models.py:158 */
  il_mlp  h;                        /* shaping function (models.py:160); h.n_layers == 0: no reward shaping */
  float*  g_u; float* g_v;          /* [R, g_u_stride] / [R, g_v_stride]; NULL = no spectral norm */
  float*  h_u; float* h_v;
  int32_t g_u_stride, g_v_stride, h_u_stride, h_v_stride;
  int32_t state_only;               /* imitation.state_only (models.py:156) */
  int32_t reward_function;          /* IL_REWARD_* */
  int32_t subtract_log_policy;      /* models.py:175 */
  float   discount;                 /* models.py:174 */
  const float* discount_r;          /* [R] per-replica discount, or NULL = discount */
} il_gailx;
typedef struct il_gailx_update_args {
  il_gailx disc;
  il_adam  opt;                     /* AdamW over the flat buffer at disc.g.params (params_floats = R * stride floats) */
  int64_t  params_floats;
  il_batch policy, expert;
  const float* eps_gp;              /* [R, B] U(0,1) (training.py:118) */
  const float* eps_mix;             /* [R, B] Beta(a, a) (training.py:106) */
  const float* logp_policy;         /* [R, B] log pi(a|s) of the policy batch (make_gail_input, models.py:148); subtract_log_policy only */
  const float* logp_expert;         /* [R, B] of the expert batch */
  const float* logp_mix;            /* [R, B] of the Mixup batch (il_gail_mix_batch of expert and policy with eps_mix) */
  int32_t R, loss_function, training, _pad;
  float grad_penalty, entropy_bonus, pos_class_prior, nonnegative_margin;
  float* out_losses;                /* [R, 2] (may be NULL) */
  void*   workspace;                /* il_gailx_workspace_bytes */
  int64_t workspace_bytes;
  const float* grad_penalty_r;      /* [R] or NULL, as in il_gail_update_args. The scalar grad_penalty > 0 selects the gradient-penalty pass for */
  const float* entropy_bonus_r;     /* every replica: one with grad_penalty_r[r] == 0 adds no penalty but still runs that pass's power iteration */
} il_gailx_update_args;
int64_t il_gailx_workspace_bytes(const il_gailx_update_args* a);
int il_gailx_update(il_handle* h, const il_gailx_update_args* a, void* stream);      /* training.py:85-134 */
int64_t il_gailx_reward_workspace_bytes(const il_gailx* disc, int R, int B);
int il_gailx_reward(il_handle* h, const il_gailx* disc, int R, const il_batch* batch, const float* log_policy, float* reward, int64_t reward_rs, int reward_ld,
                    float* logits, void* workspace, int64_t workspace_bytes, void* stream);   /* models.py:164-180, eval mode */
/* _mix_vars (training.py:79-81) on every field of the packed rows: out = eps * expert + (1 - eps) * policy */
int il_gail_mix_batch(il_handle* h, const il_batch* expert, const il_batch* policy, const float* eps, int R, const il_batch* out, void* stream);

/* ---- GMMILDiscriminator (models.py:183-201) ------------------------------------------------------------- */
/* bandwidths (models.py:193-195): gamma[r, 0:2] = 1 / (weighted median + 1e-8). workspace: il_gmmil_workspace_bytes. */
int64_t il_gmmil_workspace_bytes(int R, int B);
int il_gmmil_bandwidth(il_handle* h, int R, const il_batch* policy, const il_batch* expert, int state_only, float* gamma,
                       void* workspace, int64_t workspace_bytes, void* stream);
int il_gmmil_reward(il_handle* h, int R, const il_batch* policy, const il_batch* expert, int state_only, const float* gamma,
                    float* reward, int64_t reward_rs, int reward_ld, void* stream);

/* ---- PWILDiscriminator (models.py:216-249) -------------------------------------------------------------- */
typedef struct il_pwil {
  const float* atoms;               /* [N, d] normalised expert atoms (models.py:229), shared by all replicas */
  const float* scale;               /* [d]  (models.py:205-208) */
  const float* offset;              /* [d] */
  float*   weights;                 /* [R, N] remaining expert weights; consumed atoms have weight < 0 */
  int32_t  N, d, S, A;
  int32_t  state_only, time_horizon;
  float    reward_scale, reward_bandwidth;
  const float* reward_scale_r;      /* [R] per-replica reward_scale / reward_bandwidth, or NULL = the scalar */
  const float* reward_bandwidth_r;
} il_pwil;
int il_pwil_reset(il_handle* h, const il_pwil* p, int R, const int32_t* mask, void* stream);   /* models.py:228-230 */
int il_pwil_reward(il_handle* h, const il_pwil* p, int R, const float* state, const float* action, float* reward,
                   const int32_t* active, void* stream);                                           /* models.py:232-249 */

/* ---- synthetic batched environment (stands in for environments.py:29-40 gym/MuJoCo stepping) ------------- */
typedef struct il_env {
  const float* M;                   /* [obs, obs] */
  const float* N;                   /* [act, obs] */
  const float* c;                   /* [obs] */
  const float* w_r;                 /* [obs] */
  float*   x;                       /* [n_envs, obs] physical state */
  int32_t* t;                       /* [n_envs] steps in the current episode */
  int32_t  obs, act, absorbing, max_episode_steps, early_termination;
  float    term_threshold;
} il_env;
/* reset (environments.py:29-33): x = (2u-1)*0.1 for envs with mask != 0 (mask NULL = all); writes state [n, S].
 * Envs with mask == 0 keep their state, or receive else_state[i] when else_state != NULL (state <- next_state). */
int il_env_reset(il_handle* h, const il_env* env, int n_envs, const float* u, const int32_t* mask, float* state, const float* else_state, void* stream);
/* step (environments.py:35-40): clamp action to [-1,1], advance, reward, done (= terminated OR time limit).
 * terminal_f / timeout_f (nullable) are the floats train.py:157 stores: done && t != max, t == max.
 * frozen[i] != 0 leaves env i untouched (finished evaluation episodes). */
int il_env_step(il_handle* h, const il_env* env, int n_envs, const float* action, float* next_state, float* reward,
                int32_t* done, int32_t* timeout, float* terminal_f, float* timeout_f, const int32_t* frozen, void* stream);

/* training-loop bookkeeping of train.py:155,165-168 for R envs: running[i] += reward[i]; where done[i]: last_return[i] =
 * running[i], return_sum[i] += running[i], episodes[i] += 1, running[i] = 0. Also step_f[i] += 1 (the `step` stored by
 * memory.append, train.py:157) when step_f != NULL. */
int il_rollout_bookkeep(il_handle* h, int n_envs, const float* reward, const int32_t* done, float* running, float* last_return,
                        float* return_sum, int32_t* episodes, float* step_f, void* stream);

/* ---- evaluation (evaluation.py:11-35) --------------------------------------------------------------------- */
/* return accumulation for batched greedy episodes: returns[i] += reward[i] for non-finished episodes, then
 * finished[i] |= done[i]. n_unfinished (device scalar) receives the number of running episodes. */
int il_eval_accumulate(il_handle* h, int n_envs, const float* reward, const int32_t* done, float* returns, int32_t* finished,
                       int32_t* n_unfinished, void* stream);
/* per-rank statistics vector for the NCCL reduction (SURVEY §8e): out[0:3] = sum, sum of squares, count. */
int il_return_stats(il_handle* h, const float* returns, int64_t n, float* out3, void* stream);

/* evaluate_agent (evaluation.py:11-35) as one device program: R x episodes greedy episodes (get_greedy_action, models.py:101-102)
 * advance in lock-step inside a CUDA graph WHILE node whose condition is set on the device, so the host launches once and is not
 * involved until every episode has ended (finished episodes are frozen). The caller resets the environments first (il_env_reset
 * into `state`). Not capturable itself (it launches its own graph). */
typedef struct il_eval_args {
  il_mlp   actor;                   /* R nets */
  il_env   env;                     /* R * episodes evaluation environments (x, t hold their state) */
  int32_t  R, episodes;
  int32_t  max_steps;               /* safety bound on loop iterations (>= env.max_episode_steps) */
  int32_t  traj_T;                  /* capacity (steps) of the trajectory buffers */
  float*   state;                   /* [R * episodes, S] in: initial states (il_env_reset); scratch afterwards */
  float*   returns;                 /* [R * episodes] out: sum of rewards per episode (evaluation.py:28) */
  float*   traj_states;             /* optional [R * episodes, traj_T, S]   (return_trajectories, evaluation.py:22,33) */
  float*   traj_actions;            /* optional [R * episodes, traj_T, A] */
  float*   traj_rewards;            /* optional [R * episodes, traj_T] */
  int32_t* traj_len;                /* optional [R * episodes] steps recorded per episode */
  int64_t* out_counters;            /* optional [2]: loop iterations executed, environment steps executed */
  void*    workspace;               /* il_eval_workspace_bytes */
  int64_t  workspace_bytes;
} il_eval_args;
int64_t il_eval_workspace_bytes(const il_eval_args* a);
int il_eval_rollout(il_handle* h, const il_eval_args* a, void* stream);

/* train.py:213-219 across the seed-sharded ranks (SURVEY §8e): out3 = (sum, sum of squares, count) of this rank's returns, then
 * ncclAllReduce(sum) over `nccl_comm` (an ncclComm_t; NULL = single process) enqueued on the same stream — no host involvement.
 * il_nccl_* create that communicator from a 128-byte ncclUniqueId the caller distributes (e.g. a torch.distributed broadcast);
 * NCCL is bound at run time (libnccl.so.2, the copy the host framework already loaded). */
int il_nccl_unique_id(uint8_t* out128);                                   /* HOST pointer */
int il_nccl_comm_create(const uint8_t* id128, int rank, int world, void** comm);  /* HOST pointers */
int il_nccl_comm_destroy(void* comm);
int il_return_allreduce(il_handle* h, void* nccl_comm, const float* returns, int64_t n, float* out3, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* IL_B200_H */
