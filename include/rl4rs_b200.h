/*
 * rl4rs_b200.h -- C-ABI of the B200-native RL4RS hot path (librl4rs_b200.so).
 *
 * The reference has no FFI: its "operator API" for this path is the Python protocol
 * RecEnvBase / RecSimBase / RecState (rl4rs/env/base.py:26-57,111-175,178-273).  Each entry
 * point below names the reference interface it replaces (file:line under /root/reference).
 * The Python mirror of those classes (rl4rs_b200/env/) binds this library through ctypes
 * (rl4rs_b200/_capi.py); INTEGRATION.md shows the stub a reference maintainer would add.
 *
 * Conventions: plain pointers and sizes only (no torch types); return 0 on success, a negative
 * r4_status otherwise, r4_last_error() gives the message; nothing throws across the ABI.
 * "dev" pointers are device memory owned by the CALLER (allocated by torch on the Python side);
 * the library only borrows them for the work it enqueues on `stream` (a cudaStream_t passed as
 * void*; NULL = legacy default stream).  Every call is asynchronous on that stream.  One r4_env
 * per device, not thread-safe (the reference is single-threaded, base.py:119-130); distinct
 * handles are independent.
 */
#ifndef RL4RS_B200_H
#define RL4RS_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct r4_env r4_env;

typedef enum {
  R4_OK = 0,
  R4_ERR_ARG = -1,      /* bad argument / unsupported configuration */
  R4_ERR_STATE = -2,    /* call out of order (e.g. step before reset, step past max_steps) */
  R4_ERR_CUDA = -3,     /* CUDA runtime error (message holds cudaGetErrorString) */
  R4_ERR_NOMEM = -4
} r4_status;

/* config['...'] flags read by the reference via config.get (slate.py:22,92,98,153,245,250,299) */
enum {
  R4_FLAG_RLLIB_MASK = 1,     /* support_rllib_mask */
  R4_FLAG_D3RL_MASK = 2,      /* support_d3rl_mask */
  R4_FLAG_CONTI = 4,          /* support_conti_env */
  R4_FLAG_ONEHOT = 8,         /* support_onehot_action (action_emb = eye(action_size)) */
  R4_FLAG_RAWSTATE = 16,      /* rawstate_as_obs: no simulator forward for observations */
  R4_FLAG_INFO_FETCH = 32     /* simulator_info_fetch: expose per-item click probabilities */
};

enum { R4_ENV_SLATE = 0, R4_ENV_SEQSLATE = 1 };   /* rl4rs/__init__.py:10-18 */
/* config['algo'] (slate.py:239-242): which rl4rs/nets/<algo>.py graph the simulator is.
 *   DIEN  nets/dien.py:8-45   (sequence GRU/attention/AUGRU + dense tower + category attention; tensor-bound)
 *   DNN   nets/dnn.py:8-45    (mean-pooled category embeddings + dense tower + FC 256 + simulator_obs; gather-bound:
 *                              the sequence branch of that graph does not reach the output and is not evaluated)
 *   WIDEDEEP  nets/widedeep.py:8-45 (mean-pooled sequence embeddings -> Dense 256 | dense tower | flattened category
 *                              embeddings; 'simulator_obs' IS that 3072-wide concat, so obs buffers are f32 [B,3072])
 *   LSTM  nets/lstm.py:8-45   (Keras GRU -- hard sigmoid, reset_after False -- over each behaviour sequence and over the 21
 *                              category embeddings | dense tower | flattened category embeddings -> simulator_obs 256) */
enum { R4_SIM_DIEN = 0, R4_SIM_DNN = 1, R4_SIM_WIDEDEEP = 2, R4_SIM_LSTM = 3 };
/* width of the observation a simulator produces (256, or 3072 for widedeep) */
int r4_obs_dim(int simulator);

/* The config dict of the reference scripts (simulator_eval.py:9-12, modelfree_train.py:32-37). */
typedef struct {
  int32_t env_kind;             /* R4_ENV_SLATE | R4_ENV_SEQSLATE */
  int32_t flags;                /* R4_FLAG_* */
  int32_t batch_size;
  int32_t max_steps;            /* 9 (Slate) / 27 or 36 (SeqSlate) */
  int32_t page_items;           /* 9 */
  int32_t action_size;          /* 284 */
  int32_t action_emb_size;      /* 32 (ignored with R4_FLAG_ONEHOT) */
  int32_t maxlen;               /* 64 */
  int32_t seq_num;              /* 2 */
  int32_t dense_feature_num;    /* 432 */
  int32_t category_feature_num; /* 21 */
  int32_t category_hash_size;   /* 100000 */
  int32_t emb_size;             /* 128 */
  int32_t hidden_units;         /* 128 */
  int32_t max_rows_per_pass;    /* 0 = default; bound on simulator rows per launch group */
  int32_t simulator;            /* R4_SIM_DIEN | R4_SIM_DNN | R4_SIM_WIDEDEEP | R4_SIM_LSTM (ABI version >= 2) */
} r4_config;

/* Per-call output buffers (device, caller-owned).  NULL = not wanted.
 * Replaces the return values of RecSimBase._step / sample (base.py:157-175) and
 * SlateRecEnv.obs_fn (slate.py:244-279). */
typedef struct {
  float*   obs;          /* f32 [B,256]   simulator_obs layer (dien.py:35; [B,3072] for widedeep); NULL with RAWSTATE */
  uint8_t* action_mask;  /* u8  [B,A]     action_mask & location_mask & special_mask (slate.py:93-97) */
  double*  reward;       /* f64 [B]       slate.py:281-308 / seqslate.py:136-160 */
  uint8_t* done;         /* u8  [B]       base.py:165-168 */
  int32_t* chosen;       /* i32 [B]       item ids actually placed (kNN result in conti mode) */
  int32_t* cat;          /* i32 [B,21]    category_feature of the new state (datautil.py:59-65) */
  float*   dense;        /* f32 [B,432]   dense_feature (datautil.py:52-58) */
  int32_t* seq;          /* i32 [B,2,64]  sequence_feature (datautil.py:43-47) */
  float*   click_p;      /* f32 [B,9]     probs[:,1] of the reward pass (slate.py:298-301); written
                                          only on steps that compute a reward */
  int32_t* masked_actions; /* i32 [B,9|max_steps] d3rl 'masked_actions' (slate.py:98-104, seqslate.py:18-23) */
} r4_out;

/* ---- lifetime ---------------------------------------------------------------------------- */
/* SlateRecEnv.__init__/RecSimBase.__init__ (slate.py:223-237, base.py:114-131) */
int r4_create(const r4_config* cfg, int device, r4_env** out);
void r4_destroy(r4_env* env);
const char* r4_last_error(const r4_env* env);   /* env may be NULL: error of the last failed r4_create */

/* ---- static data ------------------------------------------------------------------------- */
/* SlateState.get_iteminfo_from_file / get_mask_from_file (slate.py:28-65).  HOST pointers,
 * n = action_size rows, row 0 = the implicit padding item.  special[i] != 0 marks the ids whose
 * special column == 2.  action_emb is f64 [n, emb_dim] (slate.py:47-52; eye(n) with ONEHOT). */
int r4_load_items(r4_env* env, const double* item_vec, int vec_dim, const double* price,
                  const uint8_t* special, const double* action_emb, int emb_dim, int n);

/* tf.train.Saver.restore (base.py:148-151): one named f32 tensor of the W-table (SURVEY.md 8a);
 * `data` may be a host or a device pointer.  r4_finalize_weights derives the fused layouts. */
int r4_load_weight(r4_env* env, const char* name, const float* data, const int64_t* shape, int rank);
int r4_finalize_weights(r4_env* env, void* stream);

/* RecDataBase (base.py:60-108): the parsed log, structure-of-arrays, DEVICE pointers that must
 * stay valid until the next r4_load_log / r4_destroy.  user_seq is pre-padded/truncated to maxlen
 * (datautil.py:43-46).  n_slots = 9 (dataset A) or 36 (b3 trajectories). */
int r4_load_log(r4_env* env, const int32_t* user_cat /*[N,10]*/, const float* user_dense /*[N,32]*/,
                const int32_t* user_seq /*[N,maxlen]*/, const int32_t* logged_items /*[N,n_slots]*/,
                const uint8_t* feedback /*[N,n_slots]*/, int64_t n_rows, int n_slots);

/* ---- episode ----------------------------------------------------------------------------- */
/* RecEnvBase.reset -> RecSimBase.sample (base.py:265-269,172-175): row_idx i32[B] (device) are
 * the log rows RecDataBase.sample chose (base.py:92-100). */
int r4_reset(r4_env* env, const int32_t* row_idx, const r4_out* out, void* stream);

/* RecEnvBase.step -> RecSimBase._step (base.py:256-263,157-170) -> SlateState.act
 * (slate.py:193-214 / seqslate.py:92-126).  action: i32[B] item ids, or with R4_FLAG_CONTI
 * f32[B,emb] (action_is_f64 = 0) / f64[B,emb] (action_is_f64 = 1) embeddings resolved by
 * get_nearest_neighbor_with_mask (slate.py:186-191). */
int r4_step(r4_env* env, const void* action, int action_is_f64, const r4_out* out, void* stream);

/* SlateState.offline_action / offline_reward (slate.py:149-174, seqslate.py:71-86).
 * items: i32[B]; emb (conti mode, may be NULL): f64[B,emb_dim]; reward: f64[B]. */
int r4_offline_action(r4_env* env, int32_t* items, double* emb, void* stream);
int r4_offline_reward(r4_env* env, double* reward, void* stream);

/* SlateState.get_violation (slate.py:133-147 / seqslate.py:52-69): i32[B] of 0/1. */
int r4_violation(r4_env* env, int32_t* out, void* stream);

/* The raw feature rows of the CURRENT state -- what RecState.state hands to obs_fn (slate.py:90-106, built by
 * slate.py:67-83,203-213 and padded by FeatureUtil.feature_extraction, datautil.py:34-69) -- without a simulator
 * pass: cat i32[B,21], dense f32[B,432], seq i32[B,2,64] (any may be NULL).  For custom obs_fn plug-ins. */
int r4_features(r4_env* env, int32_t* cat, float* dense, int32_t* seq, void* stream);

/* SlateState.get_nearest_neighbor (static, unmasked; slate.py:180-184; tutorial.ipynb:251-254) */
int r4_nearest_neighbor(r4_env* env, const void* action, int action_is_f64, int n, int32_t* out,
                        void* stream);

/* ---- introspection ----------------------------------------------------------------------- */
int r4_cur_steps(const r4_env* env);                 /* SlateState.cur_steps */
const int32_t* r4_prev_actions(const r4_env* env);   /* device i32[B,max_steps] (SlateState.prev_actions) */
int r4_copy_prev_actions(r4_env* env, int32_t* out /*dev i32[B,max_steps]*/, void* stream);
/* kernel launches issued by this handle since creation (bench.py's gpu_launches) */
int64_t r4_launch_count(const r4_env* env);
/* Per-kernel timing with CUDA events on the launching stream (bench.py's roofline leg).
 * mode 0 = off, 1 = the dominant kernel only (k_recur<256>, the AUGRU recurrence), 2 = every kernel.
 * r4_profile resets the counters; r4_profile_read synchronises the recorded events and returns, for
 * slot = 0,1,2,... the kernel name, summed device milliseconds, launches and algorithmic work
 * (FLOPs for the GEMM-shaped kernels, rows otherwise); it returns 1 past the last slot. */
int r4_profile(r4_env* env, int mode);
int r4_profile_read(r4_env* env, int slot, const char** name, double* ms, int64_t* launches, double* work);
/* ABI version of the build */
int r4_abi_version(void);
/* Which AUGRU kernel an observation / reward pass of `ctas` = 2 x ceil(rows / 128) tile-sequences runs on a device
 * with `sms` multiprocessors: 2 = k_augru_pair2 (one recurrence per 2-CTA cluster, tcgen05.mma.cta_group::2),
 * 3 = k_augru_pp (both sequences of a tile per cluster); 0 for bad arguments.  Pure host arithmetic, exposed so the
 * choice is testable and so a caller can predict the rounding regime of a launch (the two kernels agree to the parity
 * tolerance, not bit for bit).  No reference counterpart. */
int r4_augru_kernel_for(int ctas, int sms);
/* Process-wide kernel-choice overrides for parity tests and A/B timing (no reference counterpart):
 *   "augru_kernel"     0 = by r4_augru_kernel_for (default), 2 = always the pair kernel, 3 = always the ping-pong pair kernel
 *                      (two recurrences per pair)
 *   "augru_cost_pair" / "augru_cost_pp"  the per-wave costs r4_augru_kernel_for compares (positive ints)
 *   "pay_obs_reuse"    1 (default): r4_step takes the observation of a PAYING step (the last step of a slate / page) from that
 *                      step's reward pass -- the state the step leaves (rl4rs/env/slate.py:203-213, seqslate.py:104-122) is the
 *                      last of the page's complete states (slate.py:117-131, seqslate.py:27-50), so the reference runs the same
 *                      feature row through the simulator twice; 0: launch the separate observation pass as well
 *   "scores_shared_pct" share of an even CTA split given to a sequence whose cached rows are shared by all feature rows
 *                      (Slate's constant second sequence), 10..100 per cent
 * The environment variables R4_AUGRU_PAIR / R4_AUGRU_PP / R4_AUGRU_RULE / R4_NO_PAY_OBS_REUSE give the initial values.
 * Returns 0, or R4_ERR_ARG for an unknown key / out-of-range value. */
int r4_set_option(const char* key, int value);

/* ---- policy + learner (K12): MyMaskActionsModel (rllib_mask_model.py:41-62) and the RLlib PPO / A2C losses ----
 * Stateless: every pointer is caller-owned DEVICE memory.  Flat parameter layout:
 * w1[256,64] b1[64] w2[64,A] b2[A] wv[64] bv[1]  (r4_policy_num_params(A) floats). */
int r4_policy_num_params(int action_size);
/* forward + SoftQ(T=1) sampling (explore != 0) or argmax (modelfree_train.py:398-402,412-414); obs f32[n,256],
 * mask u8[n,A] -> action i32[n], logp f32[n], value f32[n], logits f32[n,A] (masked logits; may be NULL). */
int r4_policy_act(const float* params, const float* obs, const uint8_t* mask, int n, int action_size, int explore,
                  uint64_t seed, uint64_t counter, int32_t* action, float* logp, float* value, float* logits,
                  void* stream);
/* gradient of the RLlib loss over samples idx[0..n) (NULL = 0..n-1) of a rollout:
 * mode 0 PPO surrogate (mean; modelfree_train.py:179-217), mode 1 A2C (sums; :248-304).
 * scratch: f32[G * (num_params + 5)], G = min(ceil(n/4), 148) CTAs; flat_grad f32[num_params] receives the
 * deterministic sum; stats_accum f32[5] += {policy_loss, vf_loss, kl, entropy, total} * stat_scale. */
int r4_policy_grad(int mode, const float* params, const float* obs, const uint8_t* mask, const int64_t* action,
                   const float* old_logp, const float* old_logits, const float* old_value, const float* adv,
                   const float* target, const int64_t* idx, int n, int action_size, float clip, float vf_clip,
                   float vf_coeff, float kl_coeff, float ent_coeff, float inv_n, float* scratch, int G,
                   float* flat_grad, float* stats_accum, float stat_scale, void* stream);
/* Generalised advantage estimation over complete episodes (RLlib postprocessing compute_advantages, bootstrap value 0):
 * reward / value / adv / target are f32 [T, B] device arrays; target = adv + value; gamma_lambda = the product gamma * lambda
 * (rounded once by the caller, as the reference's float arithmetic does).  One launch instead of a host loop. */
int r4_gae(const float* reward, const float* value, int T, int B, float gamma, float gamma_lambda, float* adv, float* target, void* stream);
/* Adam (torch.optim.Adam semantics) with optional global-norm clipping (clip <= 0 off; norm_scratch f32[1]).
 * grad_scale multiplies the gradient first (1/world after a SUM all-reduce). step is 1-based. */
int r4_adam_step(float* params, const float* grad, float* m, float* v, int n, int step, float lr, float beta1,
                 float beta2, float eps, float grad_scale, float clip, float* norm_scratch, void* stream);

/* One PPO SGD epoch on a single GPU (num_sgd_iter = 1 of modelfree_train.py:179-217): for every full minibatch
 * perm[s .. s+mb) of the rollout, r4_policy_grad (mode 0, mean over mb) followed by r4_adam_step, with no host round
 * trip between the steps.  step0 = Adam steps already taken; returns the number of steps done (>= 0) or a negative
 * r4_status.  Multi-GPU learners call r4_policy_grad / all-reduce / r4_adam_step per step instead. */
int r4_ppo_epoch(float* params, const float* obs, const uint8_t* mask, const int64_t* action, const float* old_logp,
                 const float* old_logits, const float* old_value, const float* adv, const float* target,
                 const int64_t* perm, int n, int mb, int action_size, float clip, float vf_clip, float vf_coeff,
                 float kl_coeff, float ent_coeff, float* scratch, float* flat_grad, float* stats_accum, float* m,
                 float* v, int step0, float lr, float beta1, float beta2, float eps, float grad_clip,
                 float* norm_scratch, void* stream);

/* ---- data-parallel learner: gradient exchange over NVLink peer memory (SURVEY.md 8e; no reference counterpart:
 * the reference's multi-worker path is Ray's object store, modelfree_train.py:181,403-405) ----------------------
 * One communicator per rank (= process = GPU).  r4_comm_create allocates this rank's inbox + flags on the CURRENT
 * device; r4_comm_handle exports it (64 bytes = cudaIpcMemHandle_t) for the caller to all-gather by any means
 * (torch.distributed here); r4_comm_open maps every peer's allocation (handles in rank order, world x 64 bytes).
 * After that the SGD steps of an epoch need no host-side collective: r4_ppo_epoch_dist enqueues, per minibatch,
 * the gradient kernel and ONE kernel that reduces the local partials, pushes them into every rank's inbox, waits
 * for the peers' flags, sums in rank order and applies Adam (replicas stay bit-identical).  Every rank must call
 * it with the same n, mb and hyper-parameters.  mb = minibatch size PER RANK; the loss is the mean over
 * mb x world samples (RLlib: sgd_minibatch_size is the total over devices). */
typedef struct r4_comm r4_comm;
int r4_comm_create(int rank, int world, int n_params, r4_comm** out);
int r4_comm_handle(r4_comm* comm, void* handle_out_64);
int r4_comm_open(r4_comm* comm, const void* handles, int n_handles);
void r4_comm_destroy(r4_comm* comm);
int r4_ppo_epoch_dist(r4_comm* comm, float* params, const float* obs, const uint8_t* mask, const int64_t* action,
                      const float* old_logp, const float* old_logits, const float* old_value, const float* adv,
                      const float* target, const int64_t* perm, int n, int mb, int action_size, float clip,
                      float vf_clip, float vf_coeff, float kl_coeff, float ent_coeff, float* scratch, float* flat_grad,
                      float* stats_accum, float* m, float* v, int step0, float lr, float beta1, float beta2, float eps,
                      void* stream);
/* The exchange alone: partial gradients of ONE r4_policy_grad-style launch (scratch, G as there; the caller ran the
 * gradient kernel through r4_policy_grad_partial) -> flat_grad = sum over ranks (A2C: global-norm clipping and Adam
 * follow through r4_adam_step). */
int r4_policy_grad_partial(int mode, const float* params, const float* obs, const uint8_t* mask, const int64_t* action,
                           const float* old_logp, const float* old_logits, const float* old_value, const float* adv,
                           const float* target, const int64_t* idx, int n, int action_size, float clip, float vf_clip,
                           float vf_coeff, float kl_coeff, float ent_coeff, float inv_n, float* scratch, int G,
                           void* stream);
int r4_grad_exchange(r4_comm* comm, const float* scratch, int G, int action_size, float* flat_grad, float* stats_accum,
                     float stat_scale, void* stream);

/* ---- the simulator alone (nets/dien.py:8-45), for parity tests and kernel benchmarks ------- */
/* seq i32[R,2,64], dense f32[R,432], cat i32[R,21] (device) -> obs f32[R,256], probs f32[R,2]
 * (either may be NULL).  Runs the uncached path: GRU-1 is recomputed for every row. */
int r4_dien_forward(r4_env* env, const int32_t* seq, const float* dense, const int32_t* cat,
                    int n_rows, float* obs, float* probs, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* RL4RS_B200_H */
