/*
 * drl_b200.h -- C ABI of libdrl_b200.so: the B200 (sm_100a) implementation of the PPO
 * rollout-and-update hot path of qgallouedec/deep_rl `deep_rl/ppo.py`.
 *
 * The reference has no FFI of its own (it is a Python script); each entry point below replaces a
 * span of that script, cited as ppo.py:LINES.  Conventions:
 *   - every pointer is CALLER-OWNED DEVICE memory unless the name ends in `_host`; the library
 *     never allocates, frees or retains device memory, and keeps no state between calls;
 *   - every call is asynchronous on `stream` (a cudaStream_t passed as void*, NULL = default stream)
 *     and never synchronises with the host;
 *   - return value 0 = ok, negative = error (drl_last_error() gives the message of the calling
 *     thread's last failure); no C++ exception crosses this boundary;
 *   - one host thread per device/stream; entry points are re-entrant across threads.
 *
 * Layouts (N = envs on this rank, T = num_steps, O = obs dim, OP = padded obs stride, A = actions):
 *   rollout buffer planes are [T+1][N] with N contiguous, keeping the reference's one-slot shift
 *   (ppo.py:93-98,113-141): rew[t+1], done[t+1] belong to act[t]; val[t] = V(obs[t]); obs is
 *   [T+1][N][OP] float (OP = 4 CartPole, 8 Acrobot, pad lanes zero).
 *   sample id s = t*N + n, 0 <= s < B = T*N.
 */
#ifndef DRL_B200_H
#define DRL_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DRL_ABI_VERSION 2

enum { DRL_ENV_CARTPOLE = 0, DRL_ENV_ACROBOT = 1, DRL_ENV_MOUNTAINCAR = 2 };   /* gym ids CartPole-v1, Acrobot-v1, MountainCar-v0 */
enum { DRL_OK = 0, DRL_ERR_ARG = -1, DRL_ERR_UNSUPPORTED = -2, DRL_ERR_CUDA = -3 };

/* Batched environment: replaces gym.make + TimeLimit + RecordEpisodeStatistics + TorchWrapper
 * (ppo.py:10-22,79-80) and the manual auto-reset of ppo.py:127-129, for N envs. */
typedef struct {
    int32_t  kind;               /* DRL_ENV_* */
    int32_t  num_envs;           /* N on this rank */
    uint64_t seed;               /* Philox key (ppo.py:83-84) */
    uint32_t env_gid0;           /* global id of local env 0 (rank * N) -- Philox counter word */
    int32_t  max_episode_steps;  /* TimeLimit, 500 for CartPole-v1 / Acrobot-v1 */
    double*  state;              /* [4][N] float64, SoA (gym keeps float64 state) */
    int32_t* elapsed;            /* [N] TimeLimit counter */
    float*   ep_ret;             /* [N] running episode return (float32 like RecordEpisodeStatistics) */
    int32_t* ep_len;             /* [N] running episode length */
} drl_env_t;

/* Finished-episode log: replaces info["episode"] + the print of ppo.py:130.  One 24-byte record per finished episode (array of
 * structs: the host fetches a prefix of the log with ONE device->host copy).  All fields optional (pass a NULL drl_ep_log_t*
 * to drop the log). */
typedef struct {
    uint64_t step;       /* global step index (0-based) at which the episode ended */
    uint32_t env;        /* global env id */
    float    ret;        /* episodic return (float32 like RecordEpisodeStatistics) */
    int32_t  len;        /* episode length */
    uint32_t pad;
} drl_ep_entry_t;
typedef struct {
    uint32_t*       count;     /* [1] episodes finished (atomic; may exceed cap, entries beyond cap dropped) */
    double*         sum_ret;   /* [1] sum of finished returns */
    double*         sum_len;   /* [1] sum of finished lengths */
    drl_ep_entry_t* entries;   /* [cap] */
    uint32_t        cap;
} drl_ep_log_t;

/* Actor-critic shape (ppo.py:31-47): two separate tanh MLPs O->H->H->A and O->H->H->1. */
typedef struct {
    int32_t obs_dim;      /* O */
    int32_t hidden;       /* H (64 supported) */
    int32_t num_actions;  /* A */
    int32_t obs_stride;   /* OP */
} drl_net_t;

typedef struct {
    float*   obs;   /* [T+1][N][OP] */
    uint8_t* act;   /* [T+1][N] */
    float*   logp;  /* [T+1][N] */
    float*   val;   /* [T+1][N] */
    float*   rew;   /* [T+1][N] */
    uint8_t* done;  /* [T+1][N] */
    float*   logits; /* optional debug plane [T][N][A]: the logits each action was sampled from (NULL = not recorded);
                        lets a test feed the kernel's own logits to the oracle sampler and demand identical actions */
} drl_rollout_buf_t;

typedef struct {
    float clip_coef;  /* ppo.py:72 */
    float ent_coef;   /* ppo.py:73 */
    float vf_coef;    /* ppo.py:74 */
} drl_ppo_coef_t;

/* Device-resident counters of one trainer (caller-owned device memory, sizeof(drl_ctrl_t) bytes).  The *_ctl entry points
 * read their step / epoch / optimizer-step numbers from it instead of from by-value arguments, so that the launches of a
 * whole update can be captured ONCE in a CUDA graph and replayed: only drl_ctrl_set (outside the graph, one tiny launch whose
 * kernel parameters carry the new values) runs per update. */
#define DRL_CTRL_MAX_STEPS 64
typedef struct {
    uint64_t env_step;    /* Philox step index of the first rollout step (= step0 of drl_rollout) */
    uint32_t epoch_ctr;   /* permutation counter of the update's first epoch */
    uint32_t comm_seq;    /* sequence number of the last fused multi-GPU minibatch step before this update */
    int64_t  adam_step;   /* optimizer steps taken before this update */
    float    neg_step_size[DRL_CTRL_MAX_STEPS];   /* -lr / (1 - beta1^k) for the update's k-th optimizer step */
    float    bc2_sqrt[DRL_CTRL_MAX_STEPS];        /* sqrt(1 - beta2^k) */
} drl_ctrl_t;

int         drl_abi_version(void);
const char* drl_last_error(void);

/* ---- shapes ---- */
int drl_env_obs_dim(int32_t kind);
int drl_env_num_actions(int32_t kind);
int drl_env_obs_stride(int32_t kind);
/* canonical flat parameter count (state_dict order, ppo.py:34-47) and packed-layout float count */
int64_t drl_param_count(const drl_net_t* net);
int64_t drl_packed_count(const drl_net_t* net);
/* sample-record width in floats (8 for O<=4, 16 otherwise) */
int drl_record_width(const drl_net_t* net);
/* bytes of zero-initialised scratch the update entry points need.  One workspace serves one trainer: calls on the SAME stream
 * may share it freely; the statistics calls (drl_adv_stats, drl_adv_stats_perm) use regions disjoint from those of the
 * minibatch calls, so they may also run on a second stream while a minibatch step is in flight (but not two statistics
 * calls, or two minibatch calls, concurrently). */
size_t drl_workspace_bytes(const drl_net_t* net);

/* ---- environment (ppo.py:17,21,79,101,127-129) ---- */
int drl_env_reset(const drl_env_t* env, float* obs_out /*[N][OP]*/, void* stream);
int drl_env_observe(const drl_env_t* env, float* obs_out /*[N][OP]*/, void* stream);
int drl_env_step(const drl_env_t* env, uint64_t step, const int32_t* actions /*[N]*/, float* obs_out /*[N][OP]*/,
                 float* rew_out /*[N]*/, uint8_t* done_out /*[N]*/, const drl_ep_log_t* log, void* stream);

/* ---- model (ppo.py:49-59) ---- */
/* canonical params -> kernel layout (transposed / lane-permuted copies staged to shared memory by TMA) */
int drl_pack_params(const drl_net_t* net, const float* params, float* packed_out, void* stream);
int drl_policy_forward(const drl_net_t* net, const float* packed, const float* obs /*[n][OP]*/, int64_t n,
                       float* logits_out /*[n][A]*/, float* value_out /*[n]*/, void* stream);
/* Categorical(logits).sample() + log_prob on the Philox stream (counter = env_gid0+i, step) */
int drl_sample(const float* logits /*[n][A]*/, int64_t n, int32_t num_actions, uint64_t seed, uint32_t env_gid0,
               uint64_t step, int32_t* act_out /*[n]*/, float* logp_out /*[n]*/, void* stream);

/* ---- fused rollout, ppo.py:110-141: T x (actor+critic forward, sample, env step, stores) ---- */
#define DRL_ROLLOUT_TENSOR_CORES 1u   /* flags: hidden layers on tcgen05 (bf16 operands, fp32 accumulate), 128 envs per CTA */
int drl_rollout(const drl_env_t* env, const drl_net_t* net, const float* packed, int32_t T, uint64_t step0,
                const drl_rollout_buf_t* buf, const drl_ep_log_t* log, uint32_t flags, void* stream);

/* ---- policy evaluation on fresh episodes: every env plays episodes_per_env = K whole episodes of the frozen policy in one
 * launch (fp32 CUDA cores, hidden = 64 only; drl_evaluate_tc below for hidden = 256).  Env n starts from the reset draw of drl_env_reset (env->seed is the evaluation
 * key, env->state's contents are ignored) and takes steps t = 0, 1, ...: the action is the first index of the largest logit
 * (DRL_EVAL_GREEDY) or drl_rollout's Philox draw with step index t; TimeLimit and auto-reset as drl_env_step(step = t).
 * An env stops after its K-th finished episode, so the log receives exactly N * K entries {step, env, ret, len}; log is
 * required, with cap >= N * K.  On return env->state / elapsed / ep_ret / ep_len hold the final state.
 * trace (nullable, every plane nullable; tests): S = K * max_episode_steps rows; row t of env n holds the state the action of
 * step t was chosen in, its observation, its logits and the action; act is 0xFF in the rows after the env's quota (the other
 * planes are not written there). */
#define DRL_EVAL_GREEDY 1u   /* flags: argmax action instead of the Philox sample */
typedef struct {
    double*  state;    /* [S][N][4] */
    float*   obs;      /* [S][N][OP] */
    float*   logits;   /* [S][N][A] */
    uint8_t* act;      /* [S][N] */
} drl_eval_trace_t;
int drl_evaluate(const drl_env_t* env, const drl_net_t* net, const float* packed, int32_t episodes_per_env, uint32_t flags,
                 const drl_ep_log_t* log, const drl_eval_trace_t* trace /* nullable */, void* stream);
/* The same evaluation -- arguments, validation, streams, log and trace -- on tcgen05 with the numerics of drl_rollout's
 * DRL_ROLLOUT_TENSOR_CORES path (bf16 operands, fp32 accumulation, tanh.approx), for hidden = 256 only: one CTA steps 128
 * envs and leaves when all of them have played their K episodes.  The logits of an observation are bit-identical to those
 * drl_rollout computes for it, so a sampled evaluation replays the training rollout from the same state and keys.
 * hidden = 64 returns DRL_ERR_UNSUPPORTED (use drl_evaluate), any other width DRL_ERR_ARG. */
int drl_evaluate_tc(const drl_env_t* env, const drl_net_t* net, const float* packed, int32_t episodes_per_env, uint32_t flags,
                    const drl_ep_log_t* log, const drl_eval_trace_t* trace /* nullable */, void* stream);

/* ---- graph-replayable variants: same kernels, counters read from *ctrl (device memory) ----
 * drl_ctrl_set computes the Adam scalars of the coming n_steps optimizer steps (same fp64 host arithmetic as drl_clip_adam) and
 * writes the whole block with one kernel launch. */
int drl_ctrl_set(drl_ctrl_t* ctrl, uint64_t env_step, uint32_t epoch_ctr, uint32_t comm_seq, int64_t adam_step, int32_t n_steps,
                 double lr, double beta1, double beta2, void* stream);
int drl_rollout_ctl(const drl_env_t* env, const drl_net_t* net, const float* packed, int32_t T, const drl_ctrl_t* ctrl,
                    const drl_rollout_buf_t* buf, const drl_ep_log_t* log, uint32_t flags, void* stream);
int drl_permutation_ctl(uint32_t* idx_out, uint32_t B, uint64_t seed, const drl_ctrl_t* ctrl, uint32_t epoch_off, uint32_t rank,
                        void* stream);                       /* epoch counter = ctrl->epoch_ctr + epoch_off */
int drl_adv_stats_perm_ctl(const drl_net_t* net, const float* adv, uint32_t B, uint32_t mb_size, uint64_t seed, const drl_ctrl_t* ctrl,
                           uint32_t epoch_off, uint32_t rank, float* stats_out, void* workspace, size_t workspace_bytes, void* stream);

/* ---- GAE + returns, ppo.py:144-151; optionally packs per-sample records for the update ----
 * adv_out/ret_out are [T+1][N] (row T = 0 / val[T], as the reference leaves them).
 * rec_out (nullable) is [T*N][RW]: obs[0..O), then at the last four words logp, adv, val, act(int32 bits). */
int drl_gae(const drl_rollout_buf_t* buf, const drl_net_t* net, int32_t T, int32_t N, float gamma, float gae_lambda,
            float* adv_out, float* ret_out, float* rec_out, void* stream);

/* ---- explained variance diagnostic, ppo.py:194-195: 1 - Var(values - returns) / Var(values) over all n = (T+1)*N slots,
 * unbiased variances like torch.var; NaN when Var(values) == 0.  out [1]; fp64 accumulation, fixed-order fold. ---- */
int drl_explained_variance(const float* values, const float* returns, int64_t n, float* out, void* workspace,
                           size_t workspace_bytes, void* stream);

/* ---- minibatch permutation, ppo.py:155 ---- */
int drl_permutation(uint32_t* idx_out /*[B]*/, uint32_t B, uint64_t seed, uint32_t epoch_ctr, uint32_t rank, void* stream);

/* ---- per-minibatch advantage statistics (mean, unbiased std), ppo.py:169 ----
 * stats_out [num_minibatches][2] float; minibatch k covers idx[k*mb_size, min(B,(k+1)*mb_size)). idx NULL = identity. */
int drl_adv_stats(const drl_net_t* net, const float* rec, const uint32_t* idx, uint32_t B, uint32_t mb_size,
                  float* stats_out, void* workspace, size_t workspace_bytes, void* stream);

/* ---- loss + backward of one minibatch, ppo.py:159-187 + backward of ppo.py:190 ----
 * grad_out [P] canonical layout, mean over the mb_count samples; loss_terms_out[8] =
 * {loss, pg_loss, v_loss, entropy, approx_kl, clipfrac, 0, 0}. */
/* Same statistics for the keyed permutation of drl_permutation(seed, epoch_ctr, rank) WITHOUT a gather: adv is the
 * advantage plane in natural sample order [B]; each sample's minibatch is found by inverting the permutation.
 * At most 8 minibatches (DRL_ERR_UNSUPPORTED otherwise: use drl_adv_stats). */
int drl_adv_stats_perm(const drl_net_t* net, const float* adv, uint32_t B, uint32_t mb_size, uint64_t seed, uint32_t epoch_ctr,
                       uint32_t rank, float* stats_out, void* workspace, size_t workspace_bytes, void* stream);

#define DRL_GRAD_TENSOR_CORES 1u   /* flags: tcgen05 path (bf16 operands, fp32 accumulate) instead of FP32 CUDA cores */
int drl_ppo_minibatch_grad(const drl_net_t* net, const float* packed, const float* rec, const uint32_t* idx,
                           uint32_t mb_start, uint32_t mb_count, const float* adv_stats /*[2] mean,std*/,
                           const drl_ppo_coef_t* coef, float* grad_out, float* loss_terms_out,
                           void* workspace, size_t workspace_bytes, uint32_t flags, void* stream);

/* ---- peer-memory communicator for the fused multi-GPU minibatch step (one node, NVLink / NVSwitch) ----
 * Each rank owns one symmetric buffer (drl_comm_bytes() bytes, allocated by drl_comm_alloc -- the one place the
 * library allocates, because the memory must be exportable with cudaIpcGetMemHandle) and maps every peer's buffer
 * with drl_comm_open.  The buffer holds two generations of the rank's folded gradient and arrival flags. */
#define DRL_MAX_RANKS 8
typedef struct {
    int32_t  world, rank;
    void*    peer[DRL_MAX_RANKS];   /* peer[r] = rank r's symmetric buffer as mapped in THIS process (peer[rank] = own) */
    uint32_t seq;                   /* 1-based sequence number of this minibatch step, identical on all ranks */
    int32_t* error_flag;            /* [1] device int, set to 1 if a peer did not arrive within the timeout */
} drl_comm_t;
size_t drl_comm_bytes(const drl_net_t* net);
int drl_comm_alloc(size_t bytes, void** dev_ptr_out, void* ipc_handle_out /* 64 bytes */);
int drl_comm_open(const void* ipc_handle /* 64 bytes */, void** peer_ptr_out);
int drl_comm_close(void* peer_ptr);
int drl_comm_free(void* dev_ptr);

/* ---- single-GPU fusion of the three calls above/below: minibatch gradient, then ONE cooperative kernel that folds
 * the per-CTA partial gradients, clips by the global norm and applies Adam (ppo.py:159-192 in two launches; ONE launch on the
 * tensor-core path).  `packed` is read by the gradient kernels and refreshed by the Adam step; grad_out receives the pre-clip gradient.
 * num_steps (1..8; > 1 on the tensor-core path only): the launch runs that many CONSECUTIVE, equally sized minibatches -- minibatch s
 * covers idx[mb_start + s * mb_count, +mb_count), normalises with adv_stats[2s], [2s+1], writes loss_terms_out[8s..8s+8) and applies
 * optimizer step `step + s` -- i.e. a whole epoch of ppo.py:156-192 without leaving the kernel (the weight tiles are reloaded and the
 * record gather of the next minibatch runs ahead while the fold / clip / Adam tail of the current one finishes). */
int drl_ppo_minibatch_update(const drl_net_t* net, float* packed, const float* rec, const uint32_t* idx, uint32_t mb_start,
                             uint32_t mb_count, const float* adv_stats, const drl_ppo_coef_t* coef, float* params, float* grad_out,
                             float* exp_avg, float* exp_avg_sq, int64_t step, double lr, double beta1, double beta2, double eps,
                             double max_grad_norm, float* loss_terms_out, float* norm_out, void* workspace, size_t workspace_bytes,
                             uint32_t flags, int32_t num_steps, void* stream);
/* Multi-GPU form (tensor-core path only): the same single cooperative launch; between the local fold and the clip the
 * CTAs publish their gradient slices in the symmetric buffer, wait for every peer's arrival flag and sum the peers'
 * slices over NVLink in rank order (a one-shot all-reduce inside the kernel, identical result on every rank), then
 * clip and apply Adam on gradient / world.  grad_out receives the summed gradient. */
int drl_ppo_minibatch_update_dist(const drl_net_t* net, float* packed, const float* rec, const uint32_t* idx, uint32_t mb_start,
                                  uint32_t mb_count, const float* adv_stats, const drl_ppo_coef_t* coef, float* params,
                                  float* grad_out, float* exp_avg, float* exp_avg_sq, int64_t step, double lr, double beta1,
                                  double beta2, double eps, double max_grad_norm, float* loss_terms_out, float* norm_out,
                                  void* workspace, size_t workspace_bytes, uint32_t flags, const drl_comm_t* comm, int32_t num_steps,
                                  void* stream);

/* Graph-replayable form of the two calls above (tensor-core path): `ordinal` = index of this optimizer step inside the update
 * (Adam scalars ctrl->neg_step_size[ordinal], ctrl->bc2_sqrt[ordinal]; sequence number ctrl->comm_seq + ordinal + 1);
 * comm NULL = single GPU, otherwise its `seq` field is ignored. */
int drl_ppo_minibatch_update_ctl(const drl_net_t* net, float* packed, const float* rec, const uint32_t* idx, uint32_t mb_start,
                                 uint32_t mb_count, const float* adv_stats, const drl_ppo_coef_t* coef, float* params,
                                 float* grad_out, float* exp_avg, float* exp_avg_sq, const drl_ctrl_t* ctrl, int32_t ordinal,
                                 double beta1, double beta2, double eps, double max_grad_norm, float* loss_terms_out,
                                 float* norm_out, void* workspace, size_t workspace_bytes, uint32_t flags, const drl_comm_t* comm,
                                 int32_t num_steps, void* stream);

/* ---- clip_grad_norm_ + Adam, ppo.py:191-192 (after the gradient all-reduce) ----
 * grad is multiplied by grad_scale (1/world) first; `step` is the 1-based Adam step of this call.
 * packed_out (nullable) receives the refreshed kernel layout; norm_out (nullable, [1]) the pre-clip norm. */
int drl_clip_adam(const drl_net_t* net, float* params, const float* grad, float* exp_avg, float* exp_avg_sq,
                  int64_t step, double lr, double beta1, double beta2, double eps, double max_grad_norm,
                  double grad_scale, float* packed_out, float* norm_out, void* stream);

/* ---- replay-buffer sampling and gather (SURVEY.md 8f-4): the random-index gather family of the off-policy scripts ----
 * Storage is flat struct-of-arrays with the reference's one-slot shift (dqn.py:74-77,104-109): obs [cap+1][OP] (padded rows),
 * act [cap+1] int32, rew [cap+1], term [cap+1] u8; transition i = (obs[i], act[i], rew[i+1], term[i+1], obs[i+1]).
 * Index draws use the build's Philox stream (word 0 of philox(i, draw_ctr, TAG_REPLAY)), not numpy's / torch's MT19937. */
/* batch_inds = np.random.randint(size, size=batch)                                           dqn.py:116 */
int drl_replay_sample_uniform(uint32_t* idx_out, uint32_t batch, uint32_t size, uint64_t seed, uint64_t draw_ctr, void* stream);
/* b_observations, b_actions, b_next_observations, b_rewards, b_terminated of one batch      dqn.py:118-122, per.py:131-135 */
int drl_replay_gather(const float* obs, const int32_t* act, const float* rew, const uint8_t* term, const uint32_t* idx, uint32_t batch,
                      int32_t obs_stride, float* b_obs, float* b_next_obs, int32_t* b_act, float* b_rew, uint8_t* b_term, void* stream);
/* batch_inds = torch.multinomial(priorities, batch, replacement=True) and b_probabilities = p^alpha / sum(p^alpha) at those
 * indices (prob_out nullable)                                                                per.py:127-131 */
size_t drl_replay_scratch_bytes(uint32_t size);
int drl_replay_sample_priority(const float* priorities, uint32_t size, float alpha, uint32_t batch, uint64_t seed, uint64_t draw_ctr,
                               uint32_t* idx_out, float* prob_out, void* scratch, size_t scratch_bytes, void* stream);
/* priorities[batch_inds] = |td_errors| (last duplicate wins); max_priority = max(max_priority, written values)   per.py:144-146 */
int drl_replay_update_priorities(float* priorities, const uint32_t* idx, const float* td_errors, uint32_t batch, float* max_priority_inout,
                                 void* stream);

/* ---- REINFORCE on the device-resident CartPole (SURVEY.md 8f-2; deep_rl/reinforce.py:38-77) ----
 * Policy = Sequential(Linear(4,128), Dropout(0.6), ReLU, Linear(128,2), Softmax); params flat in state_dict order
 * (0.weight [128][4], 0.bias [128], 3.weight [2][128], 3.bias [2]) = drl_reinforce_param_count() floats.
 * drl_reinforce_episodes: every env runs ONE episode (reset, then act / step until done, at most T = max_episode_steps
 * steps; reinforce.py:55-67).  Planes [T+1][N] with the one-slot shift of the PPO buffers (rew[t+1], done[t+1] belong to
 * act[t]); slots after the end of an episode hold reward 0 / done 1.  step0 >= 1 is the global step index of the first step
 * (Philox counter); mask_bits_out (nullable, [T][N][4] words) receives the dropout keep mask of every step.
 * Returns (reinforce.py:67) = drl_gae on these planes with gae_lambda = 1 and an all-zero value plane.
 * drl_reinforce_grad: per-episode policy_loss = sum(-log_prob * (R - mean) / (std + exp(-5))) (reinforce.py:71-74) and its
 * closed-form gradient, summed over the N episodes and multiplied by grad_scale; mask_bits NULL = regenerate the Philox dropout
 * masks of (seed, env_gid0 + n, step0 + t), else use the given ones (teacher forcing).  Scratch: grad_part [N][(P + 3) / 4 * 4], loss_part [N].
 * drl_adam_step: torch.optim.Adam on a flat vector (reinforce.py:45,77; no clipping), `step` 1-based. */
int drl_reinforce_param_count(void);
int drl_reinforce_episodes(const drl_env_t* env, const float* params, int32_t T, uint64_t step0, float* obs /*[T+1][N][4]*/,
                           uint8_t* act, float* rew, uint8_t* done, int32_t* ep_len /*[N]*/, uint32_t* mask_bits_out,
                           const drl_ep_log_t* log, void* stream);
int drl_reinforce_grad(const float* params, const float* obs, const uint8_t* act, const float* returns, const int32_t* ep_len,
                       const uint32_t* mask_bits, int32_t N, uint64_t seed, uint32_t env_gid0, uint64_t step0, float grad_scale,
                       float* grad_out, float* loss_out, float* grad_part, float* loss_part, void* stream);
int drl_adam_step(float* params, const float* grad, float* exp_avg, float* exp_avg_sq, int64_t n, int64_t step, double lr, double beta1,
                  double beta2, double eps, void* stream);

/* ---- diagnostics: runs one tcgen05.mma operand-layout combination of the update kernel on caller matrices
 * (fp32 row-major in, fp32 row-major out; operands are rounded to bf16).  See csrc/umma_selftest.cu. ---- */
int drl_selftest_umma(int32_t mode, int32_t variant, const float* a, const float* b, float* d_out, void* stream);
/* y[i] = tanh.approx.f32(x[i]) -- the SFU instruction the tensor-core kernels use for their activations; lets the
 * bf16-emulating oracle (oracle/ppo_oracle.py) reproduce the kernels' activations bit for bit. */
int drl_selftest_tanh(const float* x, float* y, int64_t n, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* DRL_B200_H */
