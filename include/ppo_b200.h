/*
 * ppo_b200.h -- C-ABI of the on-device PPO rollout kernels (same library,
 * libquadx_b200.so).  These replace, for the rollout half of PPO, the
 * stable-baselines3 2.7.0 calls the reference's training script reaches
 * through `model.learn` (train_hover.py:47-60; SB3 is un-vendored, see
 * SURVEY.md 8a row X4):
 *   ActorCriticPolicy.forward            -> ppo_policy_forward
 *   RolloutBuffer.compute_returns_and_advantage -> ppo_gae
 *   VecNormalize (running obs / return statistics) -> ppo_obs_stats_update, ppo_reward_normalize
 * All pointers are device pointers on the current device; work is enqueued on
 * `stream` (cudaStream_t as void*); return 0 / negative QX_E* like quadx_b200.h.
 */
#ifndef PPO_B200_H
#define PPO_B200_H
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

#define PPO_HIDDEN 128   /* policy_kwargs=dict(net_arch=[128, 128]), train_hover.py:57 */
#define PPO_IN_PAD 32    /* observation columns padded to the MMA K granularity */
#define PPO_HEAD_PAD 16  /* action-mean columns + value column, padded to the MMA N granularity */

/* Weights of the separate tanh MLPs pi / vf (SB3 MlpPolicy), bf16, PyTorch Linear layout [out][in]:
 *   w1   [2*128][32]   rows 0..127 pi layer 1, rows 128..255 vf layer 1, input columns >= obs_dim are zero
 *   w2p  [128][128], w2v [128][128]
 *   w3   [16][256]     rows 0..act_dim-1: action_net over the pi half (cols 0..127),
 *                      row act_dim: value_net over the vf half (cols 128..255), other entries zero
 *   b1 [256], b2 [256] (pi | vf), b3 [16]  fp32;  log_std [act_dim] fp32 */
typedef struct PpoPolicy {
  const void* w1;
  const void* w2p;
  const void* w2v;
  const void* w3;
  const float* b1;
  const float* b2;
  const float* b3;
  const float* log_std;
  int32_t obs_dim;
  int32_t act_dim;
} PpoPolicy;

/* ActorCriticPolicy.forward for n rows: normalise obs with (mean, inv_std, clip) when obs_mean != NULL
 * (VecNormalize.normalize_obs), run both MLPs on the tensor cores (tcgen05, bf16 x bf16 -> fp32),
 * sample a ~ N(mean, exp(log_std)) with Philox key (seed, row0 + row) and counter step + *step_base_dev
 * (step_base_dev may be NULL; deterministic != 0: a = mean), and write
 *   actions [n, act_dim] (unclipped, what PPO stores), env_actions [n, act_dim] (clipped to [-1, 1],
 *   what the env receives), values [n], log_probs [n], obs_norm_out [n, obs_dim] (the normalised
 *   observation the policy saw, what PPO stores).  Any output may be NULL. */
int ppo_policy_forward(const PpoPolicy* p, const float* obs, int64_t obs_stride, int64_t n, const float* obs_mean,
                       const float* obs_inv_std, float obs_clip, uint64_t seed, uint64_t row0, uint64_t step,
                       const uint64_t* step_base_dev, int32_t deterministic, float* actions, float* env_actions, float* values,
                       float* log_probs, float* obs_norm_out, void* stream);

/* VecNormalize.step_wait + ActorCriticPolicy.forward in ONE launch (the rollout's per-step pair `obs_rms.update(obs)` then
 * `normalize_obs(obs)`, SB3 vec_normalize.py [RECALL], reached from model.learn, train_hover.py:60): the launch first merges the
 * n raw rows of obs into the running statistics obs_stats = {mean[obs_dim], var[obs_dim], count} (fp64, as
 * ppo_running_stats_update does), writes the refreshed fp32 obs_mean / obs_inv_std = 1 / sqrt(var + eps), and then runs
 * ppo_policy_forward with them.  stats_scratch: ppo_running_stats_scratch_bytes bytes, zeroed once, private to this stream.
 * fused != 0: the launch waits inside the kernel for its own last CTA (grid <= SM count, one CTA per SM: all resident together); do
 * not run two of these on one device at the same time from different streams.
 * fused == 0: ppo_running_stats_update followed by ppo_policy_forward as its programmatic dependent launch -- the policy kernel
 * is scheduled as the statistics blocks leave the SMs, stages its weights while the last block merges, and waits on the device
 * (griddepcontrol.wait) before it reads the statistics; same results as the two separate calls, what the rollout uses. */
int ppo_policy_forward_stats(const PpoPolicy* p, const float* obs, int64_t obs_stride, int64_t n, double* obs_stats, float eps,
                             void* stats_scratch, float* obs_mean, float* obs_inv_std, float obs_clip, uint64_t seed, uint64_t row0,
                             uint64_t step, const uint64_t* step_base_dev, int32_t deterministic, float* actions, float* env_actions,
                             float* values, float* log_probs, float* obs_norm_out, int32_t fused, void* stream);

/* SB3 collect_rollouts time-limit bootstrap: for the envs listed in the done queue of the step just taken
 * (qx_done_queue) that were truncated but not terminated, reward += gamma * V(terminal_obs). */
int ppo_bootstrap_truncated(const PpoPolicy* p, const float* terminal_obs, int64_t obs_stride, int64_t n, const float* obs_mean,
                            const float* obs_inv_std, float obs_clip, const uint32_t* done_count_dev, const uint32_t* done_idx_dev,
                            const uint8_t* terminated, const uint8_t* truncated, float gamma, float* reward_inout, void* stream);

/* The same two operations in the other order, for a rollout whose side branch must not wait for a free SM late (DESIGN.md, K2):
 * ppo_bootstrap_truncated_first STORES gamma * V(terminal_obs) into reward_out[row] for the truncated, not terminated envs of
 * the done queue; ppo_reward_normalize_add (below) then writes clip(r / sigma) + that value for exactly those rows and
 * clip(r / sigma) for all others.  Result = ppo_reward_normalize followed by ppo_bootstrap_truncated up to one rounding. */
int ppo_bootstrap_truncated_first(const PpoPolicy* p, const float* terminal_obs, int64_t obs_stride, int64_t n, const float* obs_mean,
                                  const float* obs_inv_std, float obs_clip, const uint32_t* done_count_dev, const uint32_t* done_idx_dev,
                                  const uint8_t* terminated, const uint8_t* truncated, float gamma, float* reward_out, void* stream);

/* RolloutBuffer.compute_returns_and_advantage: rewards, values, dones [T, n] (dones[t] = episode ended AT step t),
 * last_values [n]; writes advantages, returns [T, n]. */
int ppo_gae(const float* rewards, const float* values, const uint8_t* dones, const float* last_values, int32_t T, int64_t n,
            float gamma, float lam, float* advantages, float* returns, void* stream);

/* VecNormalize running statistics: merge the batch moments of x [n, dim] (row stride `stride`) into
 * stats = {mean[dim], var[dim], count} (fp64, device) with the parallel-Welford update, then refresh
 * mean_f32[dim] / inv_std_f32[dim] = 1/sqrt(var + eps).  One launch (the last block to finish does the merge).
 * `scratch`: ppo_running_stats_scratch_bytes(dim) bytes of device memory, ZERO-FILLED once before the first call and
 * owned by one stats object (it holds the per-block sums and the launch ticket); calls sharing a scratch buffer must be
 * stream-ordered. */
int ppo_running_stats_update(const float* x, int64_t stride, int64_t n, int32_t dim, double* stats, float eps, float* mean_f32,
                             float* inv_std_f32, void* scratch, void* stream);
int64_t ppo_running_stats_scratch_bytes(int32_t dim);

/* VecNormalize reward path: ret = ret * gamma + r; stats over ret (dim 1); r_norm = clip(r / sqrt(var + eps), +-clip);
 * ret = 0 where done; done_out [n] (nullable) = terminated | truncated.  `returns_acc` [n] is the per-env discounted return accumulator. */
int ppo_reward_normalize(const float* reward, const uint8_t* terminated, const uint8_t* truncated, float* returns_acc, int64_t n,
                         float gamma, float clip, float eps, double* ret_stats, float* reward_out, uint8_t* done_out, void* scratch, void* stream);
int ppo_reward_normalize_add(const float* reward, const uint8_t* terminated, const uint8_t* truncated, float* returns_acc, int64_t n,
                             float gamma, float clip, float eps, double* ret_stats, float* reward_out, uint8_t* done_out, void* scratch,
                             void* stream);

/* ---- the PPO update (SB3 PPO.train, reached by train_hover.py:60 `model.learn`) --------------------------------------
 * Flat fp32 parameter vector, in the module order of SB3's ActorCriticPolicy(net_arch=[128,128]) with separate pi / vf
 * MLPs:  pi1.W [128][obs_dim], pi1.b, pi2.W [128][128], pi2.b, action_net.W [act_dim][128], action_net.b,
 *        vf1.W, vf1.b, vf2.W, vf2.b, value_net.W [1][128], value_net.b, log_std [act_dim]
 * (39 049 floats for the hover task).  The gradient and the Adam moments use the same layout. */
int32_t ppo_update_num_params(int32_t obs_dim, int32_t act_dim);
/* device workspace one updater needs: ZERO-FILLED once before the first call; holds the minibatch statistics, the Adam
 * step counter and one partial gradient per SM */
int64_t ppo_update_workspace_bytes(int32_t obs_dim, int32_t act_dim);

/* Gradient of SB3's PPO loss on one minibatch (forward + loss + backward of both networks on the tensor cores):
 *   loss = mean(max(-A r, -A clip(r, 1 - clip_range, 1 + clip_range))) + vf_coef * mean((ret - V)^2) - ent_coef * mean(entropy)
 * with r = exp(logp - old_logp) and, when normalize_adv != 0, A = (adv - mean) / (std + 1e-8) over the minibatch.
 * The minibatch is the set of 128-row tiles tiles_dev[0 .. n_tiles) of the rollout buffers (rows 128 t .. 128 t + 127; rows
 * >= n_rows do not count): obs [n_rows, obs_dim] (normalised, as stored by ppo_policy_forward), actions [n_rows, act_dim],
 * old_logp / adv / ret [n_rows].  `p` holds the bf16 weights the forward runs with.  Writes grad_out [n_params] (mean over the
 * minibatch rows) and adds to loss_stats[0..5] (nullable) the SUMS over rows of: policy loss, squared value error,
 * old_logp - logp, clipped indicator, (r - 1) - log r, 1.  Four launches on `stream`, no host synchronisation. */
int ppo_update_minibatch(const PpoPolicy* p, const float* obs, const float* actions, const float* old_logp, const float* adv,
                         const float* ret, const int32_t* tiles_dev, int32_t n_tiles, int64_t n_rows, float clip_range, float vf_coef,
                         float ent_coef, int32_t normalize_adv, float* grad_out, float* loss_stats, void* workspace, void* stream);
/* after an all-reduce of grad over the ranks: recompute the squared norm (of grad * grad_scale) the clip in ppo_update_adam uses */
int ppo_update_grad_norm(const float* grad, int32_t n_params, float grad_scale, void* workspace, void* stream);
/* torch.nn.utils.clip_grad_norm_(max_grad_norm) + torch.optim.Adam step (bias-corrected, eps outside the square root) on the
 * flat fp32 master parameters, with g = grad * grad_scale; then the updated values are re-packed (bf16 weights, fp32 biases /
 * log_std) into the buffers of `packed_out`, which the forward kernels read.  The Adam step counter lives in the workspace. */
int ppo_update_adam(float* params, const float* grad, float* exp_avg, float* exp_avg_sq, int32_t n_params, float lr, float beta1,
                    float beta2, float eps, float max_grad_norm, float grad_scale, const PpoPolicy* packed_out, void* workspace, void* stream);
/* learning-rate schedule (SB3 `learning_rate` as a callable of the remaining progress): subsequent ppo_update_adam calls --
 * captured in a CUDA graph or not -- step with lr * scale.  The factor lives in the workspace; a fresh workspace means 1. */
int ppo_update_set_lr_scale(void* workspace, float scale, void* stream);
/* log pi(a | s) of every row of the given 128-row tiles, by the forward arithmetic of ppo_update_minibatch (actor only, nothing
 * else is touched): the counterpart of SB3's policy.evaluate_actions on a stored rollout.  Overwriting old_logp with it makes
 * the ratio of a following minibatch pass exactly 1 at unchanged weights (tests/test_gpu_update.py).  Measured: the rollout's
 * policy kernel and this pass -- the same bf16 network through different tile schedules -- agree to 4e-6 in log pi even at
 * sigma = e^-6 (approx-KL < 1e-9), so the trainer does not need it (PPOConfig.recompute_old_logp = False); it is there for
 * rollouts whose log-probs came from somewhere else (an imported SB3 policy, a replayed buffer). */
int ppo_update_recompute_logp(const PpoPolicy* p, const float* obs, const float* actions, const int32_t* tiles_dev, int32_t n_tiles,
                              int64_t n_rows, float* logp_out, void* workspace, void* stream);
/* SB3's `target_kl` early stop (PPO.train: the epoch loop ends at the first minibatch whose approx_kl exceeds 1.5 x target_kl,
 * before that minibatch's optimiser step), taken on the device so that it works per minibatch inside a captured epoch.
 * While target_kl > 0 is armed: ppo_update_minibatch appends this minibatch's sum of (ratio - 1) - log ratio and its row count to
 * the gradient -- grad_out must then hold ppo_update_num_params() + 2 floats, and a gradient all-reduce must cover them, so
 * every rank decides alike -- and ppo_update_adam turns into a no-op (no parameter / moment / step-count change) from the first
 * minibatch over the threshold until the next re-arm.  target_kl >= 0 (re-)arms with that threshold (0 = off) and clears the
 * latch; target_kl < 0 only reads.  stopped_out / skipped_out (nullable) return the latch and the number of skipped steps as
 * they were BEFORE the re-arm. */
int ppo_update_kl_stop(void* workspace, float target_kl, int32_t* stopped_out, int32_t* skipped_out, void* stream);
/* optional lower bound of log_std applied by ppo_update_adam (on != 0): keeps the exploration noise from collapsing */
int ppo_update_set_log_std_floor(void* workspace, int32_t on, float floor, void* stream);
/* read (out != NULL) and / or set (set_to >= 0) the Adam step counter: checkpoint / resume */
int ppo_update_step_count(void* workspace, int64_t set_to, int64_t* out, void* stream);

/* test hook: D[128, n] (fp32) = A x B^T through K-major (x_mn = 0: given as [rows][k]) or MN-major (x_mn = 1: given as
 * [k][rows]) shared-memory descriptors -- the transposed operand forms the backward GEMMs rely on */
int ppo_test_gemm_mn(const void* a_bf16, const void* b_bf16, float* d, int32_t n, int32_t k, int32_t a_mn, int32_t b_mn, void* stream);

/* test hook: D[128, n] (fp32) = A[128, k] x B[n, k]^T with one tcgen05.mma chain (bf16 inputs) */
int ppo_test_gemm(const void* a_bf16, const void* b_bf16, float* d, int32_t n, int32_t k, void* stream);

/* test hook: the policy forward's hidden activation, bf16(tanh(x)) for x[0 .. n), applied pairwise (x[2i] as the low half,
 * x[2i + 1] as the high half) through the same device function as the kernel's epilogue -- what a reference of the forward
 * cannot compute itself is the rounding of tanh.approx */
int ppo_test_tanh_bf16(const float* x, uint16_t* out_bf16, int64_t n, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* PPO_B200_H */
