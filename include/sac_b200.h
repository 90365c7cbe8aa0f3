/*
 * sac_b200.h -- C-ABI of the stable-baselines3 SAC actor forward (same library, libquadx_b200.so).
 * It replaces, for playing back a policy the reference trained with SAC (train_hover.py:47-58 builds
 * SAC("MlpPolicy", policy_kwargs=dict(net_arch=[128, 128]))), the call test_hover.py:7-27 reaches through
 * `model.predict(obs, deterministic=True)` (SB3 2.7.0, un-vendored, see SURVEY.md 8a row X4):
 *   VecNormalize.normalize_obs (training=False) + SACPolicy.actor(obs, deterministic=True) -> sac_actor_forward
 * Stochastic sampling (the log_std head), gSDE and activations other than ReLU are not provided.
 * All pointers are device pointers on the current device; work is enqueued on `stream` (cudaStream_t as void*);
 * return 0 / negative QX_E* like quadx_b200.h.
 */
#ifndef SAC_B200_H
#define SAC_B200_H
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

#define SAC_HIDDEN 128   /* hidden tile width: net_arch=[128, 128] (train_hover.py:57); narrower layers run zero-padded */
#define SAC_IN_PAD 32    /* observation columns padded to the MMA K granularity: obs_dim <= 32 */
#define SAC_HEAD_PAD 16  /* action columns padded to the MMA N granularity: act_dim <= 4 */

/* SB3 `Actor` (actor.latent_pi.0 / .2, actor.mu), bf16 weights in PyTorch Linear layout [out][in], 16-byte aligned,
 * entries beyond a layer's real width zero:
 *   w1 [128][32]  latent_pi.0   w2 [128][128]  latent_pi.2   w_mu [16][128]  mu (rows 0 .. act_dim-1)
 *   b1 [128], b2 [128], b_mu [16]  fp32 */
typedef struct SacActor {
  const void* w1;
  const void* w2;
  const void* w_mu;
  const float* b1;
  const float* b2;
  const float* b_mu;
  int32_t obs_dim;
  int32_t act_dim;
} SacActor;

/* SACPolicy.predict(obs, deterministic=True) for n rows (replaces SB3 Actor.forward + SquashedDiagGaussian mode):
 *   x = clip((obs - mean) * inv_std, +-obs_clip)   when obs_mean != NULL (VecNormalize.normalize_obs; obs_clip <= 0: no clip)
 *   a = tanh(W_mu relu(W2 relu(W1 x + b1) + b2) + b_mu)
 * on the tensor cores (tcgen05, bf16 x bf16 -> fp32; x and the hidden activations are rounded to bf16), the final tanh
 * evaluated in fp64 and rounded to fp32 (not tanh.approx).  obs rows are obs_stride floats apart.  Writes actions [n, act_dim] (required; in [-1, 1], the
 * action box of both tasks, so it is also what the env receives) and obs_norm_out [n, obs_dim] (nullable: the normalised
 * observation the actor saw).  obs_mean / obs_inv_std are both given or both NULL.
 * No allocation, no synchronisation, capturable in a CUDA graph.  A null or misaligned pointer (weights 16 bytes, fp32
 * buffers 4 bytes) or a bad size returns QX_EINVAL and launches nothing. */
int sac_actor_forward(const SacActor* actor, const float* obs, int64_t obs_stride, int64_t n, const float* obs_mean,
                      const float* obs_inv_std, float obs_clip, float* actions, float* obs_norm_out, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* SAC_B200_H */
