/* C ABI of the PPO update of libvnl_b200.so (SURVEY section 8 row f2).
 *
 * Replaces what one `minibatch_step` of the reference runs on the device (ppo_imitation/train.py:251-268):
 *     jax.value_and_grad(compute_ppo_intention_loss)  (ppo_imitation/intention_losses.py:91-202)
 *       over IntentionNetwork (ppo_imitation/intention_policy_network.py:20-105: Dense / relu / LayerNorm, reparameterize),
 *       the brax value MLP (ppo_networks.py:114-118 -> brax networks.make_value_network: Dense 1024-1024-1, swish),
 *       brax NormalTanhDistribution log_prob / entropy, compute_gae (-> vnl_gae, include/vnl_ppo.h);
 *     gradients.gradient_update_fn: lax.pmean of the gradients over devices (the caller's NCCL all-reduce of the flat
 *       gradient buffer) and optax.adam (vnl_adam).
 * The dense contractions run on the tensor cores (vnl_gemm_tf32: tcgen05 kind::tf32 + TMA tensor maps); everything else
 * is elementwise / row-wise fp32.  All pointers are caller-owned DEVICE memory, row-major fp32 unless said otherwise;
 * `ld*` = row stride in floats.  Calls only enqueue on `stream`; no allocation, no sync; CUDA-graph capturable.
 * Return 0 = ok, negative = argument error, positive = cudaError_t.
 */
#ifndef VNL_TRAIN_H_
#define VNL_TRAIN_H_
#include <stddef.h>
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

/* C[M, N] (+)= sum_{p < npairs} A_p[M, K] . B_p[N, K]^T (+ bias[N]).
 * a_mn_major = 0: A_p is memory [M][K] (lda between rows); 1: memory [K][M].  Same for B with N.  Pointers 16-byte aligned,
 * lda / ldb multiples of 4.  npairs = 1: plain TF32 (what XLA runs for f32 dots on NVIDIA GPUs by default); npairs = 3 with
 * (hi, hi), (hi, lo), (lo, hi) from vnl_split_tf32: fp32-class accuracy (3xTF32).  splitk > 1: the K range is cut into
 * that many slices whose partial tiles are ADDED to C with red.global.add -- the caller zeroes C first. */
int vnl_gemm_tf32(int M, int N, int K, int npairs, const float* const* A, int lda, int a_mn_major, const float* const* B, int ldb,
                  int b_mn_major, float* C, int ldc, const float* bias, int splitk, void* stream);
/* The same product with a fused activation epilogue for the swish layers of the value MLP (splitk <= 1, N a multiple of 32,
 * ldc / ldaux multiples of 4, C / aux 16-byte aligned; else -5):
 *   epilogue 1: C = pre-activation as above, aux[M, N] = swish(C)            (forward: vnl_swish_fwd without its pass over HBM)
 *   epilogue 2: C = (A . B^T) * swish'(aux[M, N]), aux = the pre-activation  (dgrad + vnl_swish_bwd in one) */
int vnl_gemm_tf32_ex(int M, int N, int K, int npairs, const float* const* A, int lda, int a_mn_major, const float* const* B, int ldb,
                     int b_mn_major, float* C, int ldc, const float* bias, int splitk, int epilogue, float* aux, int ldaux, void* stream);

/* x = hi + lo with hi = x truncated to tf32 (low 13 mantissa bits cleared), lo = x - hi (exact in fp32). */
int vnl_split_tf32(const float* x, size_t n, float* hi, float* lo, void* stream);

/* Minibatch gather out of the time-major transition buffers of the rollout: dst[(t * Bm + j) * ld_dst + c] =
 * src[(t * B + idx[j]) * width + c], columns [width, ld_dst) zero-filled (pads 795 -> 796 so that rows are 16-byte
 * multiples for TMA).  `convert_data` of ppo_imitation/train.py:279-283 (permutation + reshape) as an index list. */
int vnl_gather_rows(const float* src, int T, int B, int width, const int32_t* idx, int Bm, float* dst, int ld_dst, void* stream);

/* out[r, c] = (obs[r, c] - mean[c]) / std[c]   (brax running_statistics.normalize; ppo_imitation/train.py:220-229) */
int vnl_obs_normalize(const float* obs, int ld_obs, int rows, int width, const float* mean, const float* std, float* out, int ld_out,
                      void* stream);

/* h = LayerNorm(relu(pre)) (intention_policy_network.py:36-40, 64-68; flax LayerNorm: eps 1e-6, fast variance).
 * stats [rows, 2] = (mean, rstd) of relu(pre), kept for the backward pass.  n <= 1024 (one warp per row, 32 values per lane). */
int vnl_relu_ln_fwd(const float* pre, int ld_pre, int rows, int n, const float* scale, const float* bias, float* out, int ld_out,
                    float* stats, void* stream);
/* dpre from dy; dscale / dbias [n] are ACCUMULATED (caller zeroes).  dbias_pre (may be NULL) [n] += column sums of dpre = the bias
 * gradient of the dense layer in front of the relu, so that it needs no pass of its own.  n <= 256 (the per-column partials of a
 * warp live in registers: 8 per lane); ld_dy, ld_pre, ld_dpre >= n. */
int vnl_relu_ln_bwd(const float* dy, int ld_dy, const float* pre, int ld_pre, const float* stats, const float* scale, int rows, int n,
                    float* dpre, int ld_dpre, float* dscale, float* dbias, float* dbias_pre, void* stream);

/* swish / silu of the brax value MLP (linen.swish), elementwise over n values. */
int vnl_swish_fwd(const float* pre, size_t n, float* out, void* stream);
int vnl_swish_bwd(const float* dy, const float* pre, size_t n, float* dpre, void* stream);

/* reparameterize (intention_policy_network.py:76-79): z = mean + eps * exp(0.5 logvar), heads = [mean | logvar] [rows, 2L];
 * z is written to dec_in[:, 0:L] (the decoder input [z | normalised obs]). */
int vnl_reparam_fwd(const float* heads, const float* eps, int rows, int L, float* dec_in, int ld, void* stream);
/* dheads = [dz + kl_coef * mean | dz * 0.5 eps exp(0.5 logvar) - 0.5 kl_coef (1 - exp(logvar))] with dz = ddec_in[:, 0:L];
 * kl_coef = kl_weight / (rows * L) (kl_divergence, intention_losses.py:21-23).  Adds the KL loss value to *kl_loss. */
int vnl_heads_bwd(const float* ddec_in, int ld, const float* heads, const float* eps, int rows, int L, float kl_coef, float* dheads,
                  float* kl_loss, void* stream);

/* out[c] += sum_r w[r] * x[r, c]  (w = NULL: plain column sums: the bias gradients; with w: the value head's weight gradient) */
int vnl_colsum(const float* x, int ld, int rows, int n, const float* w, float* out, void* stream);
/* out[r] = sum_c h[r, c] * w[c] + b[0]   (value head forward: Dense(1) + squeeze) */
int vnl_rowdot(const float* h, int ld, int rows, int n, const float* w, const float* b, float* out, void* stream);
/* dh[r, c] = dv[r] * w[c]   (value head backward) */
int vnl_outer(const float* dv, int rows, const float* w, int n, float* dh, int ld, void* stream);
/* dpre[r, c] = dv[r] * w[c] * swish'(pre[r, c]): vnl_outer followed by vnl_swish_bwd without the intermediate (pre, dpre: ld = n) */
int vnl_outer_swish_bwd(const float* dv, int rows, const float* w, int n, const float* pre, float* dpre, void* stream);
/* n <= 4 scalar streams [T, B] of the unroll (reward, discount, truncation, log_prob) gathered by the minibatch's env index list in one
 * launch: dst[k][t * Bm + j] = src[k][t * B + idx[j]]; src / dst are HOST arrays of n device pointers. */
int vnl_gather_scalars(int n, const float* const* src, float* const* dst, int T, int B, const int32_t* idx, int Bm, void* stream);

/* Rollout-side sampling of brax NormalTanhDistribution (ppo_imitation/ppo_networks.py:55-83) on fp32 logits [rows, 2 nu]:
 * raw_action = loc + scale * eps_a (eps_a = NULL: the mode, `deterministic=True`), action = tanh(raw_action), log_prob(raw_action),
 * and rand_log_prob = log_prob of `rand_action` [nu] -- ONE uniform(-1, 1) draw of shape (action_size,) broadcast over the batch,
 * as the reference draws it (ppo_networks.py:68-73); rand_action / rand_log_prob may be NULL.  The fp32-accurate rollout policy
 * (policy.PrecisePolicy) = the learner's forward kernels + this one. */
int vnl_policy_sample(const float* logits, int ld, const float* eps_a, const float* rand_action, int rows, int nu, float* action,
                      float* raw_action, float* log_prob, float* rand_log_prob, void* stream);

/* brax `EvalWrapper` (envs/wrappers/training.py; installed by Evaluator at ppo_imitation/acting.py:109) folded over an unroll of T steps
 * that starts at reset: per env, episode_metrics[k] = sum_t metrics[t, k] * active_t (k < nm) and [nm] = the same for the reward,
 * active_{t+1} = active_t * (1 - done_t), episode_steps = steps of the first episode (info["steps"] while active).
 * metrics [T, B, nm], reward / done [T, B]; outputs episode_metrics [B, nm + 1], active [B], episode_steps [B]. */
int vnl_eval_metrics(int T, int B, int nm, const float* metrics, const float* reward, const float* done, float* episode_metrics, float* active,
                     float* episode_steps, void* stream);

/* Loss, part 1 (per row; intention_losses.py:149-166,189): brax NormalTanhDistribution on logits [rows, 2 nu]:
 *   target_lp[r] = log_prob(logits, raw_action), ent[r] = entropy(logits) with the sample loc + scale * eps_ent;
 *   termination[r] = (1 - discount[r]) * (1 - truncation[r]); rewards_s[r] = reward[r] * reward_scaling. */
int vnl_ppo_rows(const float* logits, int ld, const float* raw_action, const float* eps_ent, int rows, int nu, const float* discount,
                 const float* truncation, const float* reward, float reward_scaling, float* target_lp, float* ent, float* termination,
                 float* rewards_s, void* stream);
/* Loss, part 2 (intention_losses.py:177-200): advantage normalisation, clipped surrogate, value loss, entropy loss, and
 * their gradients w.r.t. logits (dlogits [rows, 2 nu], ld_d) and the baseline (dvalue [rows]).
 * metrics[8] (ACCUMULATED, caller zeroes): 0 total (without KL, added by vnl_heads_bwd into metrics[4]), 1 policy_loss, 2 v_loss,
 * 3 entropy_loss, 4 kl_loss_intention, 5 mean rho, 6 clipped fraction, 7 unused. */
int vnl_ppo_loss_bwd(const float* logits, int ld, const float* raw_action, const float* eps_ent, int rows, int nu, const float* target_lp,
                     const float* behaviour_lp, const float* ent, const float* advantages, const float* vs, const float* baseline,
                     float clipping_epsilon, float entropy_cost, int normalize_advantage, float* dlogits, int ld_d, float* dvalue,
                     float* metrics, float* scratch2, void* stream);

/* optax.adam (b1, b2, eps; eps_root 0) with constant learning rate over a flat parameter buffer.  Bias corrections
 * 1 - b^t: from the host (`step` = 1-based count of THIS update, bc_dev = NULL) or from device memory (`bc_dev` [2], written by
 * vnl_adam_tick, which also advances the device-resident step counter: the form a CUDA graph of the update replays).
 * grad_scale multiplies the gradients first (1 / world size after a SUM all-reduce = lax.pmean). */
int vnl_adam_tick(int* step_dev, float b1, float b2, float* bc_dev, void* stream);
int vnl_adam(float* params, const float* grads, float* m, float* v, size_t n, float lr, float b1, float b2, float eps, int step, float grad_scale,
             const float* bc_dev, void* stream);

/* dst[i] += src[i] for i < n (n <= 1024), each entry by one thread in launch order, no atomics: the running sum of the loss metrics
 * row of vnl_ppo_loss_bwd over the minibatch updates of an epoch (brax `training_epoch` reports their mean).  Enqueued after every
 * loss evaluation, inside the captured gradient graph, so the sum costs no host sync per update. */
int vnl_metrics_accumulate(const float* src, int n, float* dst, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* VNL_TRAIN_H_ */
