// vnl_train.cu -- the non-GEMM kernels of the PPO update (SURVEY section 8 row f2; C ABI in include/vnl_train.h):
// minibatch gather, obs normalisation, relu + LayerNorm forward / backward, swish, reparameterisation and its backward with
// the KL term, bias / weighted column sums, the value head, the PPO loss (brax NormalTanhDistribution log-prob / entropy,
// advantage normalisation, clipped surrogate, value loss) with its gradients, Adam and the 3xTF32 operand split; and the
// evaluator's reductions (EvalWrapper's episode sums, their per-clip statistics and per-frame profiles).
// All of them are HBM-bound row / elementwise passes: coalesced fp32, one warp per row where a row reduction is needed,
// fixed reduction trees inside a block; cross-block accumulation (bias / LayerNorm parameter gradients, loss scalars) uses
// red.global.add.  Reference: ppo_imitation/intention_losses.py:91-202, intention_policy_network.py:20-105, brax
// NormalTanhDistribution / networks.MLP / optax.adam semantics as restated in vnl-brax-imitation_b200/ppo.py::reference_loss.
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

#include "../../include/vnl_train.h"

namespace {

constexpr float kLog2 = 0.6931471805599453f;
constexpr float kHalfLog2Pi = 0.9189385332046727f;

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float softplus(float x) { return fmaxf(x, 0.0f) + log1pf(expf(-fabsf(x))); }  // logaddexp(x, 0)
__device__ __forceinline__ float sigmoidf(float x) { return 1.0f / (1.0f + expf(-x)); }
__device__ __forceinline__ float log_det_jac(float x) { return 2.0f * (kLog2 - x - softplus(-2.0f * x)); }  // brax TanhBijector

__global__ void split_kernel(const float* __restrict__ x, size_t n, float* __restrict__ hi, float* __restrict__ lo) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    const float v = x[i];
    const float h = __uint_as_float(__float_as_uint(v) & 0xffffe000u);
    hi[i] = h;
    lo[i] = v - h;
  }
}

__global__ void gather_kernel(const float* __restrict__ src, int B, int width, const int32_t* __restrict__ idx, int Bm, float* __restrict__ dst,
                              int ld) {
  const int row = blockIdx.x, t = row / Bm, j = row - t * Bm;
  const float* s = src + ((size_t)t * B + idx[j]) * width;
  float* d = dst + (size_t)row * ld;
  for (int c = threadIdx.x; c < ld; c += blockDim.x) d[c] = c < width ? s[c] : 0.0f;
}

__global__ void normalize_kernel(const float* __restrict__ obs, int ld_obs, int rows, int width, const float* __restrict__ mean,
                                 const float* __restrict__ sd, float* __restrict__ out, int ld_out) {
  const size_t total = (size_t)rows * width;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const int r = (int)(i / width), c = (int)(i - (size_t)r * width);
    out[(size_t)r * ld_out + c] = (obs[(size_t)r * ld_obs + c] - mean[c]) / sd[c];
  }
}

// one warp per row, n <= 1024 (n / 32 <= 32 values per lane, strided by 32: coalesced)
__global__ void relu_ln_fwd_kernel(const float* __restrict__ pre, int ld_pre, int rows, int n, const float* __restrict__ scale,
                                   const float* __restrict__ bias, float* __restrict__ out, int ld_out, float* __restrict__ stats) {
  const int lane = threadIdx.x & 31, wpb = blockDim.x >> 5;
  for (int r = blockIdx.x * wpb + (threadIdx.x >> 5); r < rows; r += gridDim.x * wpb) {
    const float* p = pre + (size_t)r * ld_pre;
    float s1 = 0.0f, s2 = 0.0f;
    for (int c = lane; c < n; c += 32) { const float x = fmaxf(p[c], 0.0f); s1 += x; s2 += x * x; }
    s1 = warp_sum(s1); s2 = warp_sum(s2);
    const float mu = s1 / (float)n, var = fmaxf(s2 / (float)n - mu * mu, 0.0f), rstd = 1.0f / sqrtf(var + 1e-6f);
    float* o = out + (size_t)r * ld_out;
    for (int c = lane; c < n; c += 32) o[c] = (fmaxf(p[c], 0.0f) - mu) * rstd * scale[c] + bias[c];
    if (lane == 0) { stats[2 * (size_t)r] = mu; stats[2 * (size_t)r + 1] = rstd; }
  }
}

// one warp per row; a block keeps per-column partials of dscale / dbias (and of the column sums of dpre = the bias gradient of the
// dense layer in front, when asked for) over its rows in registers (n <= 256: 8 per lane), adds the warps through shared memory
// and issues one red.add per column
template <int CPL>
__global__ void relu_ln_bwd_kernel(const float* __restrict__ dy, int ld_dy, const float* __restrict__ pre, int ld_pre, const float* __restrict__ stats,
                                   const float* __restrict__ scale, int rows, int n, float* __restrict__ dpre, int ld_dpre,
                                   float* __restrict__ dscale, float* __restrict__ dbias, float* __restrict__ dbias_pre) {
  extern __shared__ float sm[];  // [warps][3][n]
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, wpb = blockDim.x >> 5;
  float as[CPL], ab[CPL], ad[CPL], sc[CPL];
#pragma unroll
  for (int k = 0; k < CPL; ++k) { as[k] = ab[k] = ad[k] = 0.0f; sc[k] = lane + 32 * k < n ? scale[lane + 32 * k] : 0.0f; }
  for (int r = blockIdx.x * wpb + w; r < rows; r += gridDim.x * wpb) {
    const float mu = stats[2 * (size_t)r], rstd = stats[2 * (size_t)r + 1];
    const float* p = pre + (size_t)r * ld_pre;
    const float* g = dy + (size_t)r * ld_dy;
    float xh[CPL], gg[CPL], m1 = 0.0f, m2 = 0.0f;
#pragma unroll
    for (int k = 0; k < CPL; ++k) {
      const int c = lane + 32 * k;
      float x = 0.0f, d = 0.0f;
      if (c < n) { x = (fmaxf(p[c], 0.0f) - mu) * rstd; d = g[c]; }
      xh[k] = x;
      as[k] += d * x; ab[k] += d;
      gg[k] = d * sc[k];
      m1 += gg[k]; m2 += gg[k] * x;
    }
    m1 = warp_sum(m1) / (float)n; m2 = warp_sum(m2) / (float)n;
    float* o = dpre + (size_t)r * ld_dpre;
#pragma unroll
    for (int k = 0; k < CPL; ++k) {
      const int c = lane + 32 * k;
      if (c < n) {
        const float d = p[c] > 0.0f ? rstd * (gg[k] - m1 - xh[k] * m2) : 0.0f;
        o[c] = d;
        ad[k] += d;
      }
    }
  }
#pragma unroll
  for (int k = 0; k < CPL; ++k) {
    const int c = lane + 32 * k;
    if (c < n) { sm[(w * 3) * n + c] = as[k]; sm[(w * 3 + 1) * n + c] = ab[k]; sm[(w * 3 + 2) * n + c] = ad[k]; }
  }
  __syncthreads();
  for (int c = threadIdx.x; c < n; c += blockDim.x) {
    float a = 0.0f, b = 0.0f, d = 0.0f;
    for (int q = 0; q < wpb; ++q) { a += sm[(q * 3) * n + c]; b += sm[(q * 3 + 1) * n + c]; d += sm[(q * 3 + 2) * n + c]; }
    atomicAdd(dscale + c, a);
    atomicAdd(dbias + c, b);
    if (dbias_pre) atomicAdd(dbias_pre + c, d);
  }
}

__global__ void swish_fwd_kernel(const float* __restrict__ pre, size_t n, float* __restrict__ out) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    const float x = pre[i];
    out[i] = x * sigmoidf(x);
  }
}
__global__ void swish_bwd_kernel(const float* __restrict__ dy, const float* __restrict__ pre, size_t n, float* __restrict__ dpre) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    const float x = pre[i], s = sigmoidf(x);
    dpre[i] = dy[i] * (s + x * s * (1.0f - s));
  }
}

__global__ void reparam_fwd_kernel(const float* __restrict__ heads, const float* __restrict__ eps, int rows, int L, float* __restrict__ dec_in,
                                   int ld) {
  const size_t total = (size_t)rows * L;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const int r = (int)(i / L), l = (int)(i - (size_t)r * L);
    const float m = heads[(size_t)r * 2 * L + l], lv = heads[(size_t)r * 2 * L + L + l];
    dec_in[(size_t)r * ld + l] = m + eps[i] * expf(0.5f * lv);
  }
}
__global__ void heads_bwd_kernel(const float* __restrict__ ddec_in, int ld, const float* __restrict__ heads, const float* __restrict__ eps, int rows,
                                 int L, float kl_coef, float* __restrict__ dheads, float* __restrict__ kl_loss) {
  const size_t total = (size_t)rows * L;
  float acc = 0.0f;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const int r = (int)(i / L), l = (int)(i - (size_t)r * L);
    const float m = heads[(size_t)r * 2 * L + l], lv = heads[(size_t)r * 2 * L + L + l], dz = ddec_in[(size_t)r * ld + l];
    const float e = expf(lv);
    dheads[(size_t)r * 2 * L + l] = dz + kl_coef * m;
    dheads[(size_t)r * 2 * L + L + l] = dz * 0.5f * eps[i] * expf(0.5f * lv) - 0.5f * kl_coef * (1.0f - e);
    acc += -0.5f * kl_coef * (1.0f + lv - m * m - e);
  }
  __shared__ float red[32];
  acc = warp_sum(acc);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x < 32) {
    float v = threadIdx.x < (blockDim.x >> 5) ? red[threadIdx.x] : 0.0f;
    v = warp_sum(v);
    if (threadIdx.x == 0 && kl_loss) atomicAdd(kl_loss, v);
  }
}

// block = 32 columns x 8 row lanes; grid.x = column tiles, grid.y = row chunks
__global__ void colsum_kernel(const float* __restrict__ x, int ld, int rows, int n, const float* __restrict__ w, float* __restrict__ out) {
  __shared__ float sm[8][33];
  const int cx = threadIdx.x & 31, ry = threadIdx.x >> 5, c = blockIdx.x * 32 + cx;
  float acc = 0.0f;
  if (c < n) {
    if (w) {
#pragma unroll 4
      for (int r = blockIdx.y * 8 + ry; r < rows; r += gridDim.y * 8) acc += w[r] * x[(size_t)r * ld + c];
    } else {
#pragma unroll 4
      for (int r = blockIdx.y * 8 + ry; r < rows; r += gridDim.y * 8) acc += x[(size_t)r * ld + c];
    }
  }
  sm[ry][cx] = acc;
  __syncthreads();
  if (ry == 0 && c < n) {
    float s = 0.0f;
#pragma unroll
    for (int q = 0; q < 8; ++q) s += sm[q][cx];
    atomicAdd(out + c, s);
  }
}

__global__ void rowdot_kernel(const float* __restrict__ h, int ld, int rows, int n, const float* __restrict__ w, const float* __restrict__ b,
                              float* __restrict__ out) {
  const int lane = threadIdx.x & 31, wpb = blockDim.x >> 5;
  for (int r = blockIdx.x * wpb + (threadIdx.x >> 5); r < rows; r += gridDim.x * wpb) {
    const float* p = h + (size_t)r * ld;
    float acc = 0.0f;
    for (int c = lane; c < n; c += 32) acc += p[c] * w[c];
    acc = warp_sum(acc);
    if (lane == 0) out[r] = acc + (b ? b[0] : 0.0f);
  }
}
__global__ void outer_kernel(const float* __restrict__ dv, int rows, const float* __restrict__ w, int n, float* __restrict__ dh, int ld) {
  const size_t total = (size_t)rows * n;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const int r = (int)(i / n), c = (int)(i - (size_t)r * n);
    dh[(size_t)r * ld + c] = dv[r] * w[c];
  }
}

// one warp per row, lane = action dimension (nu <= 32)
// dpre[r, c] = dv[r] * w[c] * swish'(pre[r, c]): the value head's backward and the last hidden layer's activation backward in one pass
__global__ void outer_swish_bwd_kernel(const float* __restrict__ dv, int rows, const float* __restrict__ w, int n, const float* __restrict__ pre,
                                       float* __restrict__ dpre) {
  const size_t total = (size_t)rows * n;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const int r = (int)(i / n), c = (int)(i - (size_t)r * n);
    const float x = pre[i], s = sigmoidf(x);
    dpre[i] = dv[r] * w[c] * (s + x * s * (1.0f - s));
  }
}

// up to four [T, B] scalar streams of the unroll gathered in one launch: dst_k[t * Bm + j] = src_k[t * B + idx[j]]
struct Gather4 { const float* src[4]; float* dst[4]; };
__global__ void gather_scalars_kernel(Gather4 a, int n, int T, int B, const int32_t* __restrict__ idx, int Bm) {
  const int total = T * Bm;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    const int t = i / Bm, j = i - t * Bm;
    const size_t s = (size_t)t * B + idx[j];
#pragma unroll
    for (int k = 0; k < 4; ++k)
      if (k < n) a.dst[k][i] = a.src[k][s];
  }
}

__global__ void ppo_rows_kernel(const float* __restrict__ logits, int ld, const float* __restrict__ raw_action, const float* __restrict__ eps_ent,
                                int rows, int nu, const float* __restrict__ discount, const float* __restrict__ truncation,
                                const float* __restrict__ reward, float reward_scaling, float* __restrict__ target_lp, float* __restrict__ ent,
                                float* __restrict__ termination, float* __restrict__ rewards_s) {
  const int lane = threadIdx.x & 31, wpb = blockDim.x >> 5;
  for (int r = blockIdx.x * wpb + (threadIdx.x >> 5); r < rows; r += gridDim.x * wpb) {
    float lp = 0.0f, en = 0.0f;
    if (lane < nu) {
      const float loc = logits[(size_t)r * ld + lane], scale = softplus(logits[(size_t)r * ld + nu + lane]) + 0.001f;
      const float a = raw_action[(size_t)r * nu + lane], z = (a - loc) / scale, ls = logf(scale);
      lp = -0.5f * z * z - ls - kHalfLog2Pi - log_det_jac(a);
      en = 0.5f + kHalfLog2Pi + ls + log_det_jac(loc + scale * eps_ent[(size_t)r * nu + lane]);
    }
    lp = warp_sum(lp); en = warp_sum(en);
    if (lane == 0) {
      target_lp[r] = lp; ent[r] = en;
      termination[r] = (1.0f - discount[r]) * (1.0f - truncation[r]);
      rewards_s[r] = reward[r] * reward_scaling;
    }
  }
}

// rollout-side sampling (ppo_networks.py:55-83): raw = loc + scale * eps (or the mode, eps == NULL), log_prob(raw), action = tanh(raw),
// rand_log_prob = log_prob of ONE uniform(-1, 1) draw of shape (nu,) broadcast over the batch (ppo_networks.py:68-73)
__global__ void policy_sample_kernel(const float* __restrict__ logits, int ld, const float* __restrict__ eps_a, const float* __restrict__ rand_action,
                                     int rows, int nu, float* __restrict__ action, float* __restrict__ raw_action, float* __restrict__ log_prob,
                                     float* __restrict__ rand_log_prob) {
  const int lane = threadIdx.x & 31, wpb = blockDim.x >> 5;
  for (int r = blockIdx.x * wpb + (threadIdx.x >> 5); r < rows; r += gridDim.x * wpb) {
    float lp = 0.0f, rlp = 0.0f;
    if (lane < nu) {
      const float loc = logits[(size_t)r * ld + lane], scale = softplus(logits[(size_t)r * ld + nu + lane]) + 0.001f, ls = logf(scale);
      const float raw = eps_a ? loc + scale * eps_a[(size_t)r * nu + lane] : loc;
      raw_action[(size_t)r * nu + lane] = raw;
      action[(size_t)r * nu + lane] = tanhf(raw);
      const float z = (raw - loc) / scale;
      lp = -0.5f * z * z - ls - kHalfLog2Pi - log_det_jac(raw);
      if (rand_action) {
        const float a = rand_action[lane], zr = (a - loc) / scale;
        rlp = -0.5f * zr * zr - ls - kHalfLog2Pi - log_det_jac(a);
      }
    }
    lp = warp_sum(lp); rlp = warp_sum(rlp);
    if (lane == 0) {
      log_prob[r] = lp;
      if (rand_log_prob && rand_action) rand_log_prob[r] = rlp;
    }
  }
}

// brax EvalWrapper.step folded over an unroll that starts at reset: one thread per env walks its T steps.
__global__ void eval_metrics_kernel(int T, int B, int nm, const float* __restrict__ metrics, const float* __restrict__ reward,
                                    const float* __restrict__ done, float* __restrict__ episode_metrics, float* __restrict__ active,
                                    float* __restrict__ episode_steps) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  float act = 1.0f, steps = 0.0f, acc[16];
  for (int k = 0; k <= nm; ++k) acc[k] = 0.0f;
  for (int t = 0; t < T; ++t) {
    // episode_steps = where(active, nstate.info["steps"], episode_steps): an episode that is still active has taken t + 1 steps
    if (act != 0.0f) steps = (float)(t + 1);
    for (int k = 0; k < nm; ++k) acc[k] += metrics[((size_t)t * B + b) * nm + k] * act;
    acc[nm] += reward[(size_t)t * B + b] * act;
    act *= 1.0f - done[(size_t)t * B + b];
  }
  for (int k = 0; k <= nm; ++k) episode_metrics[(size_t)b * (nm + 1) + k] = acc[k];
  active[b] = act;
  episode_steps[b] = steps;
}

// Per-clip evaluation (vnl_eval_clip_stats / vnl_eval_frame_profile): one CTA per clip.  The CTA walks the batch kClipThreads envs
// at a time and compacts the envs of its clip with a block ballot scan (ascending env order, as done_list_kernel).  Which thread adds
// which value, and in what order, depends only on the inputs and the block size, never on launch timing: two calls are bit-identical.
constexpr int kClipThreads = 256;
constexpr int kClipWarps = kClipThreads / 32;

// This thread's slot in the ascending list of the envs of chunk [i0, i0 + kClipThreads) that belong to clip c (-1: its env does
// not); `len` = the list's length.  clip_id NULL: every env is clip 0.  The caller writes its slot, then synchronises.
__device__ __forceinline__ int clip_chunk_slot(const int* __restrict__ clip_id, int B, int i0, int c, int* wsum, int& len) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, i = i0 + threadIdx.x;
  const bool mine = i < B && (clip_id ? clip_id[i] == c : c == 0);
  const unsigned bal = __ballot_sync(0xffffffffu, mine);
  if (lane == 0) wsum[w] = __popc(bal);
  __syncthreads();
  int off = 0;
  len = 0;
  for (int q = 0; q < kClipWarps; ++q) { off += q < w ? wsum[q] : 0; len += wsum[q]; }
  return mine ? off + __popc(bal & ((1u << lane) - 1u)) : -1;
}

// Per clip: mean and population std (two passes, double) of nm + 2 columns over the clip's envs: episode_metrics[:, 0..nm], then
// episode_steps.  Lane k of every warp holds column k; warp w adds entries w, w + kClipWarps, ... of each chunk's list, and the
// warps' partials are added in warp order.
__global__ void __launch_bounds__(kClipThreads) eval_clip_stats_kernel(int B, int nm, const float* __restrict__ episode_metrics,
                                                                      const float* __restrict__ episode_steps, const int* __restrict__ clip_id,
                                                                      float* __restrict__ mean, float* __restrict__ sd, int* __restrict__ count) {
  __shared__ int s_env[kClipThreads], wsum[kClipWarps];
  __shared__ double red[kClipWarps][32], mom[2][32];
  const int c = blockIdx.x, lane = threadIdx.x & 31, w = threadIdx.x >> 5, ncol = nm + 2, ld = nm + 1;
  int total = 0;
  for (int pass = 0; pass < 2; ++pass) {  // 0: sums -> means, 1: squared deviations from them
    const double m = pass && lane < ncol ? mom[0][lane] : 0.0;
    double s = 0.0;
    total = 0;
    for (int i0 = 0; i0 < B; i0 += kClipThreads) {
      int len;
      const int slot = clip_chunk_slot(clip_id, B, i0, c, wsum, len);
      if (slot >= 0) s_env[slot] = i0 + threadIdx.x;
      __syncthreads();
      if (lane < ncol)
        for (int j = w; j < len; j += kClipWarps) {
          const int b = s_env[j];
          const double d = (double)(lane < ld ? episode_metrics[(size_t)b * ld + lane] : episode_steps[b]) - m;
          s += pass ? d * d : d;
        }
      total += len;
      __syncthreads();  // s_env and wsum are rewritten by the next chunk
    }
    if (lane < ncol) red[w][lane] = s;
    __syncthreads();
    if (threadIdx.x < ncol) {
      double a = 0.0;
      for (int q = 0; q < kClipWarps; ++q) a += red[q][threadIdx.x];
      mom[pass][threadIdx.x] = a / total;
    }
    __syncthreads();
  }
  if (threadIdx.x < ncol) {
    mean[(size_t)c * ncol + threadIdx.x] = total ? (float)mom[0][threadIdx.x] : nanf("");
    sd[(size_t)c * ncol + threadIdx.x] = total ? (float)sqrt(mom[1][threadIdx.x]) : nanf("");
  }
  if (threadIdx.x == 0) count[c] = total;
}

// Per clip and clip frame: sums of the metrics and the reward over the first-episode steps whose reward read that frame.  Thread f
// walks each chunk's list in order and adds, per env, its steps t (ascending) with clamp(start + t, 0, L - 1) == f: no two threads
// write the same bin.  Clips longer than the block go round in groups of kClipThreads frames.
__global__ void __launch_bounds__(kClipThreads) eval_frame_profile_kernel(int T, int B, int nm, const float* __restrict__ metrics,
                                                                         const float* __restrict__ reward, const float* __restrict__ episode_steps,
                                                                         const int* __restrict__ start_frame, const int* __restrict__ clip_id,
                                                                         int L, float* __restrict__ frame_sum, int* __restrict__ frame_count) {
  __shared__ int s_env[kClipThreads], s_start[kClipThreads], s_n[kClipThreads], wsum[kClipWarps];
  const int c = blockIdx.x, ld = nm + 1;
  for (int f0 = 0; f0 < L; f0 += kClipThreads) {
    const int f = f0 + threadIdx.x;
    double acc[15], racc = 0.0;  // static indices only: the metric sums stay in registers
#pragma unroll
    for (int k = 0; k < 15; ++k) acc[k] = 0.0;
    int cnt = 0;
    for (int i0 = 0; i0 < B; i0 += kClipThreads) {
      int len;
      const int slot = clip_chunk_slot(clip_id, B, i0, c, wsum, len);
      if (slot >= 0) {
        const int i = i0 + threadIdx.x;
        s_env[slot] = i;
        s_start[slot] = start_frame[i];
        s_n[slot] = min((int)episode_steps[i], T);
      }
      __syncthreads();
      if (f < L)
        for (int j = 0; j < len; ++j) {
          const int b = s_env[j], s = s_start[j], n = s_n[j];
          // the steps that bin to f: t = f - s inside the clip, and every t that clamps to f at either end
          const int lo = max(f == 0 ? 0 : f - s, 0), hi = min(f == L - 1 ? n - 1 : f - s, n - 1);
          for (int t = lo; t <= hi; ++t) {
            const size_t r = (size_t)t * B + b;
#pragma unroll
            for (int k = 0; k < 15; ++k)
              if (k < nm) acc[k] += (double)metrics[r * nm + k];
            racc += (double)reward[r];
            ++cnt;
          }
        }
      __syncthreads();  // the list is rebuilt for the next chunk
    }
    if (f < L) {
      float* out = frame_sum + ((size_t)c * L + f) * ld;
#pragma unroll
      for (int k = 0; k < 15; ++k)
        if (k < nm) out[k] = (float)acc[k];
      out[nm] = (float)racc;
      frame_count[(size_t)c * L + f] = cnt;
    }
  }
}

// mean and population std of `rows` values (jnp.mean / jnp.std), one block, fixed order
__global__ void mean_std_kernel(const float* __restrict__ x, int rows, float* __restrict__ out2) {
  __shared__ double r1[32], r2[32];
  double s1 = 0.0, s2 = 0.0;
  for (int i = threadIdx.x; i < rows; i += blockDim.x) { const double v = x[i]; s1 += v; s2 += v * v; }
  for (int o = 16; o > 0; o >>= 1) { s1 += __shfl_xor_sync(0xffffffffu, s1, o); s2 += __shfl_xor_sync(0xffffffffu, s2, o); }
  if ((threadIdx.x & 31) == 0) { r1[threadIdx.x >> 5] = s1; r2[threadIdx.x >> 5] = s2; }
  __syncthreads();
  if (threadIdx.x == 0) {
    double a = 0.0, b = 0.0;
    for (int q = 0; q < (int)(blockDim.x >> 5); ++q) { a += r1[q]; b += r2[q]; }
    const double mu = a / rows, var = b / rows - mu * mu;
    out2[0] = (float)mu;
    out2[1] = (float)sqrt(var > 0.0 ? var : 0.0);
  }
}

__global__ void ppo_loss_bwd_kernel(const float* __restrict__ logits, int ld, const float* __restrict__ raw_action, const float* __restrict__ eps_ent,
                                    int rows, int nu, const float* __restrict__ target_lp, const float* __restrict__ behaviour_lp,
                                    const float* __restrict__ ent, const float* __restrict__ advantages, const float* __restrict__ vs,
                                    const float* __restrict__ baseline, float clip_eps, float entropy_cost, int normalize,
                                    const float* __restrict__ adv_stats, float* __restrict__ dlogits, int ld_d, float* __restrict__ dvalue,
                                    float* __restrict__ metrics) {
  const int lane = threadIdx.x & 31, wpb = blockDim.x >> 5, w = threadIdx.x >> 5;
  const float invR = 1.0f / (float)rows;
  const float amu = adv_stats[0], asd = adv_stats[1];
  float m_pol = 0.0f, m_v = 0.0f, m_ent = 0.0f, m_rho = 0.0f, m_clip = 0.0f;  // lane 0 accumulates
  for (int r = blockIdx.x * wpb + w; r < rows; r += gridDim.x * wpb) {
    float A = advantages[r];
    if (normalize) A = (A - amu) / (asd + 1e-8f);
    const float rho = expf(target_lp[r] - behaviour_lp[r]);
    const float s1 = rho * A, s2 = fminf(fmaxf(rho, 1.0f - clip_eps), 1.0f + clip_eps) * A;
    const bool inside = rho >= 1.0f - clip_eps && rho <= 1.0f + clip_eps;
    // d(-min(s1, s2) / R) / d target_lp: the unclipped branch (or the tie inside the clip range) carries A rho
    const float g_lp = (inside || s1 < s2) ? -A * rho * invR : 0.0f;
    if (lane < nu) {
      const float loc = logits[(size_t)r * ld + lane], rs = logits[(size_t)r * ld + nu + lane];
      const float scale = softplus(rs) + 0.001f, a = raw_action[(size_t)r * nu + lane], e = eps_ent[(size_t)r * nu + lane];
      const float d = a - loc, inv = 1.0f / scale;
      const float t = -2.0f * tanhf(loc + scale * e);  // d log_det_jac / d sample
      const float gloc = g_lp * d * inv * inv - entropy_cost * invR * t;
      const float gscale = g_lp * (d * d * inv * inv * inv - inv) - entropy_cost * invR * (inv + t * e);
      dlogits[(size_t)r * ld_d + lane] = gloc;
      dlogits[(size_t)r * ld_d + nu + lane] = gscale * sigmoidf(rs);
    }
    if (lane == 0) {
      const float ve = vs[r] - baseline[r];
      dvalue[r] = -0.5f * invR * ve;
      m_pol += -fminf(s1, s2) * invR;
      m_v += 0.25f * ve * ve * invR;
      m_ent += -entropy_cost * ent[r] * invR;
      m_rho += rho * invR;
      m_clip += inside ? 0.0f : invR;
    }
  }
  __shared__ float red[32][5];
  if (lane == 0) { red[w][0] = m_pol; red[w][1] = m_v; red[w][2] = m_ent; red[w][3] = m_rho; red[w][4] = m_clip; }
  __syncthreads();
  if (threadIdx.x < 5) {
    float s = 0.0f;
    for (int q = 0; q < wpb; ++q) s += red[q][threadIdx.x];
    const int slot[5] = {1, 2, 3, 5, 6};
    atomicAdd(metrics + slot[threadIdx.x], s);
    if (threadIdx.x < 3) atomicAdd(metrics, s);
  }
}

__global__ void adam_tick_kernel(int* step, float b1, float b2, float* bc) {
  const int t = *step + 1;
  *step = t;
  bc[0] = 1.0f - powf(b1, (float)t);
  bc[1] = 1.0f - powf(b2, (float)t);
}
__global__ void adam_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m, float* __restrict__ v, size_t n, float lr,
                            float b1, float b2, float eps, float bc1, float bc2, float gscale, const float* __restrict__ bc_dev) {
  if (bc_dev) { bc1 = bc_dev[0]; bc2 = bc_dev[1]; }
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    const float gi = g[i] * gscale;
    const float mi = b1 * m[i] + (1.0f - b1) * gi, vi = b2 * v[i] + (1.0f - b2) * gi * gi;
    m[i] = mi; v[i] = vi;
    p[i] -= lr * (mi / bc1) / (sqrtf(vi / bc2) + eps);
  }
}

// dst[i] += src[i]: one thread per entry of a short metrics row, so every sum is added in update order (no atomics)
__global__ void metrics_accumulate_kernel(const float* __restrict__ src, int n, float* __restrict__ dst) {
  for (int i = threadIdx.x; i < n; i += blockDim.x) dst[i] += src[i];
}

inline int grid_for(size_t n, int threads) {
  size_t b = (n + threads - 1) / threads;
  if (b > 148 * 8) b = 148 * 8;
  return (int)(b < 1 ? 1 : b);
}
inline int rc() { return (int)cudaGetLastError(); }

}  // namespace

extern "C" {

int vnl_split_tf32(const float* x, size_t n, float* hi, float* lo, void* stream) {
  if (!x || !hi || !lo) return -1;
  if (n == 0) return 0;
  split_kernel<<<grid_for(n, 256), 256, 0, (cudaStream_t)stream>>>(x, n, hi, lo);
  return rc();
}

int vnl_gather_rows(const float* src, int T, int B, int width, const int32_t* idx, int Bm, float* dst, int ld_dst, void* stream) {
  if (!src || !idx || !dst || T <= 0 || B <= 0 || width <= 0 || Bm <= 0 || ld_dst < width) return -1;
  gather_kernel<<<T * Bm, 256, 0, (cudaStream_t)stream>>>(src, B, width, idx, Bm, dst, ld_dst);
  return rc();
}

int vnl_obs_normalize(const float* obs, int ld_obs, int rows, int width, const float* mean, const float* sd, float* out, int ld_out,
                      void* stream) {
  if (!obs || !mean || !sd || !out || rows <= 0 || width <= 0 || ld_obs < width || ld_out < width) return -1;
  normalize_kernel<<<grid_for((size_t)rows * width, 256), 256, 0, (cudaStream_t)stream>>>(obs, ld_obs, rows, width, mean, sd, out, ld_out);
  return rc();
}

int vnl_relu_ln_fwd(const float* pre, int ld_pre, int rows, int n, const float* scale, const float* bias, float* out, int ld_out,
                    float* stats, void* stream) {
  if (!pre || !scale || !bias || !out || !stats || rows <= 0 || n <= 0 || n > 1024 || ld_pre < n || ld_out < n) return -1;
  relu_ln_fwd_kernel<<<grid_for((size_t)rows * 32, 256), 256, 0, (cudaStream_t)stream>>>(pre, ld_pre, rows, n, scale, bias, out, ld_out, stats);
  return rc();
}

int vnl_relu_ln_bwd(const float* dy, int ld_dy, const float* pre, int ld_pre, const float* stats, const float* scale, int rows, int n,
                    float* dpre, int ld_dpre, float* dscale, float* dbias, float* dbias_pre, void* stream) {
  if (!dy || !pre || !stats || !scale || !dpre || !dscale || !dbias || rows <= 0 || n <= 0 || n > 256) return -1;
  if (ld_dy < n || ld_pre < n || ld_dpre < n) return -1;
  const int threads = 256, grid = grid_for((size_t)rows * 32, threads) < 148 ? grid_for((size_t)rows * 32, threads) : 148;
  const size_t smem = (size_t)(threads / 32) * 3 * n * sizeof(float);
  relu_ln_bwd_kernel<8><<<grid, threads, smem, (cudaStream_t)stream>>>(dy, ld_dy, pre, ld_pre, stats, scale, rows, n, dpre, ld_dpre, dscale, dbias, dbias_pre);
  return rc();
}

int vnl_swish_fwd(const float* pre, size_t n, float* out, void* stream) {
  if (!pre || !out) return -1;
  if (n == 0) return 0;  // as split and Adam: nothing to enqueue, and an earlier launch's error is not this call's to report
  swish_fwd_kernel<<<grid_for(n, 256), 256, 0, (cudaStream_t)stream>>>(pre, n, out);
  return rc();
}
int vnl_swish_bwd(const float* dy, const float* pre, size_t n, float* dpre, void* stream) {
  if (!dy || !pre || !dpre) return -1;
  if (n == 0) return 0;
  swish_bwd_kernel<<<grid_for(n, 256), 256, 0, (cudaStream_t)stream>>>(dy, pre, n, dpre);
  return rc();
}

int vnl_reparam_fwd(const float* heads, const float* eps, int rows, int L, float* dec_in, int ld, void* stream) {
  if (!heads || !eps || !dec_in || rows <= 0 || L <= 0 || ld < L) return -1;
  reparam_fwd_kernel<<<grid_for((size_t)rows * L, 256), 256, 0, (cudaStream_t)stream>>>(heads, eps, rows, L, dec_in, ld);
  return rc();
}
int vnl_heads_bwd(const float* ddec_in, int ld, const float* heads, const float* eps, int rows, int L, float kl_coef, float* dheads,
                  float* kl_loss, void* stream) {
  if (!ddec_in || !heads || !eps || !dheads || rows <= 0 || L <= 0 || ld < L) return -1;
  heads_bwd_kernel<<<grid_for((size_t)rows * L, 256), 256, 0, (cudaStream_t)stream>>>(ddec_in, ld, heads, eps, rows, L, kl_coef, dheads, kl_loss);
  return rc();
}

int vnl_colsum(const float* x, int ld, int rows, int n, const float* w, float* out, void* stream) {
  if (!x || !out || rows <= 0 || n <= 0 || ld < n) return -1;
  // 4 rows per thread: the kernel is bound by the latency of its dependent-looking row walk, not by bandwidth (32 rows per thread
  // measured 18 us for any width at 5120 rows); one red.add per column and chunk
  int chunks = (rows + 31) / 32;
  if (chunks > 512) chunks = 512;
  colsum_kernel<<<dim3((n + 31) / 32, chunks), 256, 0, (cudaStream_t)stream>>>(x, ld, rows, n, w, out);
  return rc();
}
int vnl_rowdot(const float* h, int ld, int rows, int n, const float* w, const float* b, float* out, void* stream) {
  if (!h || !w || !out || rows <= 0 || n <= 0 || ld < n) return -1;
  rowdot_kernel<<<grid_for((size_t)rows * 32, 256), 256, 0, (cudaStream_t)stream>>>(h, ld, rows, n, w, b, out);
  return rc();
}
int vnl_outer(const float* dv, int rows, const float* w, int n, float* dh, int ld, void* stream) {
  if (!dv || !w || !dh || rows <= 0 || n <= 0 || ld < n) return -1;
  outer_kernel<<<grid_for((size_t)rows * n, 256), 256, 0, (cudaStream_t)stream>>>(dv, rows, w, n, dh, ld);
  return rc();
}

int vnl_outer_swish_bwd(const float* dv, int rows, const float* w, int n, const float* pre, float* dpre, void* stream) {
  if (!dv || !w || !pre || !dpre || rows <= 0 || n <= 0) return -1;
  outer_swish_bwd_kernel<<<grid_for((size_t)rows * n, 256), 256, 0, (cudaStream_t)stream>>>(dv, rows, w, n, pre, dpre);
  return rc();
}

int vnl_gather_scalars(int n, const float* const* src, float* const* dst, int T, int B, const int32_t* idx, int Bm, void* stream) {
  if (n < 1 || n > 4 || !src || !dst || !idx || T <= 0 || B <= 0 || Bm <= 0) return -1;
  Gather4 a{};
  for (int k = 0; k < n; ++k) {
    if (!src[k] || !dst[k]) return -1;
    a.src[k] = src[k];
    a.dst[k] = dst[k];
  }
  gather_scalars_kernel<<<grid_for((size_t)T * Bm, 256), 256, 0, (cudaStream_t)stream>>>(a, n, T, B, idx, Bm);
  return rc();
}

int vnl_policy_sample(const float* logits, int ld, const float* eps_a, const float* rand_action, int rows, int nu, float* action,
                      float* raw_action, float* log_prob, float* rand_log_prob, void* stream) {
  if (!logits || !action || !raw_action || !log_prob || rows <= 0 || nu <= 0 || nu > 32 || ld < 2 * nu) return -1;
  policy_sample_kernel<<<grid_for((size_t)rows * 32, 256), 256, 0, (cudaStream_t)stream>>>(logits, ld, eps_a, rand_action, rows, nu, action, raw_action,
                                                                                          log_prob, rand_log_prob);
  return rc();
}

int vnl_eval_metrics(int T, int B, int nm, const float* metrics, const float* reward, const float* done, float* episode_metrics, float* active,
                     float* episode_steps, void* stream) {
  if (T <= 0 || B <= 0 || nm < 0 || nm > 15 || !metrics || !reward || !done || !episode_metrics || !active || !episode_steps) return -1;
  eval_metrics_kernel<<<(B + 127) / 128, 128, 0, (cudaStream_t)stream>>>(T, B, nm, metrics, reward, done, episode_metrics, active, episode_steps);
  return rc();
}

int vnl_eval_clip_stats(int B, int nm, const float* episode_metrics, const float* episode_steps, const int* clip_id, int nclips, float* mean,
                        float* std, int* count, void* stream) {
  if (B < 1 || nm < 0 || nm > 15 || nclips < 1 || !episode_metrics || !episode_steps || !mean || !std || !count) return -1;
  eval_clip_stats_kernel<<<nclips, kClipThreads, 0, (cudaStream_t)stream>>>(B, nm, episode_metrics, episode_steps, clip_id, mean, std, count);
  return rc();
}

int vnl_eval_frame_profile(int T, int B, int nm, const float* metrics, const float* reward, const float* episode_steps, const int* start_frame,
                           const int* clip_id, int nclips, int clip_len, float* frame_sum, int* frame_count, void* stream) {
  if (T < 1 || B < 1 || nm < 0 || nm > 15 || nclips < 1 || clip_len < 1) return -1;
  if (!metrics || !reward || !episode_steps || !start_frame || !frame_sum || !frame_count) return -1;
  eval_frame_profile_kernel<<<nclips, kClipThreads, 0, (cudaStream_t)stream>>>(T, B, nm, metrics, reward, episode_steps, start_frame, clip_id,
                                                                               clip_len, frame_sum, frame_count);
  return rc();
}

int vnl_ppo_rows(const float* logits, int ld, const float* raw_action, const float* eps_ent, int rows, int nu, const float* discount,
                 const float* truncation, const float* reward, float reward_scaling, float* target_lp, float* ent, float* termination,
                 float* rewards_s, void* stream) {
  if (!logits || !raw_action || !eps_ent || !discount || !truncation || !reward || !target_lp || !ent || !termination || !rewards_s) return -1;
  if (rows <= 0 || nu <= 0 || nu > 32 || ld < 2 * nu) return -1;
  ppo_rows_kernel<<<grid_for((size_t)rows * 32, 256), 256, 0, (cudaStream_t)stream>>>(logits, ld, raw_action, eps_ent, rows, nu, discount, truncation,
                                                                                     reward, reward_scaling, target_lp, ent, termination, rewards_s);
  return rc();
}

int vnl_ppo_loss_bwd(const float* logits, int ld, const float* raw_action, const float* eps_ent, int rows, int nu, const float* target_lp,
                     const float* behaviour_lp, const float* ent, const float* advantages, const float* vs, const float* baseline,
                     float clipping_epsilon, float entropy_cost, int normalize_advantage, float* dlogits, int ld_d, float* dvalue,
                     float* metrics, float* scratch2, void* stream) {
  if (!logits || !raw_action || !eps_ent || !target_lp || !behaviour_lp || !ent || !advantages || !vs || !baseline || !dlogits || !dvalue ||
      !metrics || !scratch2)
    return -1;
  if (rows <= 0 || nu <= 0 || nu > 32 || ld < 2 * nu || ld_d < 2 * nu) return -1;
  mean_std_kernel<<<1, 1024, 0, (cudaStream_t)stream>>>(advantages, rows, scratch2);
  int grid = grid_for((size_t)rows * 32, 256);
  if (grid > 148) grid = 148;
  ppo_loss_bwd_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(logits, ld, raw_action, eps_ent, rows, nu, target_lp, behaviour_lp, ent, advantages, vs,
                                                              baseline, clipping_epsilon, entropy_cost, normalize_advantage, scratch2, dlogits, ld_d,
                                                              dvalue, metrics);
  return rc();
}

int vnl_adam_tick(int* step_dev, float b1, float b2, float* bc_dev, void* stream) {
  if (!step_dev || !bc_dev) return -1;
  adam_tick_kernel<<<1, 1, 0, (cudaStream_t)stream>>>(step_dev, b1, b2, bc_dev);
  return rc();
}

int vnl_adam(float* params, const float* grads, float* m, float* v, size_t n, float lr, float b1, float b2, float eps, int step, float grad_scale,
             const float* bc_dev, void* stream) {
  if (!params || !grads || !m || !v || (!bc_dev && step < 1)) return -1;
  if (n == 0) return 0;
  const float bc1 = bc_dev ? 1.0f : 1.0f - powf(b1, (float)step), bc2 = bc_dev ? 1.0f : 1.0f - powf(b2, (float)step);
  adam_kernel<<<grid_for(n, 256), 256, 0, (cudaStream_t)stream>>>(params, grads, m, v, n, lr, b1, b2, eps, bc1, bc2, grad_scale, bc_dev);
  return rc();
}

int vnl_metrics_accumulate(const float* src, int n, float* dst, void* stream) {
  if (!src || !dst || n <= 0 || n > 1024) return -1;
  metrics_accumulate_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(src, n, dst);
  return rc();
}

}  // extern "C"
