// SAC / DrQ loss-side kernels (fp32): JAX-compatible key schedule and random fills, tanh-Gaussian
// sample + log-prob, REDQ subsample-min TD target, the three losses with their analytic gradients,
// and the fused 3-optimizer Adam + polyak update.
//
// Reference (relative to serl_launcher/serl_launcher):
//   agents/continuous/sac.py:118-132   _compute_next_actions (policy forward, sample_and_log_prob)
//   agents/continuous/sac.py:134-191   critic_loss_fn   (subsample with replacement, min, TD target, MSE)
//   agents/continuous/sac.py:193-221   policy_loss_fn   (mean over the ensemble, -mean(q - alpha*logp))
//   agents/continuous/sac.py:223-234   temperature_loss_fn + networks/lagrange.py:9-78
//   agents/continuous/sac.py:243-299   update: key split order, rng bookkeeping
//   agents/continuous/drq.py:307-308   augmentation key split
//   networks/actor_critic_nets.py:178-272   Policy / TanhMultivariateNormalDiag
//   common/common.py:124-168           target_update, apply_gradients (3 Adam txs, all tick every call)
//   common/optimizers.py:6-56          Adam + warmup schedule
// Restated in oracle/drq.py (derive_update_randomness, tanh_normal_sample_logp, update, adam_tx_update).
#include "common.cuh"
#include "serl_b200.h"

namespace serl {

// ---------------------------------------------------------------------------------------------
// Key schedule.  keys[] slots (2 words each): see SERL_KEY_* in serl_b200.h.
// ---------------------------------------------------------------------------------------------
__global__ void rng_schedule_kernel(uint32_t* rng, uint32_t* keys, int do_aug, int do_update) {
  pdl_prologue();
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  u32x2 r{rng[0], rng[1]};
  auto put = [&](int slot, u32x2 k) { keys[2 * slot] = k.x; keys[2 * slot + 1] = k.y; };
  if (do_aug) {                                     // drq.py:307-308: rng, obs_rng, next_obs_rng = split(rng, 3)
    put(SERL_KEY_CROP_OBS, jax_split_at(r, 3, 1));
    put(SERL_KEY_CROP_NEXT, jax_split_at(r, 3, 2));
    r = jax_split_at(r, 3, 0);
  }
  if (do_update) {                                  // common.py:198-200: new_rng, actor, critic, temperature = split(rng, 4)
    const u32x2 k_actor = jax_split_at(r, 4, 1), k_critic = jax_split_at(r, 4, 2), k_temp = jax_split_at(r, 4, 3);
    const u32x2 c1 = jax_split_at(k_critic, 2, 0);  // sac.py:137  rng, next_action_sample_key = split(rng)
    put(SERL_KEY_CRITIC_NEXT, jax_split_at(k_critic, 2, 1));
    put(SERL_KEY_CRITIC_SUBSAMPLE, jax_split_at(c1, 2, 1));   // sac.py:152
    put(SERL_KEY_ACTOR_DROPOUT, jax_split_at(k_actor, 4, 1)); // sac.py:197  rng, policy_rng, sample_rng, critic_rng
    put(SERL_KEY_ACTOR_SAMPLE, jax_split_at(k_actor, 4, 2));
    put(SERL_KEY_TEMP_NEXT, jax_split_at(k_temp, 2, 1));      // sac.py:224
    r = jax_split_at(r, 2, 0);                      // sac.py:288  rng, _ = split(self.state.rng)
  }
  rng[0] = r.x; rng[1] = r.y;
}

__global__ void normal_fill_kernel(const uint32_t* key, float* out, int n) {
  pdl_prologue();
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j < n) out[j] = bits_to_normal(jax_random_bits_at(u32x2{key[0], key[1]}, (uint32_t)n, (uint32_t)j));
}

// keep-mask of camera `fold`: bernoulli(fold_in(key, fold), keep, (n,)) (repo spec, oracle/drq.py::_dropout_masks)
__global__ void dropout_mask_kernel(const uint32_t* key, uint32_t fold, float keep, uint8_t* mask, int n) {
  pdl_prologue();
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= n) return;
  const u32x2 k = jax_fold_in(u32x2{key[0], key[1]}, fold);
  mask[j] = bits_to_uniform01(jax_random_bits_at(k, (uint32_t)n, (uint32_t)j)) < keep ? 1 : 0;
}

// jax.random.randint(key, (n,), 0, ensemble) (sac.py:152-158): k1, k2 = split(key); element j combines word j of
// random_bits(k1, (n,)) and random_bits(k2, (n,)) exactly like jax_randint2 does for n = 2.
__global__ void subsample_idx_kernel(const uint32_t* key, int ensemble, int32_t* out, int n) {
  pdl_prologue();
  const int j = threadIdx.x;
  if (blockIdx.x != 0 || j >= n) return;
  const u32x2 k{key[0], key[1]};
  const uint32_t span = (uint32_t)ensemble;
  const uint32_t hb = jax_random_bits_at(jax_split_at(k, 2, 0), (uint32_t)n, (uint32_t)j);
  const uint32_t lb = jax_random_bits_at(jax_split_at(k, 2, 1), (uint32_t)n, (uint32_t)j);
  uint32_t mult = 65536u % span; mult = (mult * mult) % span;
  out[j] = (int)(((hb % span) * mult + (lb % span)) % span);
}

// ---------------------------------------------------------------------------------------------
// tanh-Gaussian: std = clip(exp(log_std), lo, hi); u = mu + std*eps; a = tanh(u);
// logp = sum_i [-0.5 z^2 - log std - 0.5 log 2pi] - sum_i 2 (log 2 - u - softplus(-2u)),  z = (u - mu)/std
// ---------------------------------------------------------------------------------------------
__device__ inline float softplusf(float x) { return fmaxf(x, 0.f) + log1pf(expf(-fabsf(x))); }

__global__ void tanh_gaussian_fwd_kernel(const float* __restrict__ mu, const float* __restrict__ log_std,
                                         const float* __restrict__ eps, float std_min, float std_max,
                                         float* __restrict__ act, int ld_act, float* __restrict__ logp,
                                         float* __restrict__ u_out, float* __restrict__ std_out, int B, int A, int deterministic) {
  pdl_prologue();
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  float lp = 0.f;
  for (int i = 0; i < A; ++i) {
    const float m = mu[b * A + i];
    const float sd = fminf(fmaxf(expf(log_std[b * A + i]), std_min), std_max);
    const float e = deterministic ? 0.f : eps[b * A + i];
    const float u = m + sd * e;
    const float z = (u - m) / sd;
    lp += -0.5f * z * z - logf(sd) - 0.918938533204672742f;
    lp -= 2.f * (0.693147180559945309f - u - softplusf(-2.f * u));
    act[(size_t)b * ld_act + i] = tanhf(u);
    if (u_out) u_out[b * A + i] = u;
    if (std_out) std_out[b * A + i] = sd;
  }
  if (logp) logp[b] = lp;
}

// ---------------------------------------------------------------------------------------------
// TD target + critic loss.  One CTA; E*B is a few thousand.
//   y_b = r_b + gamma * mask_b * min_j Q'[sub_j, b]  (- alpha * logp'_b if backup_entropy)
//   loss = mean_{e,b} (Q[e,b] - y_b)^2 ; dQ[e,b] = 2 (Q - y) / (E*B) * grad_scale
// info[0..2] = {critic_loss, mean Q, mean y} * grad_scale: grad_scale = 1/world under data parallelism, so that the ONE
// SUM all-reduce that carries the gradients also turns the per-rank infos into their mean (jax.lax.pmean(grads_and_aux),
// common.py:213-214); 1 otherwise.  Same convention in actor_loss_kernel / temperature_loss_kernel.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(1024) critic_loss_kernel(const float* __restrict__ q, const float* __restrict__ q_next,
                                                           const int32_t* __restrict__ sub, int n_sub,
                                                           const float* __restrict__ rewards, const float* __restrict__ masks,
                                                           const float* __restrict__ logp_next, const float* __restrict__ lagrange,
                                                           int backup_entropy, float gamma, float grad_scale,
                                                           float* __restrict__ target_q, float* __restrict__ dq,
                                                           float* __restrict__ info, int E, int B) {
  pdl_prologue();
  __shared__ float red[64];
  float sl = 0.f, sq = 0.f, sy = 0.f, dummy = 0.f;
  for (int b = threadIdx.x; b < B; b += blockDim.x) {
    float mn;
    if (n_sub > 0) {
      mn = q_next[(size_t)sub[0] * B + b];
      for (int j = 1; j < n_sub; ++j) mn = fminf(mn, q_next[(size_t)sub[j] * B + b]);
    } else {
      mn = q_next[b];
      for (int e = 1; e < E; ++e) mn = fminf(mn, q_next[(size_t)e * B + b]);
    }
    float y = rewards[b] + gamma * masks[b] * mn;
    if (backup_entropy) y -= softplusf(lagrange[0]) * logp_next[b];
    target_q[b] = y;
    sy += y;
    for (int e = 0; e < E; ++e) {
      const float d = q[(size_t)e * B + b] - y;
      sl += d * d; sq += q[(size_t)e * B + b];
      dq[(size_t)e * B + b] = 2.f * d / (float)(E * B) * grad_scale;
    }
  }
  block_sum2(sl, sq, red);
  block_sum2(sy, dummy, red);
  if (threadIdx.x == 0) { info[0] = grad_scale * sl / (float)(E * B); info[1] = grad_scale * sq / (float)(E * B); info[2] = grad_scale * sy / (float)B; }
}

// ---------------------------------------------------------------------------------------------
// Actor loss: L = -mean_b(qbar_b - alpha * logp_b), qbar = mean_e Q_e(s, a).
// Backward w.r.t. the policy head outputs, given da = dL/da from the critic input-gradient
// (critic seeded with dQ[e,b] = -1/(E*B)):
//   du_i = da_i (1 - a_i^2) + (alpha/B) * 2 a_i ;  dmu_i = du_i ;
//   dlogstd_i = [du_i * std_i * eps_i - alpha/B] * 1[std unclipped]
// info[0..2] = {actor_loss, temperature(alpha), entropy}
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(1024) actor_loss_kernel(const float* __restrict__ q, const float* __restrict__ logp,
                                                          const float* __restrict__ lagrange, const float* __restrict__ da, int ld_da,
                                                          const float* __restrict__ act, int ld_act, const float* __restrict__ std,
                                                          const float* __restrict__ log_std, const float* __restrict__ eps,
                                                          float std_min, float std_max, float grad_scale,
                                                          float* __restrict__ dmu, float* __restrict__ dlogstd,
                                                          float* __restrict__ info, int E, int B, int A) {
  pdl_prologue();
  __shared__ float red[64];
  const float alpha = softplusf(lagrange[0]);
  float sobj = 0.f, slp = 0.f;
  for (int b = threadIdx.x; b < B; b += blockDim.x) {
    float qb = 0.f;
    for (int e = 0; e < E; ++e) qb += q[(size_t)e * B + b];
    qb /= (float)E;
    sobj += qb - alpha * logp[b];
    slp += logp[b];
    for (int i = 0; i < A; ++i) {
      const float a = act[(size_t)b * ld_act + i];
      const float du = da[(size_t)b * ld_da + i] * (1.f - a * a) + grad_scale * (alpha / (float)B) * 2.f * a;
      dmu[b * A + i] = du;
      const float raw = expf(log_std[b * A + i]);
      const bool inside = raw >= std_min && raw <= std_max;
      dlogstd[b * A + i] = inside ? (du * std[b * A + i] * eps[b * A + i] - grad_scale * alpha / (float)B) : 0.f;
    }
  }
  block_sum2(sobj, slp, red);
  if (threadIdx.x == 0) { info[0] = grad_scale * -sobj / (float)B; info[1] = grad_scale * alpha; info[2] = grad_scale * -slp / (float)B; }
}

// dQ seed for the actor pass: every entry -grad_scale/(E*B)
__global__ void fill_kernel(float* x, float v, int n) {
  pdl_prologue();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) x[i] = v;
}

// Temperature loss: L = softplus(lambda) * (entropy - target), entropy = -mean logp'.  dL/dlambda = sigmoid(lambda) * (...)
__global__ void __launch_bounds__(1024) temperature_loss_kernel(const float* __restrict__ logp, const float* __restrict__ lagrange,
                                                                float target_entropy, float grad_scale, float* __restrict__ dlagrange,
                                                                float* __restrict__ info, int B) {
  pdl_prologue();
  __shared__ float red[64];
  float s = 0.f, dummy = 0.f;
  for (int b = threadIdx.x; b < B; b += blockDim.x) s += logp[b];
  block_sum2(s, dummy, red);
  if (threadIdx.x == 0) {
    const float ent = -s / (float)B, lam = lagrange[0];
    info[0] = grad_scale * softplusf(lam) * (ent - target_entropy);
    dlagrange[0] = grad_scale * (1.f / (1.f + expf(-lam))) * (ent - target_entropy);
  }
}

// ---------------------------------------------------------------------------------------------
// Fused optimizer step over the flat trainable buffer.
// Every `update` call ticks all three txs (common.py:142-147).  A trainable leaf whose gradient under a tx is
// identically zero keeps zero moments and a zero update there, so only the txs that ever see a non-zero gradient
// need state: one per leaf, except the proprio-encoder leaves [aux_lo, aux_hi), which the critic loss AND the actor
// loss both differentiate (encoding.py:48-70: stop_gradient covers the image embeddings only) - they carry a second
// (actor-tx) moment pair in the aux tail.  For group gid: g = live ? grad : 0.
//   m = b1 m + (1-b1) g ; v = b2 v + (1-b2) g^2 ; p += -lr_t * (m / (1-b1^t)) / (sqrt(v / (1-b2^t)) + eps)
// then, if polyak: target = p_new * tau + target * (1 - tau)   (common.py:131-133, over the whole tree).
// counts[3] (device, int32) are incremented by the tail thread; lr_t follows optimizers.py:23-29.
// ---------------------------------------------------------------------------------------------
struct AdamArgs {
  float* p; float* target; float* m; float* v; const float* grad;
  int n;
  int seg_end[3];            // flat layout: [0,seg_end[0]) group 0, gap, [seg_end[0]+gap,seg_end[1]) group 1, ...
  int live[3];
  int32_t* counts;           // per group
  float lr[3]; int warmup[3];
  float b1, b2, eps, tau;
  int polyak;
  float* lr_out;             // (3) learning rates actually used (info["*_lr"])
  int gap, aux_lo, aux_hi, aux_off;   // info gap after group 0; leaves with a second (actor-tx) Adam state at [i + aux_off]
};

// one optax adam transform on one element: returns the update -lr * mhat / (sqrt(vhat) + eps)
__device__ inline float adam_update(const AdamArgs& a, int gid, float g, float* mp, float* vp) {
  const int cnt = a.counts[gid];
  const float t = (float)(cnt + 1);
  const float lr = cnt < a.warmup[gid] ? a.lr[gid] * ((float)cnt / (float)a.warmup[gid]) : a.lr[gid];
  const float m = a.b1 * *mp + (1.f - a.b1) * g;
  const float v = a.b2 * *vp + (1.f - a.b2) * g * g;
  *mp = m; *vp = v;
  const float mhat = m / (1.f - powf(a.b1, t));
  const float vhat = v / (1.f - powf(a.b2, t));
  return (mhat / (sqrtf(vhat) + a.eps)) * (-lr);             // optax: scale_by_adam then scale(-lr)
}

__global__ void adam_polyak_kernel(const AdamArgs a) {
  pdl_prologue();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= a.n) return;
  if (i >= a.seg_end[0] && i < a.seg_end[0] + a.gap) return;   // info scalars, not parameters
  const int gid = i < a.seg_end[0] ? 0 : (i < a.seg_end[1] ? 1 : 2);
  float u = adam_update(a, gid, a.live[gid] ? a.grad[i] : 0.f, a.m + i, a.v + i);
  if (i >= a.aux_lo && i < a.aux_hi) {                         // second transform (actor tx); updates summed in tx order actor, critic
    const int j = i + a.aux_off;
    u = adam_update(a, 1, a.live[1] ? a.grad[j] : 0.f, a.m + j, a.v + j) + u;
  }
  const float pn = a.p[i] + u;
  a.p[i] = pn;
  if (a.polyak) a.target[i] = pn * a.tau + a.target[i] * (1.f - a.tau);
}

// ---------------------------------------------------------------------------------------------
// Behaviour cloning (agents/continuous/bc.py:36-76): Dense -> tanh layers of the launcher's BC policy (MLP without LayerNorm,
// utils/launcher.py:26-47) and the loss  -mean_b log N(a_b; mu_b, diag(std_b^2)),  std = clip(exp(log_std), std_min, std_max).
// ---------------------------------------------------------------------------------------------
__global__ void tanh_fwd_kernel(const float* __restrict__ z, float* __restrict__ out, int n) {
  pdl_prologue();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = tanhf(z[i]);
}
__global__ void tanh_bwd_kernel(const float* __restrict__ dt, const float* __restrict__ t, float* __restrict__ dz, int n) {
  pdl_prologue();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) { const float tv = t[i]; dz[i] = dt[i] * (1.f - tv * tv); }
}
// info[0] = actor_loss, info[1] = mse (both * grad_scale: see critic_loss_kernel); one CTA
__global__ void __launch_bounds__(1024) bc_loss_kernel(const float* __restrict__ mu, const float* __restrict__ log_std, const float* __restrict__ act,
                                                       float std_min, float std_max, float grad_scale, float* __restrict__ dmu,
                                                       float* __restrict__ dls, float* __restrict__ info, int B, int A) {
  pdl_prologue();
  __shared__ float red[64];
  float sl = 0.f, sm = 0.f;
  const float inv = grad_scale / (float)B;
  for (int b = threadIdx.x; b < B; b += blockDim.x) {
    float lp = 0.f, se = 0.f;
    for (int j = 0; j < A; ++j) {
      const float m = mu[b * A + j], ls = log_std[b * A + j], a = act[b * A + j];
      const float raw = expf(ls);
      const float sd = fminf(fmaxf(raw, std_min), std_max);
      const float d = a - m, z = d / sd;
      lp += -0.5f * z * z - logf(sd) - 0.918938533204672742f;
      se += d * d;
      dmu[b * A + j] = -(d / (sd * sd)) * inv;                                   // d(-logp)/dmu
      const float dsd = -(d * d / (sd * sd * sd) - 1.f / sd) * inv;               // d(-logp)/dstd
      dls[b * A + j] = (raw > std_min && raw < std_max) ? dsd * raw : 0.f;       // clip passes the gradient strictly inside only
    }
    sl -= lp; sm += se;
  }
  block_sum2(sl, sm, red);
  if (threadIdx.x == 0) { info[0] = sl * inv; info[1] = sm * inv; }
}

// ---------------------------------------------------------------------------------------------
// Reward classifier (examples/async_cable_route_drq/train_reward_classifier.py:122-137): optax.sigmoid_binary_cross_entropy(x, y).mean()
// restated in the stable form relu(x) - x*y + log1p(exp(-|x|)); gradient (sigmoid(x) - y) / B.  Accuracy is the reference's
// predicate (nn.sigmoid(logit) >= 0.5) == label evaluated literally in fp32 on the eval logit: 1 / (1 + expf(-x)) >= 0.5f, which
// holds for every x >= 0 AND for negative x with |x| < ~6e-8 (expf(-x) rounds to 1 there), like the reference's fp32 sigmoid.
// info[0] = loss, info[1] = accuracy (both * grad_scale, see critic_loss_kernel); one CTA, fixed-order reduction (no atomics).
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(1024) bce_logits_loss_kernel(const float* __restrict__ x, const float* __restrict__ xe,
                                                               const float* __restrict__ y, int B, float grad_scale,
                                                               float* __restrict__ dlogit, float* __restrict__ info) {
  pdl_prologue();
  __shared__ float red[64];
  float sl = 0.f, sa = 0.f;
  const float inv = grad_scale / (float)B;
  for (int b = threadIdx.x; b < B; b += blockDim.x) {
    const float v = x[b], lab = y[b];
    sl += fmaxf(v, 0.f) - v * lab + log1pf(expf(-fabsf(v)));
    dlogit[b] = (1.f / (1.f + expf(-v)) - lab) * inv;
    const bool pred = 1.f / (1.f + expf(-xe[b])) >= 0.5f;
    sa += ((pred ? 1.f : 0.f) == lab) ? 1.f : 0.f;
  }
  block_sum2(sl, sa, red);
  if (threadIdx.x == 0) { info[0] = sl * inv; info[1] = sa * inv; }
}

__global__ void adam_tick_kernel(const AdamArgs a) {
  pdl_prologue();
  const int gid = threadIdx.x;
  if (gid < 3) {
    const int cnt = a.counts[gid];
    if (a.lr_out) a.lr_out[gid] = cnt < a.warmup[gid] ? a.lr[gid] * ((float)cnt / (float)a.warmup[gid]) : a.lr[gid];
    a.counts[gid] = cnt + 1;
  }
}

}  // namespace serl

using namespace serl;
#define ST(s) static_cast<cudaStream_t>(s)

extern "C" int serl_rng_schedule(uint32_t* rng_state, uint32_t* keys, int do_aug, int do_update, void* stream) {
  launch_k(rng_schedule_kernel, 1, 32, 0, ST(stream), rng_state, keys, do_aug, do_update);
  return check_launch("rng_schedule_kernel");
}

extern "C" int serl_host_rng_schedule(uint32_t* rng, uint32_t* keys, int do_aug, int do_update) {
  // host mirror of rng_schedule_kernel (same __host__ __device__ primitives) for CPU tests
  u32x2 r{rng[0], rng[1]};
  auto put = [&](int slot, u32x2 k) { keys[2 * slot] = k.x; keys[2 * slot + 1] = k.y; };
  if (do_aug) { put(SERL_KEY_CROP_OBS, jax_split_at(r, 3, 1)); put(SERL_KEY_CROP_NEXT, jax_split_at(r, 3, 2)); r = jax_split_at(r, 3, 0); }
  if (do_update) {
    const u32x2 k_actor = jax_split_at(r, 4, 1), k_critic = jax_split_at(r, 4, 2), k_temp = jax_split_at(r, 4, 3);
    const u32x2 c1 = jax_split_at(k_critic, 2, 0);
    put(SERL_KEY_CRITIC_NEXT, jax_split_at(k_critic, 2, 1));
    put(SERL_KEY_CRITIC_SUBSAMPLE, jax_split_at(c1, 2, 1));
    put(SERL_KEY_ACTOR_DROPOUT, jax_split_at(k_actor, 4, 1));
    put(SERL_KEY_ACTOR_SAMPLE, jax_split_at(k_actor, 4, 2));
    put(SERL_KEY_TEMP_NEXT, jax_split_at(k_temp, 2, 1));
    r = jax_split_at(r, 2, 0);
  }
  rng[0] = r.x; rng[1] = r.y;
  return SERL_OK;
}

extern "C" int serl_normal_fill(const uint32_t* key, float* out, int n, void* stream) {
  launch_k(normal_fill_kernel, ceil_div(n, 128), 128, 0, ST(stream), key, out, n);
  return check_launch("normal_fill_kernel");
}

extern "C" int serl_dropout_mask_fill(const uint32_t* key, uint32_t fold, float keep, uint8_t* mask, int n, void* stream) {
  launch_k(dropout_mask_kernel, ceil_div(n, 256), 256, 0, ST(stream), key, fold, keep, mask, n);
  return check_launch("dropout_mask_kernel");
}

extern "C" int serl_subsample_idx(const uint32_t* key, int ensemble, int32_t* out, int n, void* stream) {
  if (n < 1 || n > 32 || ensemble < 1 || ensemble > 65535) { set_last_error("serl_subsample_idx: need 1 <= n <= 32, 1 <= ensemble < 65536"); return SERL_ERR_INVALID; }
  launch_k(subsample_idx_kernel, 1, 32, 0, ST(stream), key, ensemble, out, n);
  return check_launch("subsample_idx_kernel");
}

extern "C" int serl_tanh_gaussian_fwd(const float* mu, const float* log_std, const float* eps, float std_min, float std_max,
                                      float* act, int ld_act, float* logp, float* u_out, float* std_out, int B, int A,
                                      int deterministic, void* stream) {
  if (!deterministic && !eps) { set_last_error("serl_tanh_gaussian_fwd: eps required unless deterministic"); return SERL_ERR_INVALID; }
  launch_k(tanh_gaussian_fwd_kernel, ceil_div(B, 128), 128, 0, ST(stream), mu, log_std, eps, std_min, std_max, act, ld_act, logp, u_out,
                                                                    std_out, B, A, deterministic);
  return check_launch("tanh_gaussian_fwd_kernel");
}

extern "C" int serl_critic_loss(const float* q, const float* q_next, const int32_t* sub, int n_sub, const float* rewards,
                                const float* masks, const float* logp_next, const float* lagrange, int backup_entropy,
                                float gamma, float grad_scale, float* target_q, float* dq, float* info, int E, int B, void* stream) {
  launch_k(critic_loss_kernel, 1, 1024, 0, ST(stream), q, q_next, sub, n_sub, rewards, masks, logp_next, lagrange, backup_entropy, gamma,
                                                 grad_scale, target_q, dq, info, E, B);
  return check_launch("critic_loss_kernel");
}

extern "C" int serl_fill_f32(float* x, float v, int n, void* stream) {
  launch_k(fill_kernel, ceil_div(n, 256), 256, 0, ST(stream), x, v, n);
  return check_launch("fill_kernel");
}

extern "C" int serl_actor_loss(const float* q, const float* logp, const float* lagrange, const float* da, int ld_da,
                               const float* act, int ld_act, const float* std, const float* log_std, const float* eps,
                               float std_min, float std_max, float grad_scale, float* dmu, float* dlogstd, float* info,
                               int E, int B, int A, void* stream) {
  launch_k(actor_loss_kernel, 1, 1024, 0, ST(stream), q, logp, lagrange, da, ld_da, act, ld_act, std, log_std, eps, std_min, std_max,
                                                grad_scale, dmu, dlogstd, info, E, B, A);
  return check_launch("actor_loss_kernel");
}

extern "C" int serl_temperature_loss(const float* logp, const float* lagrange, float target_entropy, float grad_scale,
                                     float* dlagrange, float* info, int B, void* stream) {
  launch_k(temperature_loss_kernel, 1, 1024, 0, ST(stream), logp, lagrange, target_entropy, grad_scale, dlagrange, info, B);
  return check_launch("temperature_loss_kernel");
}

extern "C" int serl_tanh_fwd(const float* z, float* out, int n, void* stream) {
  launch_k(tanh_fwd_kernel, ceil_div(n, 256), 256, 0, ST(stream), z, out, n);
  return check_launch("tanh_fwd_kernel");
}
extern "C" int serl_tanh_bwd(const float* dt, const float* t, float* dz, int n, void* stream) {
  launch_k(tanh_bwd_kernel, ceil_div(n, 256), 256, 0, ST(stream), dt, t, dz, n);
  return check_launch("tanh_bwd_kernel");
}
extern "C" int serl_bc_loss(const float* mu, const float* log_std, const float* actions, float std_min, float std_max, float grad_scale,
                            float* dmu, float* dlogstd, float* info, int B, int A, void* stream) {
  if (!mu || !log_std || !actions || !dmu || !dlogstd || !info || B < 1 || A < 1) { set_last_error("serl_bc_loss: invalid arguments"); return SERL_ERR_INVALID; }
  launch_k(bc_loss_kernel, 1, 1024, 0, ST(stream), mu, log_std, actions, std_min, std_max, grad_scale, dmu, dlogstd, info, B, A);
  return check_launch("bc_loss_kernel");
}

extern "C" int serl_adam_polyak(const serl_adam_desc* d, void* stream) {
  if (!d || d->n < 1 || !d->params || !d->m || !d->v || !d->grad || !d->counts) { set_last_error("serl_adam_polyak: invalid descriptor"); return SERL_ERR_INVALID; }
  if (d->polyak && !d->target) { set_last_error("serl_adam_polyak: polyak needs target"); return SERL_ERR_INVALID; }
  AdamArgs a{};
  a.p = d->params; a.target = d->target; a.m = d->m; a.v = d->v; a.grad = d->grad; a.n = d->n; a.counts = d->counts;
  for (int g = 0; g < 3; ++g) { a.seg_end[g] = d->seg_end[g]; a.live[g] = d->live[g]; a.lr[g] = d->lr[g]; a.warmup[g] = d->warmup[g]; }
  a.b1 = d->b1; a.b2 = d->b2; a.eps = d->eps; a.tau = d->tau; a.polyak = d->polyak; a.lr_out = d->lr_out;
  a.gap = d->gap; a.aux_lo = d->aux_lo; a.aux_hi = d->aux_hi; a.aux_off = d->aux_off;
  if (a.gap < 0 || a.aux_lo > a.aux_hi || (a.aux_hi > a.aux_lo && (a.aux_lo < 0 || a.aux_hi > d->seg_end[0] || a.aux_lo + a.aux_off < d->n))) {
    set_last_error("serl_adam_polyak: invalid gap / aux range"); return SERL_ERR_INVALID;
  }
  launch_k(adam_polyak_kernel, ceil_div(d->n, 256), 256, 0, ST(stream), a);
  if (int e = check_launch("adam_polyak_kernel")) return e;
  launch_k(adam_tick_kernel, 1, 32, 0, ST(stream), a);
  return check_launch("adam_tick_kernel");
}

extern "C" int serl_bce_logits_loss(const float* logits, const float* eval_logits, const float* labels, int B, float grad_scale,
                                    float* dlogit, float* info, void* stream) {
  if (!logits || !eval_logits || !labels || !dlogit || !info || B < 1) { set_last_error("serl_bce_logits_loss: invalid arguments"); return SERL_ERR_INVALID; }
  launch_k(bce_logits_loss_kernel, 1, 1024, 0, ST(stream), logits, eval_logits, labels, B, grad_scale, dlogit, info);
  return check_launch("bce_logits_loss_kernel");
}
