// minppo_b200 -- the PPO loss of one minibatch row and its hand-derived gradient seeds (train.py:218-243; oracle/ppo_numpy.py),
// shared by fused_step.cuh and head_loss.cu, and the Gaussian log-density term shared with the policy kernels.
#pragma once

#include "common.cuh"

namespace minppo {

// d/dx min(max(x, lo), hi) with the 0.5/0.5 tie split of jnp.minimum / jnp.maximum
MINPPO_DEVINL float dclip(float x, float lo, float hi) {
  return (x > lo && x < hi) ? 1.f : ((x == lo || x == hi) ? 0.5f : 0.f);
}

// distrax: log N(z; 0, 1) of one action component; a row's log-prob is their sum minus sum log|scale| (train.py:160, 223)
MINPPO_DEVINL float gauss_logp_term(float z) {
  constexpr float HALF_LOG_2PI = 0.91893853320467274178f;
  return -0.5f * z * z - HALF_LOG_2PI;
}

// clipped surrogate: loss = min(l1, l2), g_logp = dL/dlogp; logr and ratio feed the statistics sums.  adv_raw is the row's
// advantage, normalised with the minibatch sums adv_sum and adv_sq; inv_n = 1 / minibatch size.
struct PpoActorRow { float loss, g_logp, logr, ratio; };
MINPPO_DEVINL PpoActorRow ppo_actor_row(float logp, float logp_old, float adv_raw, float adv_sum, float adv_sq, float inv_n,
                                        float clip_eps) {
  const float logr = logp - logp_old;
  const float ratio = expf(logr);                                              // train.py:234
  const float adv_mean = adv_sum * inv_n;
  const float adv_std = sqrtf(adv_sq * inv_n);
  const float adv = (adv_raw - adv_mean) / (adv_std + 1e-8f);                  // train.py:235
  const float lo = 1.f - clip_eps, hi = 1.f + clip_eps;
  const float l1 = ratio * adv;
  const float l2 = fminf(fmaxf(ratio, lo), hi) * adv;                          // train.py:237
  const float loss = fminf(l1, l2);                                            // train.py:238
  const float w1 = l1 < l2 ? 1.f : (l1 == l2 ? 0.5f : 0.f);
  const float dmin = (w1 + (1.f - w1) * dclip(ratio, lo, hi)) * adv;
  return {loss, -inv_n * dmin * ratio, logr, ratio};
}

// clipped value loss, train.py:226-231: loss = max(vl, vlc), g_v = dL/dv; dv = v - v_old feeds the statistics sums
struct PpoValueRow { float loss, g_v, dv; };
MINPPO_DEVINL PpoValueRow ppo_value_row(float v, float v_old, float tgt, float inv_n, float clip_eps, float vf_coef) {
  const float dv = v - v_old;
  const float v_clip = v_old + fminf(fmaxf(dv, -clip_eps), clip_eps);
  const float e1 = v - tgt, e2 = v_clip - tgt;
  const float vl = e1 * e1, vlc = e2 * e2;
  const float loss = fmaxf(vl, vlc);
  const float wa = vl > vlc ? 1.f : (vl == vlc ? 0.5f : 0.f);
  return {loss, vf_coef * 0.5f * inv_n * (wa * 2.f * e1 + (1.f - wa) * 2.f * e2 * dclip(dv, -clip_eps, clip_eps)), dv};
}

// terms of the statistics sums (LOSS_SUMS [2..4]); approx-KL (r - 1) - log r as expm1: no cancellation at small log r
MINPPO_DEVINL float approx_kl_term(float logr) { return expm1f(logr) - logr; }
MINPPO_DEVINL float ratio_clipped(float ratio, float clip_eps) { return fabsf(ratio - 1.f) > clip_eps ? 1.f : 0.f; }
MINPPO_DEVINL float value_clipped(float dv, float clip_eps) { return fabsf(dv) > clip_eps ? 1.f : 0.f; }

}  // namespace minppo
