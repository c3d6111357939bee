// minppo_b200 -- output heads + PPO loss + backward seed (replaces the tail of
// ActorCritic.__call__ and all of _loss_fn, /root/reference/minppo/train.py:78-83, 218-243,
// and the part of jax.value_and_grad (train.py:246) that touches the heads).
//
// Per 64-row tile of the minibatch (rows = gathered transitions), fp32 SIMT:
//   mean = h_a W3a + b3a ; v = h_c W3c + b3c                       (heads, N = A and 1)
//   logp, ratio, clipped surrogate, clipped value loss              (train.py:223-239)
//   g_mean = dL/dmean, g_v = dL/dv, dL/dlog_std                      (hand-derived; oracle/ppo_numpy.py)
//   dZ_a = (g_mean W3a^T) * f'(h_a), dZ_c = (g_v W3c^T) * f'(h_c)   -> bf16, feeds the tcgen05 GEMMs
//   per-tile partial sums of dW3, db3, db of the last hidden layer, dlog_std and the loss terms
// Partials are written per tile (no atomics) and reduced in fixed order by the optimizer kernel.
//
// Rows >= count (padding of the last 128-row GEMM tile, or rows another GPU owns) produce
// exact zeros everywhere.
#include "common.cuh"
#include "minppo_internal.h"

namespace minppo {

constexpr int HL_ROWS = 64;
constexpr int HL_THREADS = 256;

MINPPO_DEVINL float dclip(float x, float lo, float hi) {
  // d/dx min(max(x, lo), hi) with the 0.5/0.5 tie split of jnp.minimum / jnp.maximum
  return (x > lo && x < hi) ? 1.f : ((x == lo || x == hi) ? 0.5f : 0.f);
}

template <int AMAX>
__global__ void __launch_bounds__(HL_THREADS) head_loss_kernel(const HeadLossArgs a) {
  extern __shared__ __align__(16) uint8_t hl_smem[];
  const int H = a.H, A = a.A;
  const int HS = H + 8;                        // padded bf16 row stride
  __nv_bfloat16* hA = reinterpret_cast<__nv_bfloat16*>(hl_smem);
  __nv_bfloat16* hC = hA + HL_ROWS * HS;
  float* w3a = reinterpret_cast<float*>(hC + HL_ROWS * HS);       // [H][AMAX+1]
  float* w3c = w3a + H * (AMAX + 1);                              // [H]
  float* gm = w3c + H;                                            // [64][AMAX]  g_mean
  float* gv = gm + HL_ROWS * AMAX;                                // [64]
  float* red = gv + HL_ROWS;                                      // [8][AMAX + 4] warp partials

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int tile = blockIdx.x;
  const int row0 = tile * HL_ROWS;
  const int count = min(*a.count, a.cap);
  const float* P = a.params;

  // ---- stage weights and the two activation tiles --------------------------------------
  for (int i = tid; i < H * AMAX; i += HL_THREADS) {
    const int k = i / AMAX, j = i % AMAX;
    w3a[k * (AMAX + 1) + j] = j < A ? P[a.off_w3a + k * A + j] : 0.f;
  }
  for (int i = tid; i < H; i += HL_THREADS) w3c[i] = P[a.off_w3c + i];
  {
    const int chunks = H / 8;                                      // 16-byte chunks per row
    for (int i = tid; i < HL_ROWS * chunks; i += HL_THREADS) {
      const int r = i / chunks, c = i % chunks;
      const uint4 va = *reinterpret_cast<const uint4*>(a.h_a + static_cast<size_t>(row0 + r) * a.ldh + c * 8);
      const uint4 vc = *reinterpret_cast<const uint4*>(a.h_c + static_cast<size_t>(row0 + r) * a.ldh + c * 8);
      *reinterpret_cast<uint4*>(hA + r * HS + c * 8) = va;
      *reinterpret_cast<uint4*>(hC + r * HS + c * 8) = vc;
    }
  }
  __syncthreads();

  // ---- phase 1: heads.  4 threads per row, k interleaved in pairs across the quad ---------
  const int r = tid >> 2, part = tid & 3;
  float acc[AMAX];
  float accv = 0.f;
#pragma unroll
  for (int j = 0; j < AMAX; ++j) acc[j] = 0.f;
  for (int k0 = part * 2; k0 < H; k0 += 8) {
    const uint32_t wa = *reinterpret_cast<const uint32_t*>(hA + r * HS + k0);
    const uint32_t wc = *reinterpret_cast<const uint32_t*>(hC + r * HS + k0);
    const float a0 = bf16_lo(wa), a1 = bf16_hi(wa);
    const float* w0 = w3a + k0 * (AMAX + 1);
    const float* w1 = w0 + (AMAX + 1);
#pragma unroll
    for (int j = 0; j < AMAX; ++j) acc[j] = fmaf(a1, w1[j], fmaf(a0, w0[j], acc[j]));
    accv = fmaf(bf16_hi(wc), w3c[k0 + 1], fmaf(bf16_lo(wc), w3c[k0], accv));
  }
#pragma unroll
  for (int j = 0; j < AMAX; ++j) {
    acc[j] += __shfl_xor_sync(0xffffffffu, acc[j], 1);
    acc[j] += __shfl_xor_sync(0xffffffffu, acc[j], 2);
  }
  accv += __shfl_xor_sync(0xffffffffu, accv, 1);
  accv += __shfl_xor_sync(0xffffffffu, accv, 2);

  // ---- phase 2: loss and gradient seeds, one thread per row (part == 0) -------------------
  float dls[AMAX];                       // this row's contribution to d/dlog_std
  float s_val = 0.f, s_act = 0.f;
#pragma unroll
  for (int j = 0; j < AMAX; ++j) dls[j] = 0.f;
  const int grow = row0 + r;
  const bool live = (part == 0) && (grow < count);
  if (part == 0) {
    float g_mean[AMAX];
    float g_v = 0.f;
#pragma unroll
    for (int j = 0; j < AMAX; ++j) g_mean[j] = 0.f;
    if (live) {
      const int src = a.rowidx[grow];
      const float inv_n = a.inv_mb;
      // distrax: z = (a - loc) * (1/scale); log_prob = sum(-z^2/2 - log(2pi)/2) - sum(log|scale|)
      float z[AMAX], inv_s[AMAX];
      float quad = 0.f, logdet = 0.f;
#pragma unroll
      for (int j = 0; j < AMAX; ++j) {
        if (j < A) {
          const float scale = expf(P[a.off_logstd + j]);
          inv_s[j] = 1.f / scale;
          const float mean = acc[j] + P[a.off_b3a + j];
          z[j] = (a.action[static_cast<size_t>(src) * A + j] - mean) * inv_s[j];
          quad += -0.5f * z[j] * z[j] - 0.91893853320467274178f;
          logdet += logf(fabsf(scale));
        } else { z[j] = 0.f; inv_s[j] = 0.f; }
      }
      const float logp = quad - logdet;
      const float ratio = expf(logp - a.logp_old[src]);                          // train.py:234
      const float adv_mean = (*a.adv_sum) * inv_n;
      const float adv_std = sqrtf((*a.adv_sq) * inv_n);
      const float adv = (a.adv[src] - adv_mean) / (adv_std + 1e-8f);             // train.py:235
      const float lo = 1.f - a.clip_eps, hi = 1.f + a.clip_eps;
      const float l1 = ratio * adv;
      const float l2 = fminf(fmaxf(ratio, lo), hi) * adv;                        // train.py:237
      s_act = fminf(l1, l2);                                                     // train.py:238
      const float w1 = l1 < l2 ? 1.f : (l1 == l2 ? 0.5f : 0.f);
      const float dmin = (w1 + (1.f - w1) * dclip(ratio, lo, hi)) * adv;
      const float g_logp = -inv_n * dmin * ratio;
#pragma unroll
      for (int j = 0; j < AMAX; ++j) {
        g_mean[j] = g_logp * (z[j] * inv_s[j]);
        dls[j] = g_logp * (z[j] * z[j] - 1.f);
      }
      // value loss, train.py:226-231
      const float v = accv + P[a.off_b3c];
      const float v_old = a.v_old[src], tgt = a.tgt[src];
      const float dvv = v - v_old;
      const float v_clip = v_old + fminf(fmaxf(dvv, -a.clip_eps), a.clip_eps);
      const float e1 = v - tgt, e2 = v_clip - tgt;
      const float vl = e1 * e1, vlc = e2 * e2;
      s_val = fmaxf(vl, vlc);
      const float wa = vl > vlc ? 1.f : (vl == vlc ? 0.5f : 0.f);
      g_v = a.vf_coef * 0.5f * inv_n * (wa * 2.f * e1 + (1.f - wa) * 2.f * e2 * dclip(dvv, -a.clip_eps, a.clip_eps));
    }
#pragma unroll
    for (int j = 0; j < AMAX; ++j) gm[r * AMAX + j] = g_mean[j];
    gv[r] = g_v;
  }
  // reduce loss sums and dlog_std over the tile (fixed order: lanes, then warps)
#pragma unroll
  for (int j = 0; j < AMAX; ++j) dls[j] = warp_sum(dls[j]);
  s_val = warp_sum(s_val);
  s_act = warp_sum(s_act);
  if (lane == 0) {
#pragma unroll
    for (int j = 0; j < AMAX; ++j) red[warp * (AMAX + 4) + j] = dls[j];
    red[warp * (AMAX + 4) + AMAX] = s_val;
    red[warp * (AMAX + 4) + AMAX + 1] = s_act;
  }
  __syncthreads();

  float* part_out = a.partials + static_cast<size_t>(tile) * a.partial_stride;
  if (tid < AMAX + 2) {
    float s = 0.f;
    for (int w = 0; w < HL_THREADS / 32; ++w) s += red[w * (AMAX + 4) + tid];
    if (tid < A) part_out[a.po_logstd + tid] = s;
    else if (tid == AMAX) part_out[a.po_loss + 0] = s;
    else if (tid == AMAX + 1) part_out[a.po_loss + 1] = s;
  }
  // head bias grads: db3a[j] = sum_r g_mean[r][j], db3c = sum_r g_v[r]
  if (tid < A + 1) {
    float s = 0.f;
    if (tid < A) { for (int rr = 0; rr < HL_ROWS; ++rr) s += gm[rr * AMAX + tid]; part_out[a.po_b3a + tid] = s; }
    else { for (int rr = 0; rr < HL_ROWS; ++rr) s += gv[rr]; part_out[a.po_b3c] = s; }
  }

  // ---- phase 3: thread = hidden column c.  dZ tiles, dW3, bias grads of the last hidden layer
  for (int c = tid; c < H; c += HL_THREADS) {
    float w[AMAX], dw[AMAX];
#pragma unroll
    for (int j = 0; j < AMAX; ++j) { w[j] = w3a[c * (AMAX + 1) + j]; dw[j] = 0.f; }
    const float wc = w3c[c];
    float dwc = 0.f, dba = 0.f, dbc = 0.f;
    for (int rr = 0; rr < HL_ROWS; ++rr) {
      const float ha = __bfloat162float(hA[rr * HS + c]);
      const float hc = __bfloat162float(hC[rr * HS + c]);
      float da = 0.f;
#pragma unroll
      for (int j = 0; j < AMAX; ++j) {
        const float g = gm[rr * AMAX + j];
        da = fmaf(g, w[j], da);
        dw[j] = fmaf(ha, g, dw[j]);
      }
      const float g_v = gv[rr];
      dwc = fmaf(hc, g_v, dwc);
      const float fa = a.act_a == ACTK_RELU ? (ha > 0.f ? 1.f : 0.f) : (1.f - ha * ha);
      const float fc = a.act_c == ACTK_RELU ? (hc > 0.f ? 1.f : 0.f) : (1.f - hc * hc);
      const __nv_bfloat16 za = __float2bfloat16_rn(da * fa);
      const __nv_bfloat16 zc = __float2bfloat16_rn(g_v * wc * fc);
      a.dz_a[static_cast<size_t>(row0 + rr) * a.ldh + c] = za;
      a.dz_c[static_cast<size_t>(row0 + rr) * a.ldh + c] = zc;
      dba += __bfloat162float(za);
      dbc += __bfloat162float(zc);
    }
#pragma unroll
    for (int j = 0; j < AMAX; ++j)
      if (j < A) part_out[a.po_w3a + c * A + j] = dw[j];
    part_out[a.po_w3c + c] = dwc;
    part_out[a.po_bh_a + c] = dba;
    part_out[a.po_bh_c + c] = dbc;
  }
}

size_t head_loss_smem_bytes(int H, int amax) {
  return static_cast<size_t>(2) * HL_ROWS * (H + 8) * 2 + static_cast<size_t>(H) * (amax + 1) * 4 + H * 4 +
         HL_ROWS * amax * 4 + HL_ROWS * 4 + 8 * (amax + 4) * 4 + 64;
}

int head_loss_init() {
  // H = 512 with the 32-wide template: 212,416 bytes (above 200 KB, below the 227 KB a block may opt in to)
  const int smax = static_cast<int>(head_loss_smem_bytes(MAX_HIDDEN, 32));
  cudaError_t e = cudaFuncSetAttribute(head_loss_kernel<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, smax);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(head_loss_kernel<16>, cudaFuncAttributeMaxDynamicSharedMemorySize, smax);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(head_loss_kernel<32>, cudaFuncAttributeMaxDynamicSharedMemorySize, smax);
  return e == cudaSuccess ? 0 : MINPPO_ERR_CUDA;
}

int head_loss_launch(const HeadLossArgs& a, int tiles, cudaStream_t stream) {
  if (a.A > 32) return MINPPO_ERR_ARG;
  const int amax = a.A <= 8 ? 8 : (a.A <= 16 ? 16 : 32);
  const size_t smem = head_loss_smem_bytes(a.H, amax);
  if (amax == 8) head_loss_kernel<8><<<tiles, HL_THREADS, smem, stream>>>(a);
  else if (amax == 16) head_loss_kernel<16><<<tiles, HL_THREADS, smem, stream>>>(a);
  else head_loss_kernel<32><<<tiles, HL_THREADS, smem, stream>>>(a);
  return cudaGetLastError() == cudaSuccess ? 0 : MINPPO_ERR_CUDA;
}

}  // namespace minppo
