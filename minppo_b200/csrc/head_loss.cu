// minppo_b200 -- output heads + PPO loss + backward seed (replaces the tail of
// ActorCritic.__call__ and all of _loss_fn, /root/reference/minppo/train.py:78-83, 218-243,
// and the part of jax.value_and_grad (train.py:246) that touches the heads).
//
// Per 64-row tile of the minibatch (rows = gathered transitions), fp32 SIMT:
//   mean = h_a W3a + b3a ; v = h_c W3c + b3c                       (heads, N = A and 1)
//   logp, ratio, clipped surrogate, clipped value loss              (train.py:223-239)
//   g_mean = dL/dmean, g_v = dL/dv, dL/dlog_std                      (hand-derived; oracle/ppo_numpy.py)
//   dZ_a = (g_mean W3a^T) * f'(h_a), dZ_c = (g_v W3c^T) * f'(h_c)   -> bf16, feeds the tcgen05 GEMMs
//   per-tile partial sums of dW3, db3, dlog_std, the loss terms and the statistics sums (LOSS_SUMS)
// Partials are written per tile (no atomics) and reduced in fixed order by the optimizer kernel.
//
// Rows >= count (padding of the last 128-row GEMM tile, or rows another GPU owns) produce
// exact zeros everywhere.
//
// AMAX = 64 (act_dim 33..64): the whole fp32 head kernel W3a (H x 65 floats) does not fit beside the two activation
// tiles at H > 384, so phase 1 stages it HL_KCHUNK rows at a time, and phase 3 reads each thread's row of it from the
// arena.  Every thread accumulates the same terms in the same order as with the whole kernel resident.
#include "common.cuh"
#include "minppo_internal.h"
#include "ppo_math.cuh"

namespace minppo {

constexpr int HL_ROWS = 64;
constexpr int HL_THREADS = 256;
constexpr int HL_KCHUNK = 256;          // rows of W3a per phase-1 stage (AMAX > 32)
static_assert(HL_KCHUNK % 8 == 0, "phase 1 steps k by 8 across a quad");

// rows [k0, k0 + rows) of the head kernel W3a -> w3a[rows][AMAX + 1], columns >= A zero
template <int AMAX>
MINPPO_DEVINL void hl_stage_w3a(float* w3a, const float* P, int off_w3a, int A, int k0, int rows, int tid) {
  for (int i = tid; i < rows * AMAX; i += HL_THREADS) {
    const int k = i / AMAX, j = i % AMAX;
    w3a[k * (AMAX + 1) + j] = j < A ? P[off_w3a + (k0 + k) * A + j] : 0.f;
  }
}

template <int AMAX>
__global__ void __launch_bounds__(HL_THREADS) head_loss_kernel(const HeadLossArgs a) {
  extern __shared__ __align__(16) uint8_t hl_smem[];
  constexpr bool CHUNKED = AMAX > 32;
  const int H = a.H, A = a.A;
  const int HS = H + 8;                        // padded bf16 row stride
  __nv_bfloat16* hA = reinterpret_cast<__nv_bfloat16*>(hl_smem);
  __nv_bfloat16* hC = hA + HL_ROWS * HS;
  float* w3a = reinterpret_cast<float*>(hC + HL_ROWS * HS);       // [H][AMAX+1]  (AMAX > 32: [HL_KCHUNK][AMAX+1])
  float* w3c = w3a + (CHUNKED ? HL_KCHUNK : H) * (AMAX + 1);       // [H]
  float* gm = w3c + H;                                            // [64][AMAX]  g_mean
  float* gv = gm + HL_ROWS * AMAX;                                // [64]
  float* red = gv + HL_ROWS;                                      // [8][AMAX + 8] warp partials: dlog_std, then LOSS_SUMS

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int tile = blockIdx.x;
  const int row0 = tile * HL_ROWS;
  const LossOperands& L = a.loss;
  const int32_t* rowidx_s = L.rowidx + static_cast<size_t>(L.step) * L.cap;   // this step's row list
  const int count = min(L.count[L.step], L.cap);
  const float* P = a.params;

  // ---- stage weights and the two activation tiles --------------------------------------
  // (the AMAX <= 32 loops are kept as they are rather than shared with the chunked ones: sharing them changes the
  // compiled code of the instances every act_dim <= 32 runs)
  if constexpr (CHUNKED) {
    hl_stage_w3a<AMAX>(w3a, P, a.off.w3a, A, 0, min(H, HL_KCHUNK), tid);
  } else {
    for (int i = tid; i < H * AMAX; i += HL_THREADS) {
      const int k = i / AMAX, j = i % AMAX;
      w3a[k * (AMAX + 1) + j] = j < A ? P[a.off.w3a + k * A + j] : 0.f;
    }
  }
  for (int i = tid; i < H; i += HL_THREADS) w3c[i] = P[a.off.w3c + i];
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
  if constexpr (CHUNKED) {
    for (int kc = 0; kc < H; kc += HL_KCHUNK) {              // the same k sequence per thread, one stage at a time
      if (kc > 0) {
        __syncthreads();
        hl_stage_w3a<AMAX>(w3a, P, a.off.w3a, A, kc, min(H - kc, HL_KCHUNK), tid);
        __syncthreads();
      }
      for (int k0 = kc + part * 2; k0 < min(H, kc + HL_KCHUNK); k0 += 8) {
        const uint32_t wa = *reinterpret_cast<const uint32_t*>(hA + r * HS + k0);
        const uint32_t wc = *reinterpret_cast<const uint32_t*>(hC + r * HS + k0);
        const float a0 = bf16_lo(wa), a1 = bf16_hi(wa);
        const float* w0 = w3a + (k0 - kc) * (AMAX + 1);
        const float* w1 = w0 + (AMAX + 1);
#pragma unroll
        for (int j = 0; j < AMAX; ++j) acc[j] = fmaf(a1, w1[j], fmaf(a0, w0[j], acc[j]));
        accv = fmaf(bf16_hi(wc), w3c[k0 + 1], fmaf(bf16_lo(wc), w3c[k0], accv));
      }
    }
  } else {
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
  float s_val = 0.f, s_act = 0.f, s_vclip = 0.f, s_kl = 0.f, s_clip = 0.f;   // the LOSS_SUMS terms of this row
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
      const int src = rowidx_s[grow];
      float z[AMAX], inv_s[AMAX];
      float quad = 0.f, logdet = 0.f;
#pragma unroll
      for (int j = 0; j < AMAX; ++j) {
        if (j < A) {
          const float scale = expf(P[a.off.logstd + j]);
          inv_s[j] = 1.f / scale;
          const float mean = acc[j] + P[a.off.b3a + j];
          z[j] = (L.action[static_cast<size_t>(src) * A + j] - mean) * inv_s[j];
          quad += gauss_logp_term(z[j]);
          logdet += logf(fabsf(scale));
        } else { z[j] = 0.f; inv_s[j] = 0.f; }
      }
      const PpoActorRow ar = ppo_actor_row(quad - logdet, L.logp_old[src], L.adv[src], L.adv_sum[L.step], L.adv_sq[L.step],
                                           L.inv_mb, L.clip_eps);
      s_act = ar.loss; s_kl = approx_kl_term(ar.logr); s_clip = ratio_clipped(ar.ratio, L.clip_eps);
#pragma unroll
      for (int j = 0; j < AMAX; ++j) {
        g_mean[j] = ar.g_logp * (z[j] * inv_s[j]);
        dls[j] = ar.g_logp * (z[j] * z[j] - 1.f);
      }
      const PpoValueRow vr = ppo_value_row(accv + P[a.off.b3c], L.v_old[src], L.tgt[src], L.inv_mb, L.clip_eps, L.vf_coef);
      s_val = vr.loss; s_vclip = value_clipped(vr.dv, L.clip_eps); g_v = vr.g_v;
    }
#pragma unroll
    for (int j = 0; j < AMAX; ++j) gm[r * AMAX + j] = g_mean[j];
    gv[r] = g_v;
  }
  // reduce loss sums and dlog_std over the tile (fixed order: lanes, then warps)
#pragma unroll
  for (int j = 0; j < AMAX; ++j) dls[j] = warp_sum(dls[j]);
  const float sums[LOSS_SUMS] = {warp_sum(s_val), warp_sum(s_act), warp_sum(s_vclip), warp_sum(s_kl), warp_sum(s_clip)};
  if (lane == 0) {
#pragma unroll
    for (int j = 0; j < AMAX; ++j) red[warp * (AMAX + 8) + j] = dls[j];
#pragma unroll
    for (int j = 0; j < LOSS_SUMS; ++j) red[warp * (AMAX + 8) + AMAX + j] = sums[j];
  }
  __syncthreads();

  float* part_out = a.partials + static_cast<size_t>(tile) * a.partial_stride;
  if (tid < AMAX + LOSS_SUMS) {
    float s = 0.f;
    for (int w = 0; w < HL_THREADS / 32; ++w) s += red[w * (AMAX + 8) + tid];
    if (tid < A) part_out[a.po_logstd + tid] = s;
    else if (tid >= AMAX) part_out[a.po_loss + tid - AMAX] = s;
  }
  // head bias grads: db3a[j] = sum_r g_mean[r][j], db3c = sum_r g_v[r]
  if (tid < A + 1) {
    float s = 0.f;
    if (tid < A) { for (int rr = 0; rr < HL_ROWS; ++rr) s += gm[rr * AMAX + tid]; part_out[a.po_b3a + tid] = s; }
    else { for (int rr = 0; rr < HL_ROWS; ++rr) s += gv[rr]; part_out[a.po_b3c] = s; }
  }

  // ---- phase 3: thread = hidden column c.  dZ tiles, dW3
  // (AMAX > 32: row c of W3a read from the arena, which stays in L2; shared memory holds only a k-chunk of it)
  for (int c = tid; c < H; c += HL_THREADS) {
    float w[AMAX], dw[AMAX];
#pragma unroll
    for (int j = 0; j < AMAX; ++j) {
      if constexpr (CHUNKED) w[j] = j < A ? __ldg(P + a.off.w3a + c * A + j) : 0.f;
      else w[j] = w3a[c * (AMAX + 1) + j];
      dw[j] = 0.f;
    }
    const float wc = w3c[c];
    float dwc = 0.f;
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
    }
#pragma unroll
    for (int j = 0; j < AMAX; ++j)
      if (j < A) part_out[a.po_w3a + c * A + j] = dw[j];
    part_out[a.po_w3c + c] = dwc;
  }
}

constexpr size_t head_loss_smem_bytes(int H, int amax) {
  return static_cast<size_t>(2) * HL_ROWS * (H + 8) * 2 +
         static_cast<size_t>(amax > 32 ? HL_KCHUNK : H) * (amax + 1) * 4 + H * 4 +
         HL_ROWS * amax * 4 + HL_ROWS * 4 + 8 * (amax + 8) * 4 + 64;
}
static_assert(LOSS_SUMS <= 8, "head_loss_kernel: the loss sums share the 8 spare floats of a warp's row of red");
// H = 512: 212,544 bytes with the 32-wide template, 220,736 with the 64-wide one (its W3a staged in 256-row chunks):
// above 200 KB, within the 227 KB a block may opt in to
constexpr int HL_SMEM_OPTIN = 227 * 1024;
static_assert(head_loss_smem_bytes(MAX_HIDDEN, 32) <= HL_SMEM_OPTIN, "head_loss_kernel<32> shared memory at H = 512");
static_assert(head_loss_smem_bytes(MAX_HIDDEN, 64) <= HL_SMEM_OPTIN, "head_loss_kernel<64> shared memory at H = 512");

int head_loss_init() {
  const int smax = static_cast<int>(head_loss_smem_bytes(MAX_HIDDEN, 32));
  cudaError_t e = cudaFuncSetAttribute(head_loss_kernel<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, smax);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(head_loss_kernel<16>, cudaFuncAttributeMaxDynamicSharedMemorySize, smax);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(head_loss_kernel<32>, cudaFuncAttributeMaxDynamicSharedMemorySize, smax);
  if (e == cudaSuccess)
    e = cudaFuncSetAttribute(head_loss_kernel<64>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                             static_cast<int>(head_loss_smem_bytes(MAX_HIDDEN, 64)));
  return e == cudaSuccess ? 0 : MINPPO_ERR_CUDA;
}

int head_loss_launch(const HeadLossArgs& a, int tiles, cudaStream_t stream) {
  if (a.A > MAX_ACT_DIM) return MINPPO_ERR_ARG;
  const int amax = head_amax(a.A);
  const size_t smem = head_loss_smem_bytes(a.H, amax);
  if (amax == 8) head_loss_kernel<8><<<tiles, HL_THREADS, smem, stream>>>(a);
  else if (amax == 16) head_loss_kernel<16><<<tiles, HL_THREADS, smem, stream>>>(a);
  else if (amax == 32) head_loss_kernel<32><<<tiles, HL_THREADS, smem, stream>>>(a);
  else head_loss_kernel<64><<<tiles, HL_THREADS, smem, stream>>>(a);
  return cudaGetLastError() == cudaSuccess ? 0 : MINPPO_ERR_CUDA;
}

}  // namespace minppo
