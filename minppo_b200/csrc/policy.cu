// minppo_b200 -- policy / value heads for the rollout (forward only): output heads, Gaussian sample, log-prob, value
// (replaces the tail of ActorCritic.__call__ plus pi.sample / pi.log_prob at /root/reference/minppo/train.py:78-83,
// 157-160, and the bootstrap value at train.py:182-183).
//
// The hidden layers run on the tensor cores (umma_gemm_kernel<EPI_ACT>, same bf16 weight images and the same rounding
// points as the learner's forward pass, so the log_prob stored in Memory equals what the first PPO epoch recomputes);
// this kernel is the fp32 SIMT tail, 4 threads per env row:
//   mean = h_a W3a + b3a ; value = h_c W3c + b3c
//   rng, action_rng = split(rng)                                              (train.py:158)
//   eps[n][j] = jax.random.normal(action_rng, (N, A))[n][j]    -- distrax Normal(0,1)._sample_n, flat index n*A + j of
//               the GLOBAL [N, A] draw (an env-sharded rank generates only its rows; the values are the same)
//   action = mean + exp(log_std) * eps                                         (train.py:159; distrax ScalarAffine)
//   log_prob = sum_j(-z_j^2/2 - log(2 pi)/2) - sum_j log|scale_j|, z = (action - mean) * (1/scale)   (train.py:160)
// jax.random.normal: bits -> [1,2) mantissa trick -> uniform(nextafter(-1,0), 1) -> sqrt(2) * erf_inv(u), with XLA's
// single-precision erf_inv (Giles' polynomial).  Bits are bit-exact with the oracle; erf_inv agrees to ~1 ulp.
#include "common.cuh"
#include "minppo_internal.h"
#include "threefry.cuh"
#include "policy_math.cuh"
#include "ppo_math.cuh"

namespace minppo {

constexpr int PH_ROWS = 64;
constexpr int PH_THREADS = 256;

template <int AMAX>
__global__ void __launch_bounds__(PH_THREADS) policy_head_kernel(const PolicyHeadArgs a) {
  extern __shared__ __align__(16) uint8_t ph_smem[];
  const int H = a.H, A = a.A;
  float* w3a = reinterpret_cast<float*>(ph_smem);       // [H][AMAX+1]
  float* w3c = w3a + H * (AMAX + 1);                    // [H]
  __shared__ uint32_t s_key[4];                         // [0..1] = rng', [2..3] = action_rng
  const int tid = threadIdx.x;
  const float* P = a.params;
  const bool actor = a.h_a != nullptr;

  if (actor) {
    for (int i = tid; i < H * AMAX; i += PH_THREADS) {
      const int k = i / AMAX, j = i % AMAX;
      w3a[k * (AMAX + 1) + j] = j < A ? P[a.off.w3a + k * A + j] : 0.f;
    }
  }
  for (int i = tid; i < H; i += PH_THREADS) w3c[i] = P[a.off.w3c + i];
  if (tid == 0 && a.key_in) {
    const uint32_t k[2] = {a.key_in[0], a.key_in[1]};
    uint32_t r[2], s[2];
    key_split(k, a.mode, r, s);                         // rng, action_rng = jax.random.split(rng)
    s_key[0] = r[0]; s_key[1] = r[1]; s_key[2] = s[0]; s_key[3] = s[1];
    if (blockIdx.x == 0 && a.key_out) { a.key_out[0] = r[0]; a.key_out[1] = r[1]; }
  }
  __syncthreads();

  // ---- heads: 4 threads per row, 16-byte chunks of the activation row dealt round-robin over the quad ----
  const int r = tid >> 2, part = tid & 3;
  const int row = blockIdx.x * PH_ROWS + r;
  const bool live = row < a.rows;
  float acc[AMAX];
  float accv = 0.f;
#pragma unroll
  for (int j = 0; j < AMAX; ++j) acc[j] = 0.f;
  if (live) {
    const int chunks = H >> 3;
    const uint4* ha = actor ? reinterpret_cast<const uint4*>(a.h_a + static_cast<size_t>(row) * a.ldh) : nullptr;
    const uint4* hc = reinterpret_cast<const uint4*>(a.h_c + static_cast<size_t>(row) * a.ldh);
    for (int c = part; c < chunks; c += 4) {
      const uint4 vc = __ldg(hc + c);
      const uint32_t wc[4] = {vc.x, vc.y, vc.z, vc.w};
#pragma unroll
      for (int q = 0; q < 4; ++q)
        accv = fmaf(bf16_hi(wc[q]), w3c[c * 8 + 2 * q + 1], fmaf(bf16_lo(wc[q]), w3c[c * 8 + 2 * q], accv));
      if (actor) {
        const uint4 va = __ldg(ha + c);
        const uint32_t wa[4] = {va.x, va.y, va.z, va.w};
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const float a0 = bf16_lo(wa[q]), a1 = bf16_hi(wa[q]);
          const float* w0 = w3a + (c * 8 + 2 * q) * (AMAX + 1);
          const float* w1 = w0 + (AMAX + 1);
#pragma unroll
          for (int j = 0; j < AMAX; ++j) acc[j] = fmaf(a1, w1[j], fmaf(a0, w0[j], acc[j]));
        }
      }
    }
  }
#pragma unroll
  for (int j = 0; j < AMAX; ++j) {
    acc[j] += __shfl_xor_sync(0xffffffffu, acc[j], 1);
    acc[j] += __shfl_xor_sync(0xffffffffu, acc[j], 2);
  }
  accv += __shfl_xor_sync(0xffffffffu, accv, 1);
  accv += __shfl_xor_sync(0xffffffffu, accv, 2);
  if (!live || part != 0) return;

  if (a.value) a.value[row] = accv + P[a.off.b3c];
  if (!actor) return;
  const uint32_t akey[2] = {s_key[2], s_key[3]};
  const uint32_t gbase = static_cast<uint32_t>((a.n0 + row) * A);           // flat index of eps[n][0] in the global draw
  float quad = 0.f, logdet = 0.f;
#pragma unroll
  for (int j = 0; j < AMAX; ++j) {
    if (j < A) {
      const float mean = acc[j] + P[a.off.b3a + j];
      float act = mean;
      if (a.mean_out) a.mean_out[static_cast<size_t>(row) * A + j] = mean;
      const float scale = expf(P[a.off.logstd + j]);
      if (a.key_in) {
        const float eps = normal_from_bits(random_bits_at(akey, a.mode, gbase + j, static_cast<uint32_t>(a.n_total)));
        act = __fadd_rn(mean, __fmul_rn(scale, eps));
      }
      if (a.action) a.action[static_cast<size_t>(row) * A + j] = act;
      const float z = (act - mean) * (1.f / scale);
      quad += gauss_logp_term(z);
      logdet += logf(fabsf(scale));
    }
  }
  if (a.log_prob) a.log_prob[row] = quad - logdet;
}

static constexpr size_t policy_head_smem(int H, int amax) { return (static_cast<size_t>(H) * (amax + 1) + H) * 4; }
// H = 512 with the 64-wide template: 135,168 bytes
constexpr int PH_SMEM_OPTIN = 200 * 1024;
static_assert(policy_head_smem(MAX_HIDDEN, 64) <= PH_SMEM_OPTIN, "policy_head_kernel<64> shared memory at H = 512");

int policy_head_init() {
  cudaError_t e = cudaFuncSetAttribute(policy_head_kernel<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, PH_SMEM_OPTIN);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(policy_head_kernel<16>, cudaFuncAttributeMaxDynamicSharedMemorySize, PH_SMEM_OPTIN);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(policy_head_kernel<32>, cudaFuncAttributeMaxDynamicSharedMemorySize, PH_SMEM_OPTIN);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(policy_head_kernel<64>, cudaFuncAttributeMaxDynamicSharedMemorySize, PH_SMEM_OPTIN);
  return e == cudaSuccess ? 0 : MINPPO_ERR_CUDA;
}

int policy_head_launch(const PolicyHeadArgs& a, cudaStream_t stream) {
  if (a.A > MAX_ACT_DIM || a.H % 8 != 0 || a.rows <= 0) { set_error("policy head: unsupported shape"); return MINPPO_ERR_ARG; }
  const int amax = head_amax(a.A);
  const size_t smem = policy_head_smem(a.H, amax);
  const int blocks = (a.rows + PH_ROWS - 1) / PH_ROWS;
  if (amax == 8) policy_head_kernel<8><<<blocks, PH_THREADS, smem, stream>>>(a);
  else if (amax == 16) policy_head_kernel<16><<<blocks, PH_THREADS, smem, stream>>>(a);
  else if (amax == 32) policy_head_kernel<32><<<blocks, PH_THREADS, smem, stream>>>(a);
  else policy_head_kernel<64><<<blocks, PH_THREADS, smem, stream>>>(a);
  const cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) { set_error("policy_head launch failed: %s", cudaGetErrorString(e)); return MINPPO_ERR_CUDA; }
  return 0;
}

}  // namespace minppo
