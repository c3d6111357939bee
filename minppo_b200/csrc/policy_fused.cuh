// minppo_b200 -- the rollout's policy / value step in ONE launch (2-hidden-layer nets):
//   pi, value = network.apply(params, last_obs); rng, action_rng = split(rng); action = pi.sample(seed=action_rng);
//   log_prob = pi.log_prob(action)                     (/root/reference/minppo/train.py:157-160; bootstrap value: 182-183)
//
// The forward half of the fused learner step (fused_step.cuh) with the sampler as its epilogue: one CTA = one 128-env
// tile x one net.  The fp32 observation rows are converted to bf16 on the way into the X slots (no separate image
// pass), the hidden layers run on the tcgen05 tensor cores against the learner's own bf16 weight images, the output
// heads as bf16 hi/lo pairs exactly like the learner's forward pass -- so a trajectory collected through this kernel is
// seen by the first PPO epoch with ratio == 1 and v == v_old up to fp32 rounding of the final sums.  The actor CTAs then
// draw eps = jax.random.normal(action_rng, (N, A)) at the GLOBAL flat index n * A + j (an env-sharded rank generates
// exactly its rows of the global sample), form the action and its log-prob; the critic CTAs write the value.
// Same shared-memory layout, warp roles and tensor maps as fused_step.cuh.
#pragma once

#include "fused_step.cuh"
#include "policy_math.cuh"
#include "ppo_math.cuh"

namespace minppo {

struct alignas(64) PolicyNet {
  CUtensorMap tm_w0, tm_w1;      // weight images, box {64 out, 32 in} (fused_step.cuh)
  const float* b0;
  const float* b1;
  const uint4* w2img;            // head kernel^T bf16 hi / lo image
  const float* b2;
  int act, aout;
};

struct alignas(64) PolicyParams {
  PolicyNet net[2];
  const float* obs;              // [rows][D] fp32 (last_obs of this rank's envs)
  const float* log_std;          // arena pointer
  const uint32_t* key_in;        // RunnerState.rng [2]; null = no sampling (action = mean)
  uint32_t* key_out;             // rng after the split; may be null
  float* action;                 // [rows][A] or null
  float* log_prob;               // [rows] or null
  float* value;                  // [rows] or null
  float* mean_out;               // [rows][A] or null
  long long n0, n_total;         // first GLOBAL env of this rank; elements of the global normal draw (N * A)
  int rows, D, Dp, H, A, mode;
  int net_first;                 // 0: actor + critic CTAs; 1: critic only (grid = tiles)
};

template <int AP>
__global__ void __launch_bounds__(FS_THREADS, 1) policy_fused_kernel(const __grid_constant__ PolicyParams p) {
  using LY = FsLayout<AP>;
  constexpr int NS = LY::NS, NS1 = LY::NS1, PG = LY::PG;
  extern __shared__ uint8_t smem_raw[];
  __shared__ uint32_t tmem_slot;
  __shared__ uint32_t s_key[4];                         // [0..1] = rng', [2..3] = action_rng
  const uint32_t raw = smem_u32(smem_raw);
  const uint32_t base = (raw + 1023u) & ~1023u;
  uint8_t* sm = smem_raw + (base - raw);
  float* bias_s = reinterpret_cast<float*>(sm + LY::BIAS);
  float* hb = reinterpret_cast<float*>(sm + LY::HB);            // [0, AP) head bias, [AP, 2AP) log_std, [2AP, 3AP) scale
  uint64_t* bars = reinterpret_cast<uint64_t*>(sm + LY::BARS);
  uint64_t* l1_full = bars;             // [8]
  uint64_t* l1_empty = bars + 8;        // [8]
  uint64_t* x_full = bars + 16;         // [4]
  uint64_t* x_empty = bars + 20;        // [4]
  uint64_t* full_bar = bars + 24;       // [4]
  uint64_t* empty_bar = bars + 28;      // [4]
  uint64_t* accf0 = bars + 32;
  uint64_t* accf1 = bars + 33;
  uint64_t* headf = bars + 34;
  uint64_t* h2r = bars + 39;
  uint64_t* h1r = bars + 41;            // [4]

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int net = p.net_first ? 1 : (static_cast<int>(blockIdx.x) & 1);
  const int tile = p.net_first ? static_cast<int>(blockIdx.x) : (static_cast<int>(blockIdx.x) >> 1);
  const PolicyNet& G = p.net[net];
  const int H = p.H, nkH = H >> 6, nk0 = p.Dp >> 6;
  const uint32_t R0 = base + LY::R0, R1 = base + LY::R1, RB = base + LY::RB, W2T = base + LY::W2T;
  auto l1_stage = [&](int s) -> uint32_t { return s < NS ? RB + s * FS_STAGE : R0 + (s - NS) * FS_STAGE; };

  if (threadIdx.x == FS_WORKERS) {
    for (int s = 0; s < 8; ++s) { mbar_init(&l1_full[s], 1); mbar_init(&l1_empty[s], 1); }
    for (int s = 0; s < 4; ++s) {
      mbar_init(&x_full[s], FS_NWW); mbar_init(&x_empty[s], 1);
      mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1);
      mbar_init(&h1r[s], FS_NWW);
    }
    mbar_init(accf0, 1); mbar_init(accf1, 1); mbar_init(headf, 1);
    mbar_init(h2r, FS_NWW);
    fence_mbar_init();
  }
  if (warp == FS_MMA_WARP) {
    tmem_alloc(&tmem_slot, 512);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_slot;
  const uint32_t acc0 = tmem_base, acc1 = tmem_base + 256, acc_head = tmem_base;   // heads reuse acc0 (drained by epilogue 1)

  if (warp == FS_TMA_WARP) {
    if (elect_one()) {
      tma_prefetch_desc(&G.tm_w0); tma_prefetch_desc(&G.tm_w1);
      const uint32_t bytes = static_cast<uint32_t>(H) * 64u;
      const int n1 = 2 * nk0;
      for (int j = 0; j < n1; ++j) {
        const int s = j % NS1;
        if (j >= NS1) mbar_wait(&l1_empty[s], ((j / NS1) - 1) & 1);
        mbar_arrive_expect_tx(&l1_full[s], bytes);
        const uint32_t dst = l1_stage(s);
        for (int c = 0; c < nkH; ++c) tma_load_2d(dst + c * 4096, &G.tm_w0, &l1_full[s], c * 64, j * 32);
      }
      const int n2 = 2 * nkH;
      for (int i = 0; i < n2; ++i) {
        const int s = i % NS;
        if (i < NS) {
          int jl = -1;
          for (int j = s; j < n1; j += NS1) jl = j;
          if (jl >= 0) mbar_wait(&l1_empty[s], (jl / NS1) & 1);
        } else {
          mbar_wait(&empty_bar[s], ((i / NS) - 1) & 1);
        }
        mbar_arrive_expect_tx(&full_bar[s], bytes);
        const uint32_t dst = RB + s * FS_STAGE;
        for (int c = 0; c < nkH; ++c) tma_load_2d(dst + c * 4096, &G.tm_w1, &full_bar[s], c * 64, i * 32);
      }
    }
  } else if (warp == FS_MMA_WARP) {
    if (elect_one()) {
      const uint32_t idesc_bmn = umma_idesc_bf16(128, static_cast<uint32_t>(H), 0u, 1u);
      for (int kb = 0; kb < nk0; ++kb) {
        const int xs = kb & 3;
        mbar_wait_spin(&x_full[xs], (kb >> 2) & 1);
        for (int hb2 = 0; hb2 < 2; ++hb2) {
          const int j = 2 * kb + hb2, s = j % NS1;
          mbar_wait_spin(&l1_full[s], (j / NS1) & 1);
          tc_fence_after();
          const uint32_t sa = R1 + xs * 16384 + hb2 * 64, sb = l1_stage(s);
#pragma unroll
          for (int jj = 0; jj < 2; ++jj)
            umma_bf16(acc0, umma_smem_desc(sa + jj * 32, 16, 1024), umma_smem_desc(sb + jj * 2048, 4096, 1024), idesc_bmn,
                      (j > 0 || jj > 0) ? 1u : 0u);
          umma_commit(&l1_empty[s]);
        }
        umma_commit(&x_empty[xs]);
      }
      umma_commit(accf0);
      int i = 0;
      for (int kb = 0; kb < nkH; ++kb) {
        mbar_wait_spin(&h1r[kb], 0);
        for (int hb2 = 0; hb2 < 2; ++hb2, ++i) {
          const int s = i % NS;
          mbar_wait_spin(&full_bar[s], (i / NS) & 1);
          tc_fence_after();
          const uint32_t sa = R0 + kb * 16384 + hb2 * 64, sb = RB + s * FS_STAGE;
#pragma unroll
          for (int jj = 0; jj < 2; ++jj)
            umma_bf16(acc1, umma_smem_desc(sa + jj * 32, 16, 1024), umma_smem_desc(sb + jj * 2048, 4096, 1024), idesc_bmn,
                      (i > 0 || jj > 0) ? 1u : 0u);
          umma_commit(&empty_bar[s]);
        }
      }
      umma_commit(accf1);
      // heads: [out_hi | out_lo] = H2 [W2_hi | W2_lo] -> acc0 columns [0, 2AP) (all of h1r has been waited for: acc0 is drained)
      mbar_wait_spin(h2r, 0);
      tc_fence_after();
      const uint32_t idesc_h = umma_idesc_bf16(128, 2u * AP, 0u, 0u);
      uint32_t accum = 0;
      for (int kb = 0; kb < nkH; ++kb)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          umma_bf16(acc_head, umma_smem_desc(R1 + kb * 16384 + j * 32, 16, 1024),
                    umma_smem_desc(W2T + kb * PG + j * 32, 16, 1024), idesc_h, accum);
          accum = 1;
        }
      umma_commit(headf);
    }
  } else {
    // ===================== workers =====================
    const int wt = static_cast<int>(threadIdx.x);
    const int q = warp & 3, sub = warp >> 2;
    const int erow = q * 32 + lane;
    const int act = G.act, aout = G.aout;
    // ---- observation rows of this tile: fp32 -> bf16 into the X slots (K-major, SW128); thread = (row, 16-column quarter)
    const int xrow = wt >> 2, xq = wt & 3;
    const int grow = tile * 128 + xrow;
    const float* orow = p.obs + static_cast<size_t>(grow < p.rows ? grow : 0) * p.D;
    const bool rlive = grow < p.rows;
    auto fill_block = [&](int kb) {
      const int c0 = kb * 64 + xq * 16;
      float v[16];
#pragma unroll
      for (int e = 0; e < 16; ++e) v[e] = (rlive && c0 + e < p.D) ? __ldg(orow + c0 + e) : 0.f;
      const uint32_t dst = R1 + (kb & 3) * 16384 + xrow * 128;
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const int chunk = xq * 2 + h;
        sts128(dst + ((chunk ^ (xrow & 7)) << 4),
               make_uint4(pack_bf16x2(v[8 * h], v[8 * h + 1]), pack_bf16x2(v[8 * h + 2], v[8 * h + 3]),
                          pack_bf16x2(v[8 * h + 4], v[8 * h + 5]), pack_bf16x2(v[8 * h + 6], v[8 * h + 7])));
      }
    };
    for (int i = wt; i < (H * AP) >> 2; i += FS_WORKERS) cp_async_16(W2T + i * 16, G.w2img + i);
    cp_async_commit();
    float bv = 0.f;
    if (wt < 256) bv = wt < H ? __ldg(G.b0 + wt) : 0.f;
    else bv = wt - 256 < H ? __ldg(G.b1 + wt - 256) : 0.f;
    float hbv = 0.f;
    if (wt < AP) hbv = wt < aout ? __ldg(G.b2 + wt) : 0.f;
    else if (wt < 2 * AP) hbv = (net == 0 && wt - AP < aout) ? __ldg(p.log_std + wt - AP) : 0.f;
    for (int kb = 0; kb < nk0; ++kb) {
      if (kb >= FS_XSLOTS) mbar_wait(&x_empty[kb & 3], ((kb >> 2) - 1) & 1);
      fill_block(kb);
      fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) mbar_arrive(&x_full[kb & 3]);
    }
    bias_s[wt] = bv;
    if (wt < 2 * AP) hb[wt] = hbv;
    if (wt >= AP && wt < 2 * AP) hb[AP + wt] = expf(hbv);         // scale = exp(log_std)
    if (net == 0 && wt == 2 * AP && p.key_in) {
      const uint32_t k[2] = {p.key_in[0], p.key_in[1]};
      uint32_t r[2], s[2];
      key_split(k, p.mode, r, s);                               // rng, action_rng = jax.random.split(rng)
      s_key[0] = r[0]; s_key[1] = r[1]; s_key[2] = s[0]; s_key[3] = s[1];
      if (tile == 0 && p.key_out) { p.key_out[0] = r[0]; p.key_out[1] = r[1]; }
    }
    cp_async_wait<0>();
    fence_proxy_async_smem();
    worker_bar();
    // ---- epilogue 1: H1 -> R0 (published in 64-column blocks) ----
    mbar_wait(accf0, 0);
    tc_fence_after();
    epilogue_act(acc0, R0, bias_s, act, erow, q, sub * 16, 64, nkH, h1r);
    // ---- epilogue 2: H2 -> R1 ----
    mbar_wait(accf1, 0);
    tc_fence_after();
    epilogue_act(acc1, R1, bias_s + 256, act, erow, q, sub * (H >> 2), 16, H >> 6, nullptr);
    fence_proxy_async_smem();
    tc_fence_before();
    __syncwarp();
    if (lane == 0) mbar_arrive(h2r);
    // ---- heads, sample, log-prob / value: thread = env row (sub == 0 warps) ----
    mbar_wait(headf, 0);
    tc_fence_after();
    if (sub == 0) {
      const uint32_t th = acc_head + (static_cast<uint32_t>(q * 32) << 16);
      const int row = tile * 128 + erow;
      const bool live = row < p.rows;
      if (net == 1) {
        const float ohi = tmem_ld_32x1(th);
        const float olo = tmem_ld_32x1(th + AP);
        tmem_ld_wait();
        if (live && p.value) p.value[row] = (ohi + olo) + hb[0];
      } else {
        const uint32_t akey[2] = {s_key[2], s_key[3]};
        const uint32_t gbase = static_cast<uint32_t>((p.n0 + row) * p.A);      // flat index of eps[n][0] in the global draw
        float quad = 0.f, logdet = 0.f;
#pragma unroll
        for (int c = 0; c < AP / 16; ++c) {
          float ohi[16], olo[16];
          tmem_ld_32x16(th + 16 * c, ohi);
          tmem_ld_32x16(th + AP + 16 * c, olo);
          tmem_ld_wait();
          if (live) {
#pragma unroll
            for (int jj = 0; jj < 16; ++jj) {
              const int j = 16 * c + jj;
              if (j < aout) {
                const float mean = (ohi[jj] + olo[jj]) + hb[j];
                const float scale = hb[2 * AP + j];
                float a = mean;
                if (p.mean_out) p.mean_out[static_cast<size_t>(row) * p.A + j] = mean;
                if (p.key_in) {
                  const float eps = normal_from_bits(random_bits_at(akey, p.mode, gbase + j, static_cast<uint32_t>(p.n_total)));
                  a = __fadd_rn(mean, __fmul_rn(scale, eps));
                }
                if (p.action) p.action[static_cast<size_t>(row) * p.A + j] = a;
                const float z = (a - mean) * (1.f / scale);
                quad += gauss_logp_term(z);
                logdet += logf(fabsf(scale));
              }
            }
          }
        }
        if (live && p.log_prob) p.log_prob[row] = quad - logdet;
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == FS_MMA_WARP) tmem_dealloc(tmem_base, 512);
}

inline cudaError_t policy_fused_launch(const PolicyParams& p, int tiles, cudaStream_t stream, int ap) {
  const int grid = p.net_first ? tiles : 2 * tiles;
  return ap == 16 ? launch_kernel(policy_fused_kernel<16>, grid, FS_THREADS, FsLayout<16>::BYTES, stream, false, p)
                  : launch_kernel(policy_fused_kernel<32>, grid, FS_THREADS, FsLayout<32>::BYTES, stream, false, p);
}
inline cudaError_t policy_fused_init_attrs() {
  cudaError_t e = cudaFuncSetAttribute(policy_fused_kernel<16>, cudaFuncAttributeMaxDynamicSharedMemorySize, FsLayout<16>::BYTES);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(policy_fused_kernel<32>, cudaFuncAttributeMaxDynamicSharedMemorySize, FsLayout<32>::BYTES);
  return e;
}

}  // namespace minppo
