// minppo_b200 -- bf16 operand images: the observation image of an update, and the weight images the tcgen05 GEMMs and
// the fused kernels read, from the fp32 parameter arena (at the start of an update and of a rollout policy step).  The
// optimizer, which also rewrites the weight images after every minibatch step, is dwopt_kernel (dwopt.cuh).
// With observation normalization (minppo_obs_norm) the observation image is normalized and also yields the batch
// moments of the raw observations, which the finalize and merge kernels below fold into the running statistics.
#include "common.cuh"
#include "minppo_internal.h"
#include "obs_norm.cuh"
#include "opt_common.cuh"

namespace minppo {

// fp32 [rows][cols] -> bf16 [rows][ld] (zero padded); used for the observation image and
// for the initial weight images.
// NORM: every element is normalized with the running statistics at entry (obs_norm.cuh) before the bf16 rounding.
// MAXP > 0 (with NORM): also the per-column Welford moments (count, mean, M2) of the RAW observations, in fp64: each lane
// keeps those of its (at most MAXP) column pairs in registers over the rows of its warp, the warps of a block are merged
// in warp order through shared memory, and warp 0 writes the block's partial to na.part[blockIdx.x] ([2][ld]: mean, M2).
// The row -> warp -> block mapping and the merge order depend on (rows, ld) only, so the moments are bit-reproducible;
// obs_moments_finalize_kernel merges the partials.  dst may be null there (minppo_obs_norm_fold: moments only).
// Launched with 256 threads (obs_moments_finalize_kernel counts the rows of a block from that).
template <bool NORM, int MAXP>
__global__ void f32_to_bf16_image_kernel(const float* __restrict__ src, __nv_bfloat16* __restrict__ dst,
                                         long long rows, int cols, int ld, const ObsNormArgs na) {
  // one warp per row, lanes along the row: coalesced 256-byte loads / 128-byte stores, no index division
  const int lane = threadIdx.x & 31;
  const long long nwarps = (static_cast<long long>(gridDim.x) * blockDim.x) >> 5;
  const int pairs = ld >> 1;
  if constexpr (!NORM) {
  for (long long r = (blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x) >> 5; r < rows; r += nwarps) {
    const float* s = src + r * cols;
    uint32_t* d = reinterpret_cast<uint32_t*>(dst + r * ld);
#pragma unroll 4
    for (int p = lane; p < pairs; p += 32) {
      const int c = 2 * p;
      const float x0 = c < cols ? __ldcs(s + c) : 0.f;          // the fp32 trajectory is read once per update
      const float x1 = c + 1 < cols ? __ldcs(s + c + 1) : 0.f;
      d[p] = pack_bf16x2(x0, x1);
    }
  }
  } else {
    extern __shared__ __align__(16) unsigned char norm_smem[];
    float* s_mean = reinterpret_cast<float*>(norm_smem);              // [ld] entry mean
    float* s_scale = s_mean + ld;                                     // [ld] 1 / sqrt(var + eps)
    for (int c = threadIdx.x; c < cols; c += blockDim.x) {
      s_mean[c] = na.mean[c];
      s_scale[c] = obs_norm_scale(na.var[c], na.eps);
    }
    __syncthreads();
    auto norm = [&](float x, int c) { return c < cols ? obs_norm_apply(x, s_mean[c], s_scale[c], na.clip) : 0.f; };
    if constexpr (MAXP == 0) {
      for (long long r = (blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x) >> 5; r < rows; r += nwarps) {
        const float* s = src + r * cols;
        uint32_t* d = reinterpret_cast<uint32_t*>(dst + r * ld);
#pragma unroll 4
        for (int p = lane; p < pairs; p += 32) {
          const int c = 2 * p;
          const float x0 = c < cols ? __ldcs(s + c) : 0.f;
          const float x1 = c + 1 < cols ? __ldcs(s + c + 1) : 0.f;
          d[p] = pack_bf16x2(norm(x0, c), norm(x1, c + 1));
        }
      }
    } else {
      double wm[2 * MAXP], wq[2 * MAXP], wn = 0.0;                   // column c = 2 (lane + 32 k) + h -> [2 k + h]
#pragma unroll
      for (int i = 0; i < 2 * MAXP; ++i) { wm[i] = 0.0; wq[i] = 0.0; }
      // RB rows of the warp per pass, all loads issued before the (serially dependent) moment updates
      constexpr int RB = MAXP <= 8 ? 2 : 1;
      for (long long r0 = (blockIdx.x * static_cast<long long>(blockDim.x) + threadIdx.x) >> 5; r0 < rows; r0 += RB * nwarps) {
        float x[RB][2 * MAXP];
#pragma unroll
        for (int j = 0; j < RB; ++j) {
          const long long r = r0 + j * nwarps;
          const float* s = src + (r < rows ? r : r0) * cols;
#pragma unroll
          for (int k = 0; k < MAXP; ++k) {
            const int c = 2 * (lane + 32 * k);
            x[j][2 * k] = c < cols ? __ldcs(s + c) : 0.f;
            x[j][2 * k + 1] = c + 1 < cols ? __ldcs(s + c + 1) : 0.f;
          }
        }
#pragma unroll
        for (int j = 0; j < RB; ++j) {
          const long long r = r0 + j * nwarps;
          if (r >= rows) break;
          uint32_t* d = dst ? reinterpret_cast<uint32_t*>(dst + r * ld) : nullptr;
          wn += 1.0;
          const double inv = __drcp_rn(wn);
#pragma unroll
          for (int k = 0; k < MAXP; ++k) {
            const int p = lane + 32 * k;
            if (p >= pairs) continue;
            if (d) d[p] = pack_bf16x2(norm(x[j][2 * k], 2 * p), norm(x[j][2 * k + 1], 2 * p + 1));
#pragma unroll
            for (int h = 0; h < 2; ++h) {
              if (2 * p + h >= cols) continue;
              const double xv = x[j][2 * k + h];
              const double dl = __dsub_rn(xv, wm[2 * k + h]);
              wm[2 * k + h] = __fma_rn(dl, inv, wm[2 * k + h]);
              wq[2 * k + h] = __fma_rn(dl, __dsub_rn(xv, wm[2 * k + h]), wq[2 * k + h]);
            }
          }
        }
      }
      // merge the warps of the block into warp 0, in warp order (Chan et al.), through one shared-memory slot
      __shared__ double slot_n;
      double* slot = reinterpret_cast<double*>(norm_smem + 2 * static_cast<size_t>(ld) * sizeof(float));   // [2][ld]
      const int warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
      for (int w = 1; w < nw; ++w) {
        if (warp == w) {
          if (lane == 0) slot_n = wn;
#pragma unroll
          for (int i = 0; i < 2 * MAXP; ++i) {
            const int c = 2 * (lane + 32 * (i >> 1)) + (i & 1);
            if (c < cols) { slot[c] = wm[i]; slot[ld + c] = wq[i]; }
          }
        }
        __syncthreads();
        const double nb = slot_n;
        if (warp == 0 && nb > 0.0) {
          const double n = __dadd_rn(wn, nb);
          const double f = __ddiv_rn(nb, n), g = __ddiv_rn(__dmul_rn(wn, nb), n);
#pragma unroll
          for (int i = 0; i < 2 * MAXP; ++i) {
            const int c = 2 * (lane + 32 * (i >> 1)) + (i & 1);
            if (c >= cols) continue;
            const double dl = __dsub_rn(slot[c], wm[i]);
            wm[i] = __fma_rn(dl, f, wm[i]);
            wq[i] = __dadd_rn(__dadd_rn(wq[i], slot[ld + c]), __dmul_rn(__dmul_rn(dl, dl), g));
          }
          wn = n;
        }
        __syncthreads();
      }
      if (warp == 0) {
        double* out = na.part + static_cast<size_t>(blockIdx.x) * 2 * ld;
#pragma unroll
        for (int i = 0; i < 2 * MAXP; ++i) {
          const int c = 2 * (lane + 32 * (i >> 1)) + (i & 1);
          if (c < cols) { out[c] = wm[i]; out[ld + c] = wq[i]; }
        }
      }
    }
  }
}

// Rows counted by blocks [0, b) of the moments instance: row r belongs to warp r % nwarps, warp w to block w / 8.
__device__ __forceinline__ double obs_rows_before(long long b, long long rows, long long nwarps) {
  const long long w = 8 * b;
  return static_cast<double>((rows / nwarps) * w + (w < rows % nwarps ? w : rows % nwarps));
}

// The block partials of f32_to_bf16_image_kernel<true, MAXP> merged in block order (fp64, Chan et al.) into this rank's
// batch moments out = [rows, mean[cols], M2[cols]].  One thread per column; the per-block weights of the merge depend
// only on the counts, which every thread block derives from (rows, nblk).
constexpr int OBS_MOM_THREADS = 128;
__global__ void __launch_bounds__(OBS_MOM_THREADS) obs_moments_finalize_kernel(const double* __restrict__ part, int nblk,
                                                                              int ld, int cols, long long rows,
                                                                              double* __restrict__ out) {
  __shared__ double f[OBS_NORM_MAX_BLOCKS], g[OBS_NORM_MAX_BLOCKS];
  const long long nwarps = 8LL * nblk;
  for (int b = threadIdx.x; b < nblk; b += blockDim.x) {
    const double na = obs_rows_before(b, rows, nwarps);
    const double n = obs_rows_before(b + 1, rows, nwarps);
    const double nb = __dsub_rn(n, na);
    f[b] = nb > 0.0 ? __ddiv_rn(nb, n) : 0.0;
    g[b] = nb > 0.0 ? __ddiv_rn(__dmul_rn(na, nb), n) : 0.0;
  }
  __syncthreads();
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c == 0) out[0] = static_cast<double>(rows);
  if (c >= cols) return;
  double m = 0.0, q = 0.0;
#pragma unroll 8
  for (int b = 0; b < nblk; ++b) {
    const double* pb = part + static_cast<size_t>(b) * 2 * ld;
    const double dl = __dsub_rn(pb[c], m);
    m = __fma_rn(dl, f[b], m);
    q = __dadd_rn(__dadd_rn(q, pb[ld + c]), __dmul_rn(__dmul_rn(dl, dl), g[b]));
  }
  out[1 + c] = m;
  out[1 + cols + c] = q;
}

// Folds the batch moments of W ranks ([W][stride] of [n, mean[D], M2[D]], merged in rank order) into the running
// statistics, in place: Chan's parallel update in fp64, stored as f32 mean / var and f64 count
// (include/minppo_b200.h, minppo_obs_norm).  One block: every thread reads the entry count before thread 0 replaces it.
__global__ void obs_norm_merge_kernel(const double* __restrict__ mom, int W, int stride, int D, float* mean, float* var,
                                      double* count) {
  const double n = count[0];
  __syncthreads();
  for (int c = threadIdx.x; c < D; c += blockDim.x) {
    double nb = mom[0], mb = mom[1 + c], qb = mom[1 + D + c];
    for (int r = 1; r < W; ++r) {
      const double* o = mom + static_cast<size_t>(r) * stride;
      const double n2 = o[0], nn = __dadd_rn(nb, n2);
      const double dl = __dsub_rn(o[1 + c], mb);
      mb = __dadd_rn(mb, __ddiv_rn(__dmul_rn(dl, n2), nn));
      qb = __dadd_rn(__dadd_rn(qb, o[1 + D + c]), __ddiv_rn(__dmul_rn(__dmul_rn(__dmul_rn(dl, dl), nb), n2), nn));
      nb = nn;
    }
    // n' = n + n_b;  mean' = mean + d n_b / n';  var' = (var n + M2_b + d^2 n n_b / n') / n'
    const double n1 = __dadd_rn(n, nb);
    const double mu = mean[c], v = var[c];
    const double dl = __dsub_rn(mb, mu);
    mean[c] = static_cast<float>(__dadd_rn(mu, __ddiv_rn(__dmul_rn(dl, nb), n1)));
    var[c] = static_cast<float>(__ddiv_rn(__dadd_rn(__dadd_rn(__dmul_rn(v, n), qb),
                                                    __ddiv_rn(__dmul_rn(__dmul_rn(__dmul_rn(dl, dl), n), nb), n1)), n1));
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    double nb = mom[0];
    for (int r = 1; r < W; ++r) nb = __dadd_rn(nb, mom[static_cast<size_t>(r) * stride]);
    count[0] = __dadd_rn(n, nb);
  }
}

// weight images from the fp32 arena (ctx_create / set_params): same mapping as the apply phase
__global__ void weight_images_kernel(const OptArgs a) {
  const int gthreads = gridDim.x * blockDim.x;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < a.P; i += gthreads) {
    int l = 0;
    while (l + 1 < a.nleaves && i >= a.leaf[l + 1].offset) ++l;
    write_images(a.leaf[l], i, a.params[i]);
  }
}

int weight_images_launch(const OptArgs& a, cudaStream_t stream) {
  weight_images_kernel<<<148, 256, 0, stream>>>(a);
  return cudaGetLastError() == cudaSuccess ? 0 : MINPPO_ERR_CUDA;
}

int obs_image_launch(const float* obs, __nv_bfloat16* img, long long rows, int cols, int ld, cudaStream_t stream) {
  long long blocks = (rows + 7) / 8;                      // 8 warps per block, one row per warp and pass
  if (blocks > 148LL * 16) blocks = 148LL * 16;
  if (blocks < 1) blocks = 1;
  f32_to_bf16_image_kernel<false, 0><<<static_cast<unsigned>(blocks), 256, 0, stream>>>(obs, img, rows, cols, ld, ObsNormArgs{});
  return cudaGetLastError() == cudaSuccess ? 0 : MINPPO_ERR_CUDA;
}

// Grid of the moments instances: 8 rows per block and pass, capped at one wave of the blocks the register-resident
// moments (4 doubles per column pair, MAXP pairs per lane) leave room for: 3, 2 and 1 block(s) per SM of 148 for
// MAXP = 4, 8, 16 (-Xptxas -v: 74, 114 and 215 registers).  Depends on (rows, ld) only.
static int obs_maxp(int ld) { return ld <= 256 ? 4 : (ld <= 512 ? 8 : 16); }
int obs_norm_blocks(long long rows, int ld) {
  const int maxp = obs_maxp(ld);
  const long long cap = 148LL * (maxp == 4 ? 3 : (maxp == 8 ? 2 : 1));
  long long blocks = (rows + 7) / 8;
  if (blocks > cap) blocks = cap;
  return static_cast<int>(blocks < 1 ? 1 : blocks);
}

int obs_norm_image_launch(const float* obs, __nv_bfloat16* img, long long rows, int cols, int ld, const ObsNormArgs& na,
                          cudaStream_t stream) {
  const size_t smem = 2 * static_cast<size_t>(ld) * sizeof(float) + (na.part ? 2 * static_cast<size_t>(ld) * sizeof(double) : 0);
  if (!na.part) {                                        // normalized image only (layer-wise policy step)
    long long blocks = (rows + 7) / 8;
    if (blocks > 148LL * 16) blocks = 148LL * 16;
    if (blocks < 1) blocks = 1;
    f32_to_bf16_image_kernel<true, 0><<<static_cast<unsigned>(blocks), 256, smem, stream>>>(obs, img, rows, cols, ld, na);
  } else {
    if (ld > OBS_NORM_MAX_D) return MINPPO_ERR_UNSUPPORTED;
    const unsigned blocks = static_cast<unsigned>(obs_norm_blocks(rows, ld));
    switch (obs_maxp(ld)) {
      case 4: f32_to_bf16_image_kernel<true, 4><<<blocks, 256, smem, stream>>>(obs, img, rows, cols, ld, na); break;
      case 8: f32_to_bf16_image_kernel<true, 8><<<blocks, 256, smem, stream>>>(obs, img, rows, cols, ld, na); break;
      default: f32_to_bf16_image_kernel<true, 16><<<blocks, 256, smem, stream>>>(obs, img, rows, cols, ld, na); break;
    }
  }
  return cudaGetLastError() == cudaSuccess ? 0 : MINPPO_ERR_CUDA;
}

int obs_moments_finalize_launch(const double* part, long long rows, int cols, int ld, double* out, cudaStream_t stream) {
  const int blocks = (cols + OBS_MOM_THREADS - 1) / OBS_MOM_THREADS;
  obs_moments_finalize_kernel<<<blocks, OBS_MOM_THREADS, 0, stream>>>(part, obs_norm_blocks(rows, ld), ld, cols, rows, out);
  return cudaGetLastError() == cudaSuccess ? 0 : MINPPO_ERR_CUDA;
}

int obs_norm_merge_launch(const double* moments, int W, int stride, int D, float* mean, float* var, double* count,
                          cudaStream_t stream) {
  obs_norm_merge_kernel<<<1, 256, 0, stream>>>(moments, W, stride, D, mean, var, count);
  return cudaGetLastError() == cudaSuccess ? 0 : MINPPO_ERR_CUDA;
}

}  // namespace minppo
