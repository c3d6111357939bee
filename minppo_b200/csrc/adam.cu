// minppo_b200 -- bf16 operand images: the observation image of an update, and the weight images the tcgen05 GEMMs and
// the fused kernels read, from the fp32 parameter arena (at the start of an update and of a rollout policy step).  The
// optimizer, which also rewrites the weight images after every minibatch step, is dwopt_kernel (dwopt.cuh).
#include "common.cuh"
#include "minppo_internal.h"
#include "opt_common.cuh"

namespace minppo {

// fp32 [rows][cols] -> bf16 [rows][ld] (zero padded); used for the observation image and
// for the initial weight images.
__global__ void f32_to_bf16_image_kernel(const float* __restrict__ src, __nv_bfloat16* __restrict__ dst,
                                         long long rows, int cols, int ld) {
  // one warp per row, lanes along the row: coalesced 256-byte loads / 128-byte stores, no index division
  const int lane = threadIdx.x & 31;
  const long long nwarps = (static_cast<long long>(gridDim.x) * blockDim.x) >> 5;
  const int pairs = ld >> 1;
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
  f32_to_bf16_image_kernel<<<static_cast<unsigned>(blocks), 256, 0, stream>>>(obs, img, rows, cols, ld);
  return cudaGetLastError() == cudaSuccess ? 0 : MINPPO_ERR_CUDA;
}

}  // namespace minppo
