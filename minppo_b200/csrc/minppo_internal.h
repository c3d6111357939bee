// minppo_b200 -- declarations shared between the .cu translation units (not part of the ABI).
#pragma once

#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

#include "../../include/minppo_b200.h"

namespace minppo {

enum : int { ACTK_TANH = 0, ACTK_RELU = 1, ACTK_TANH_FAST = 2 };   // == ACT_* in umma_gemm.cuh

// widest model.hidden_size: hidden layers wider than one 256-column GEMM tile run as two column groups
constexpr int MAX_HIDDEN = 512;
// widest act_dim: above 32 (FS_MAX_AP) the heads run on the layer-wise kernels' 64-wide templates
constexpr int MAX_ACT_DIM = 64;
// head template width of the layer-wise kernels (head_loss_kernel, policy_head_kernel) for act_dim A
inline int head_amax(int A) { return A <= 8 ? 8 : (A <= 16 ? 16 : (A <= 32 ? 32 : 64)); }

// Per-minibatch sums the loss kernels hand to the optimizer kernel: a block of LOSS_SUMS floats in every per-tile partial
// (at po_loss), reduced in fixed order into gflat[P + i] and, on env-sharded ranks, all-reduced with the gradient:
//   [0] sum max(vl, vlc)   [1] sum min(l1, l2)   [2] value-clip count |v - v_old| > clip_eps
//   [3] approx-KL sum of expm1(log r) - log r    [4] ratio-clip count |r - 1| > clip_eps
// [0], [1] are the loss sums; [2..4] exist only for the per-step statistics (minppo_update_with_stats) and feed nothing else.
constexpr int LOSS_SUMS = 5;

// ---- gae.cu ------------------------------------------------------------------------------
void gae_plan(int T, long long N, int sm_count, int* vec, int* chunks, int* seg_len);
int gae_launch(const float* reward, const float* value, const uint8_t* done, const float* last_val, float* adv,
               float* tgt, int T, long long N, float gamma, float gl, int sm_count, int force_chunks,
               cudaStream_t stream);

// ---- prng_sort.cu ------------------------------------------------------------------------
size_t perm_workspace_bytes(int epochs, long long B);
// Sorts `epochs` permutations: perm_out[j] = permutation of epoch epoch_first + j * epoch_step of the update's key chain;
// key_out = the key after key_epochs splits (-1: epochs).
int perm_launch(const uint32_t* key_in_dev, uint32_t* key_out_dev, int mode, int epochs, long long B,
                int32_t* perm_out, void* ws, size_t ws_bytes, cudaStream_t stream, int epoch_first = 0,
                int epoch_step = 1, int key_epochs = -1);
int perm_launch_count(long long B);

// ---- minibatch.cu ------------------------------------------------------------------------
// rowidx[(e*M+k)*cap + j] = local flat index of the j-th row of minibatch (e,k) that this rank
// owns, in permutation order; entries j >= count are 0.  counts[e*M+k] = number owned.
int compact_rows_launch(const int32_t* perms, int32_t* rowidx, int32_t* counts, int E, int M, long long B, int mb,
                        int cap, int N, int n0, int Nl, int* err_flag, cudaStream_t stream);
// stats[s] = sum of adv over owned rows of minibatch s = e*M+k (pass 0); stats[EM+s] = sum (adv - mean)^2
// with mean = stats[s] / mb (pass 1, after the sums have been all-reduced if sharded).
int adv_stats_launch(const float* adv, const int32_t* rowidx, const int32_t* counts, float* stats, int EM, int cap,
                     int mb, int pass, cudaStream_t stream);

// arena offsets of the output-head leaves (kernel and bias of each net's head, log_std)
struct HeadOffsets {
  int w3a, b3a, w3c, b3c, logstd;
};

// Inputs of the PPO loss of one minibatch step (ppo_math.cuh), read by the fused step kernel and head_loss_kernel.  The row
// lists and sums cover every step of the update; a kernel reads those of minibatch step `step`.
struct LossOperands {
  const int32_t* rowidx;         // [E*M][cap] local flat transition index per minibatch row
  const int32_t* count;          // [E*M] rows owned by this rank in each minibatch
  const float* adv_sum;          // [E*M] sum adv over the GLOBAL minibatch
  const float* adv_sq;           // [E*M] sum (adv - mean)^2 over the GLOBAL minibatch
  const float* action;           // [Bl][A]
  const float* v_old;            // [Bl]   Memory.value
  const float* logp_old;         // [Bl]   Memory.log_prob
  const float* adv;              // [Bl]
  const float* tgt;              // [Bl]
  int cap;                       // row-list stride
  int step;                      // minibatch step e * M + k of this launch
  float inv_mb, clip_eps, vf_coef;
};

// ---- head_loss.cu ------------------------------------------------------------------------
struct HeadLossArgs {
  const __nv_bfloat16* h_a;      // last hidden activation, actor  [M_pad][ldh]
  const __nv_bfloat16* h_c;      // last hidden activation, critic [M_pad][ldh]
  __nv_bfloat16* dz_a;           // out: dL/dz of the last hidden layer (actor)
  __nv_bfloat16* dz_c;
  const float* params;           // fp32 arena
  LossOperands loss;
  float* partials;               // [tiles][partial_stride]
  int partial_stride;
  int po_w3a, po_b3a, po_w3c, po_b3c, po_logstd, po_loss;   // offsets inside a partial
  HeadOffsets off;                                            // offsets inside the arena
  int H, A, ldh;
  int act_a, act_c;              // ACTK_* of the hidden layers
};
int head_loss_init();
int head_loss_launch(const HeadLossArgs& a, int tiles, cudaStream_t stream);

// ---- policy.cu ---------------------------------------------------------------------------
struct PolicyHeadArgs {
  const __nv_bfloat16* h_a;      // last hidden activation, actor  [rows_pad][ldh]; null = critic only (bootstrap value)
  const __nv_bfloat16* h_c;      // last hidden activation, critic [rows_pad][ldh]
  const float* params;           // fp32 arena
  HeadOffsets off;
  int H, A, ldh;
  int rows;                      // env rows of this rank
  long long n0;                  // first GLOBAL env index of this rank
  long long n_total;             // elements of the global normal draw, N * A
  const uint32_t* key_in;        // RunnerState.rng [2]; null = no sampling (action = mean)
  uint32_t* key_out;             // rng after `rng, action_rng = split(rng)`; may be null; must not alias key_in
  int mode;                      // MINPPO_PRNG_*
  float* action;                 // [rows][A] or null
  float* log_prob;               // [rows] or null
  float* value;                  // [rows] or null
  float* mean_out;               // [rows][A] or null
};
int policy_head_init();
int policy_head_launch(const PolicyHeadArgs& a, cudaStream_t stream);

// ---- adam.cu -----------------------------------------------------------------------------
struct OptLeaf {
  int offset;                    // first element in the arena
  int cols;                      // kernel: out features; bias / log_std: length
  const float* grad_src;         // partial buffer base
  int src_offset;                // offset of this leaf inside one partial
  int nparts;                    // partials to sum (fixed order)
  int part_stride;               // floats between consecutive partials
  float grad_bias;               // constant added to every element (-ent_coef for log_std)
  __nv_bfloat16* img_n;          // bf16 image [in][cols] of a hidden kernel (the B operand of the forward GEMMs as MN-major
                                 // and of the dX GEMMs as K-major), or null
  uint8_t* img_w2;               // output-head kernels: 16 KB bf16 hi / lo image of kernel^T in the fused kernel's
                                 // shared-memory layout (fused_step.cuh FS_W2T), or null
  int late;                      // 1: partials are written by the dW GEMM (hidden kernels), summed in 16-byte units
  int size;                      // elements of this leaf (host-computed: the kernels never walk the table serially)
  int ap;                        // img_w2: padded head width of the image (16 or 32 rows per hi / lo half)
  // late leaves in dwopt.cuh: the completion counters of the dW GEMM tiles that write this leaf's partials (all 0 when the
  // GEMM ran as a launch of its own)
  int tile0;                     // counter of the layer's first tile (column group 0, m-tile 0); tiles run m-tile fastest
  int tile_n;                    // tiles of the layer (column groups x 128-row m-tiles)
  int tile_split;                // hidden kernels: columns of column group 0; 0 (biases): an element needs every tile
};
struct OptArgs {
  OptLeaf leaf[MINPPO_MAX_LEAVES];
  int nleaves, P, A;
  int n_early;                   // elements of the leaves with late == 0
  int do_apply;
  float* gflat;                  // [P + 8] reduced gradient (minppo_ctx_read buffer 3 returns the last one), then the LOSS_SUMS sums
  const float* loss_src;         // loss partial sums (LOSS_SUMS per partial)
  int loss_src_offset, loss_nparts, loss_part_stride;
  float* params; float* mu; float* nu;
  int32_t* count;
  float* block_ss;               // [grid]
  unsigned long long* barrier;
  int* err_flag;
  float* losses_out;             // [4] or null
  float* stats_out;              // [E * M][4] per-step statistics (approx_kl, clip_fraction, value_clip_fraction, grad_norm) or null
  float* gnorm_out;              // [1] or null
  int off_logstd;
  int anneal, anneal_div, num_updates;
  float lr, max_norm, b1, b2, one_minus_b1, one_minus_b2, eps, eps_root;
  float inv_mb, vf_coef, ent_coef, entropy_const;
};
int weight_images_launch(const OptArgs& a, cudaStream_t stream);
int obs_image_launch(const float* obs, __nv_bfloat16* img, long long rows, int cols, int ld, cudaStream_t stream);

// Observation normalization (include/minppo_b200.h, minppo_obs_norm): operands of the normalizing image kernel.
constexpr int OBS_NORM_MAX_D = 1024;          // widest padded observation row whose moments the image kernel accumulates
constexpr int OBS_NORM_MAX_BLOCKS = 148 * 3;  // most block partials of one moments pass (obs_norm_blocks)
struct ObsNormArgs {
  const float* mean;             // [cols] running statistics at entry (read only)
  const float* var;              // [cols]
  float eps, clip;               // clip <= 0: no clamp
  double* part;                  // null: normalized image only; else the per-block moments [obs_norm_blocks][2][ld]
};
int obs_norm_blocks(long long rows, int ld);
// Normalized observation image (img may be null when na.part is set: moments only), plus the block partials of the raw
// observations' moments when na.part is set (ld <= OBS_NORM_MAX_D).
int obs_norm_image_launch(const float* obs, __nv_bfloat16* img, long long rows, int cols, int ld, const ObsNormArgs& na,
                          cudaStream_t stream);
// The partials of an obs_norm_image_launch over `rows` rows merged into out = [rows, mean[cols], M2[cols]] (f64).
int obs_moments_finalize_launch(const double* part, long long rows, int cols, int ld, double* out, cudaStream_t stream);
// The moments of W ranks ([W][stride], rank order) folded into the running statistics in place.
int obs_norm_merge_launch(const double* moments, int W, int stride, int D, float* mean, float* var, double* count,
                          cudaStream_t stream);

// ---- launch helper: optional programmatic-dependent-launch edge to the preceding kernel ------
template <typename Kern, typename Arg>
inline cudaError_t launch_kernel(Kern kern, unsigned grid, unsigned block, size_t smem, cudaStream_t stream, bool pdl,
                                 const Arg& arg) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(grid, 1, 1);
  cfg.blockDim = dim3(block, 1, 1);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at;
  cfg.numAttrs = pdl ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kern, arg);
}

// Variadic form for the small per-update kernels (sort passes, row lists, advantage statistics): always launched with
// the programmatic-serialization attribute; each of them starts with griddep_wait(); griddep_launch(); so the launch
// latency of kernel K + 1 hides behind kernel K while every read still follows K's completion.
template <typename... KArgs, typename... Args>
inline cudaError_t launch_chain(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream, Args... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  at[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = at;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kern, static_cast<KArgs>(args)...);
}

// ---- error plumbing (learner.cu) -----------------------------------------------------------
void set_error(const char* fmt, ...);

}  // namespace minppo
