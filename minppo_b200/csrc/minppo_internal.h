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

// ---- head_loss.cu ------------------------------------------------------------------------
struct HeadLossArgs {
  const __nv_bfloat16* h_a;      // last hidden activation, actor  [M_pad][ldh]
  const __nv_bfloat16* h_c;      // last hidden activation, critic [M_pad][ldh]
  __nv_bfloat16* dz_a;           // out: dL/dz of the last hidden layer (actor)
  __nv_bfloat16* dz_c;
  const float* params;           // fp32 arena
  const int32_t* rowidx;         // [cap] local flat transition index per minibatch row
  const int32_t* count;          // [1] rows owned by this rank in this minibatch
  const float* adv_sum;          // [1] sum adv over the GLOBAL minibatch
  const float* adv_sq;           // [1] sum (adv - mean)^2 over the GLOBAL minibatch
  const float* action;           // [Bl][A]
  const float* v_old;            // [Bl]   Memory.value
  const float* logp_old;         // [Bl]   Memory.log_prob
  const float* adv;              // [Bl]
  const float* tgt;              // [Bl]
  float* partials;               // [tiles][partial_stride]
  int partial_stride;
  int po_w3a, po_b3a, po_w3c, po_b3c, po_logstd, po_bh_a, po_bh_c, po_loss;   // offsets inside a partial
  int off_w3a, off_b3a, off_w3c, off_b3c, off_logstd;                          // offsets inside the arena
  int H, A, ldh, cap;
  int act_a, act_c;              // ACTK_* of the hidden layers
  float inv_mb, clip_eps, vf_coef;
};
int head_loss_init();
int head_loss_launch(const HeadLossArgs& a, int tiles, cudaStream_t stream);

// ---- policy.cu ---------------------------------------------------------------------------
struct PolicyHeadArgs {
  const __nv_bfloat16* h_a;      // last hidden activation, actor  [rows_pad][ldh]; null = critic only (bootstrap value)
  const __nv_bfloat16* h_c;      // last hidden activation, critic [rows_pad][ldh]
  const float* params;           // fp32 arena
  int off_w3a, off_b3a, off_w3c, off_b3c, off_logstd;
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
  __nv_bfloat16* img_t;          // unused (was: transposed image); kept null
  __nv_bfloat16* img_n;          // bf16 image [in][ld_n] of a hidden kernel, ld_n == cols (the B operand of the
                                 // forward GEMMs as MN-major and of the dX GEMMs as K-major), or null
  int ld_t, ld_n;
  uint8_t* img_w2;               // output-head kernels: 16 KB bf16 hi / lo image of kernel^T in the fused kernel's
                                 // shared-memory layout (fused_step.cuh FS_W2T), or null
  int late;                      // 1: partials are written by the dW GEMM of the same launch (hidden kernels)
  int size;                      // elements of this leaf (host-computed: the kernels never walk the table serially)
  int ap;                        // img_w2: padded head width of the image (16 or 32 rows per hi / lo half)
};
struct OptArgs {
  OptLeaf leaf[MINPPO_MAX_LEAVES];
  int nleaves, P, A;
  int n_early;                   // elements of the leaves with late == 0
  int do_reduce, do_apply;
  int keep_gflat;                // also store the reduced gradient when reduce+apply are fused (tests)
  float* gflat;                  // [P + 4]
  const float* loss_src;         // loss partial sums (2 per partial)
  int loss_src_offset, loss_nparts, loss_part_stride;
  float* params; float* mu; float* nu;
  int32_t* count;
  float* block_ss;               // [grid]
  unsigned long long* barrier;
  int* err_flag;
  float* losses_out;             // [4] or null
  float* gnorm_out;              // [1] or null
  int off_logstd;
  int anneal, anneal_div, num_updates;
  float lr, max_norm, b1, b2, one_minus_b1, one_minus_b2, eps, eps_root;
  float inv_mb, vf_coef, ent_coef, entropy_const;
};
int opt_launch(const OptArgs& a, int blocks, cudaStream_t stream, bool pdl = false);
int opt_max_params(int blocks);
int weight_images_launch(const OptArgs& a, cudaStream_t stream);
int obs_image_launch(const float* obs, __nv_bfloat16* img, long long rows, int cols, int ld, cudaStream_t stream);

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
