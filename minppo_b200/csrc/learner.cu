// minppo_b200 -- context, step orchestration and the C ABI (include/minppo_b200.h).
//
// One learner update (replaces /root/reference/minppo/train.py:185-281):
//   per update : GAE -> all E permutations -> per-minibatch row lists -> advantage statistics
//                -> bf16 observation image
//   per (epoch, minibatch), strictly sequential (train.py:268, 274):
//     fwd  layer 0      tcgen05 GEMM, A rows gathered by index, bias+activation epilogue
//     fwd  layer 1..L-1 tcgen05 GEMM (TMA both operands)
//     heads + PPO loss + dZ of the last hidden layer (SIMT fp32)
//     bwd  layer L-1..1 tcgen05 GEMM dA = dZ W^T, f' epilogue
//     dW   all layers   tcgen05 split-K GEMM act^T dZ (+ bias-gradient column sums ones x dZ) -> per-split partials
//     optimizer         partial reduction [+ NCCL all-reduce] + global-norm clip + Adam + bf16 images
// The whole sequence is captured into one CUDA graph per pointer set.
#include <cuda.h>
#include <dlfcn.h>
#include <math.h>
#include <algorithm>
#include <nccl.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <vector>

#include "common.cuh"
#include "minppo_internal.h"
#include "umma_gemm.cuh"
#include "fused_step.cuh"
#include "dwopt.cuh"
#include "policy_fused.cuh"

namespace minppo {

// ------------------------------------------------------------------------------------------
// errors
// ------------------------------------------------------------------------------------------
static thread_local char g_err[512] = "";
void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}
#define CK(call)                                                                          \
  do {                                                                                    \
    cudaError_t e_ = (call);                                                              \
    if (e_ != cudaSuccess) {                                                              \
      set_error("%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
      return MINPPO_ERR_CUDA;                                                             \
    }                                                                                     \
  } while (0)
#define RET(call)            \
  do {                       \
    int r_ = (call);         \
    if (r_ != 0) return r_;  \
  } while (0)

// ------------------------------------------------------------------------------------------
// driver entry point for tensor-map encoding (no link-time libcuda dependency)
// ------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  }
  return fn;
}
// bf16 2-D row-major tensor [outer][inner] with `ld` elements per row; box {box_inner, box_outer}; 128B swizzle
static int make_tmap(CUtensorMap* m, const void* base, uint64_t inner, uint64_t outer, uint64_t ld,
                     uint32_t box_inner, uint32_t box_outer) {
  EncodeTiledFn fn = get_encode_fn();
  if (!fn) { set_error("cuTensorMapEncodeTiled entry point not available"); return MINPPO_ERR_CUDA; }
  cuuint64_t dims[2] = {inner, outer};
  cuuint64_t strides[1] = {ld * 2};
  cuuint32_t box[2] = {box_inner, box_outer};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled failed (%d)", static_cast<int>(r)); return MINPPO_ERR_CUDA; }
  return 0;
}

// fp32 3-D tensor [d2][d1][d0] (d0 contiguous), box {32, 128, 1}, 128B swizzle: split-K partial stores
static int make_tmap_f32_3d(CUtensorMap* m, const void* base, uint64_t d0, uint64_t d1, uint64_t d2) {
  EncodeTiledFn fn = get_encode_fn();
  if (!fn) { set_error("cuTensorMapEncodeTiled entry point not available"); return MINPPO_ERR_CUDA; }
  cuuint64_t dims[3] = {d0, d1, d2};
  cuuint64_t strides[2] = {d0 * 4, d0 * d1 * 4};
  cuuint32_t box[3] = {32, 128, 1};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = fn(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<void*>(base), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled (f32 3d) failed (%d)", static_cast<int>(r)); return MINPPO_ERR_CUDA; }
  return 0;
}

// ------------------------------------------------------------------------------------------
// NCCL, loaded lazily so that single-GPU use never needs the library
// ------------------------------------------------------------------------------------------
struct NcclApi {
  ncclResult_t (*GetUniqueId)(ncclUniqueId*);
  ncclResult_t (*CommInitRank)(ncclComm_t*, int, ncclUniqueId, int);
  ncclResult_t (*AllReduce)(const void*, void*, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t);
  ncclResult_t (*Broadcast)(const void*, void*, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t);
  ncclResult_t (*GroupStart)();
  ncclResult_t (*GroupEnd)();
  ncclResult_t (*CommDestroy)(ncclComm_t);
  const char* (*GetErrorString)(ncclResult_t);
  bool ok;
};
static NcclApi* nccl_api() {
  static NcclApi api = {};
  static bool tried = false;
  if (!tried) {
    tried = true;
    void* h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
    if (!h) h = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
    if (h) {
      api.GetUniqueId = reinterpret_cast<decltype(api.GetUniqueId)>(dlsym(h, "ncclGetUniqueId"));
      api.CommInitRank = reinterpret_cast<decltype(api.CommInitRank)>(dlsym(h, "ncclCommInitRank"));
      api.AllReduce = reinterpret_cast<decltype(api.AllReduce)>(dlsym(h, "ncclAllReduce"));
      api.Broadcast = reinterpret_cast<decltype(api.Broadcast)>(dlsym(h, "ncclBroadcast"));
      api.GroupStart = reinterpret_cast<decltype(api.GroupStart)>(dlsym(h, "ncclGroupStart"));
      api.GroupEnd = reinterpret_cast<decltype(api.GroupEnd)>(dlsym(h, "ncclGroupEnd"));
      api.CommDestroy = reinterpret_cast<decltype(api.CommDestroy)>(dlsym(h, "ncclCommDestroy"));
      api.GetErrorString = reinterpret_cast<decltype(api.GetErrorString)>(dlsym(h, "ncclGetErrorString"));
      api.ok = api.GetUniqueId && api.CommInitRank && api.AllReduce && api.Broadcast && api.GroupStart && api.GroupEnd &&
               api.CommDestroy && api.GetErrorString;
    }
  }
  return api.ok ? &api : nullptr;
}

// ------------------------------------------------------------------------------------------
// parameter layout
// ------------------------------------------------------------------------------------------
struct LeafInfo {
  int net;       // 0 actor (MLP_0), 1 critic (MLP_1), 2 log_std
  int layer;     // Dense_<layer>
  int is_kernel;
  long long offset, rows, cols;
};
static long long build_layout(const minppo_config& c, std::vector<LeafInfo>* out) {
  long long off = 0;
  const int L = c.num_layers;
  for (int net = 0; net < 2; ++net) {
    long long fan_in = c.obs_dim;
    for (int l = 0; l <= L; ++l) {
      const long long o = l < L ? c.hidden_size : (net == 0 ? c.act_dim : 1);
      if (out) out->push_back({net, l, 0, off, 1, o});
      off += o;
      if (out) out->push_back({net, l, 1, off, fan_in, o});
      off += fan_in * o;
      fan_in = o;
    }
  }
  if (out) out->push_back({2, 0, 0, off, 1, c.act_dim});
  off += c.act_dim;
  return off;
}

static int validate_config(const minppo_config& c) {
  if (c.num_envs <= 0 || c.num_steps <= 0 || c.num_minibatches <= 0 || c.update_epochs <= 0 || c.obs_dim <= 0 ||
      c.act_dim <= 0 || c.num_layers < 1) {
    set_error("non-positive size in minppo_config");
    return MINPPO_ERR_ARG;
  }
  if (c.hidden_size % 64 != 0 || c.hidden_size > MAX_HIDDEN || c.hidden_size <= 0) {
    set_error("model.hidden_size=%d unsupported: must be a multiple of 64 and <= %d", c.hidden_size, MAX_HIDDEN);
    return MINPPO_ERR_UNSUPPORTED;
  }
  // wider than one GEMM tile: every hidden layer of both nets is two column groups of the weight-gradient launch
  if (c.hidden_size > GEMM_MAXN && 2 * c.num_layers * 2 > GEMM_MAX_GROUPS) {
    set_error("num_layers=%d unsupported at model.hidden_size=%d: hidden_size > %d allows num_layers <= %d", c.num_layers,
              c.hidden_size, GEMM_MAXN, GEMM_MAX_GROUPS / 4);
    return MINPPO_ERR_UNSUPPORTED;
  }
  if (c.act_dim > MAX_ACT_DIM) {
    set_error("act_dim=%d unsupported (<= %d)", c.act_dim, MAX_ACT_DIM);
    return MINPPO_ERR_UNSUPPORTED;
  }
  if (2 * (c.num_layers + 1) * 2 + 1 > OPT_TAB_LEAVES) { set_error("too many layers"); return MINPPO_ERR_UNSUPPORTED; }
  if (2 * c.num_layers > 6) { set_error("num_layers=%d unsupported (<= 3)", c.num_layers); return MINPPO_ERR_UNSUPPORTED; }
  const long long B = static_cast<long long>(c.num_envs) * c.num_steps;
  const long long mb = B / c.num_minibatches;
  if (mb * c.num_minibatches != B) {
    // train.py:253-255
    set_error("`batch_size` must be equal to `num_steps * num_envs`");
    return MINPPO_ERR_ARG;
  }
  if (c.world_size < 1 || c.rank < 0 || c.rank >= c.world_size || c.num_envs % c.world_size != 0) {
    set_error("bad sharding: world_size=%d rank=%d num_envs=%d", c.world_size, c.rank, c.num_envs);
    return MINPPO_ERR_ARG;
  }
  if (c.prng_mode != MINPPO_PRNG_LEGACY && c.prng_mode != MINPPO_PRNG_PARTITIONABLE) {
    set_error("bad prng_mode %d", c.prng_mode);
    return MINPPO_ERR_ARG;
  }
  if (B > 0x7fffffffLL) { set_error("batch too large"); return MINPPO_ERR_UNSUPPORTED; }
  return 0;
}

}  // namespace minppo

using namespace minppo;

// ------------------------------------------------------------------------------------------
// context
// ------------------------------------------------------------------------------------------
struct NetBufs {
  std::vector<__nv_bfloat16*> act;     // act[l], l = 1..L   [M_pad][H]
  std::vector<__nv_bfloat16*> dz;      // dz[l],  l = 1..L   [M_pad][H]
  std::vector<__nv_bfloat16*> wn;      // wn[l],  l = 0..L-1 [in_pad_l][H]: bf16 image of the kernel as stored ([in][out]; rows >= in are 0)
  std::vector<float*> dw_part;         // dw_part[l], l = 0..L-1 [S][in_l][H]
  uint8_t* w2img;                      // head kernel^T bf16 hi / lo image (16 KB, fused path)
  std::vector<float*> dbias;           // dbias[l], l = 0..L-1 [S][H]: bias-gradient partials from the dW GEMM (ones x dz[l+1])
  std::vector<CUtensorMap> m_act_k, m_act_mn, m_dz_k, m_dz_mn, m_wn_mn, m_wn, m_dw;
  std::vector<CUtensorMap> m_wn_h;     // m_wn_h[l]: box {64 out, 32 in} -- half-k-block stages of the fused step kernel (MN-major B)
  CUtensorMap m_w1k_h;                 // wn[1]: box {64 out, H/2 in} -- (k-block, N half) stages of the fused kernel's dH1 GEMM (K-major B)
  // m_wn_mn[l]: box {64 out, 64 in} -- MN-major B of the forward GEMMs;  m_wn[2 l + j] (l >= 1): box {64 out, N_j in} -- K-major
  // B of dX for column group j (col_group)
};

struct UpdatePtrs {
  float *params, *mu, *nu;
  int32_t* count;
  const float *obs, *action, *value, *reward, *log_prob;
  const uint8_t* done;
  const float* last_val;
  const uint32_t* key_in;
  uint32_t* key_out;
  float* losses_out;
  float* stats_out;
  bool operator==(const UpdatePtrs& o) const { return memcmp(this, &o, sizeof(*this)) == 0; }
};

struct minppo_ctx {
  minppo_config cfg;
  int device, sm_count;
  int T, N, Nl, n0, M, E, L, H, D, Dp, A;
  long long B, Bl, P;
  int mb, m_tiles, tiles64;   // 128- and 64-row tiles of plan.row_cap
  struct minppo_plan plan;    // kernel path (minppo_plan)
  std::vector<LeafInfo> leaves;
  // device buffers
  std::vector<void*> allocs;
  float *adv, *tgt, *stats, *gflat, *block_ss, *head_part, *gnorms, *losses_scratch;
  long long* trace;           // debug cycle stamps of the fused kernel [2*m_tiles][FS_TRACE_SLOTS]
  long long* trace2;          // debug cycle stamps of the dwopt kernel [sm_count][8]
  bool trace_on;
  int32_t *perms, *rowidx, *counts;
  int32_t* perm_tmp;          // world_size > 1: the epochs THIS rank sorts ([ceil(E / W)][B]); broadcast into perms
  void* perm_ws;
  size_t perm_ws_bytes;
  __nv_bfloat16* obs_img;
  __nv_bfloat16* xg;           // gathered observation rows of the current minibatch [M_pad][Dp] (fused path)
  CUtensorMap m_xg_k, m_xg_mn;
  unsigned long long* barrier;
  unsigned int* dw_done;      // dwopt_kernel's split-K tile completion counters [sm_count + 2][DWOPT_DONE_STRIDE]
  int* err_flag;
  NetBufs net[2];
  int head_stride, po_w3a, po_b3a, po_w3c, po_b3c, po_logstd, po_loss;
  int po_db[2][2];            // fused path: [net][layer] hidden-bias gradient partials (column sums of dZ), H floats each
  HeadOffsets head;           // arena offsets of the output-head leaves
  // graph cache
  cudaStream_t cap_stream;
  cudaStream_t side_stream;    // fork/join branch of an update: operand staging (observation + weight images) runs beside
  cudaEvent_t ev_fork, ev_join;  // the GAE -> permutation -> row-list chain (independent until the first minibatch step)
  // One instantiated graph per POINTER SET, least recently used first out (a caller that alternates between a few
  // buffer sets -- ping-pong rng keys, double-buffered trajectories -- replays instead of re-capturing ~290 nodes).
  struct CachedGraph { cudaGraph_t graph; cudaGraphExec_t exec; UpdatePtrs ptrs; long long launches; };
  std::vector<CachedGraph> graphs;
  long long launches;
  // nccl
  ncclComm_t comm;
  bool have_comm;
  // gradient exchange over peer memory (dwopt.cuh PeerXchg)
  float* xchg;                // [stage | pad | result] (world_size > 1; dwopt.cuh PeerXchg), exported by CUDA IPC
  unsigned int* xseq;
  PeerXchg px;
  bool peers_set;
  void* peer_ptr[MINPPO_MAX_RANKS];
  // policy / value inference for the rollout (minppo_policy_step): bf16 image of last_obs and the hidden activations
  int pol_tiles;               // 128-row tiles over the Nl envs of this rank
  __nv_bfloat16* pol_img;      // [pol_tiles * 128][Dp]
  __nv_bfloat16* pol_act[2][MINPPO_MAX_LEAVES];   // [net][l], l = 1..L: [pol_tiles * 128][H]
  CUtensorMap m_pol_img_k, m_pol_act_k[2][MINPPO_MAX_LEAVES];
  // per-kernel-class event profiling (eager mode only)
  bool profiling;
  std::vector<cudaEvent_t> prof_events;      // pairs (begin, end)
  std::vector<int> prof_class;               // class of each pair
  size_t prof_used;
};

enum : int { PC_GAE = 0, PC_PERM, PC_PREP, PC_OBS_IMAGE, PC_WEIGHT_IMAGES, PC_FWD_GEMM, PC_HEAD_LOSS, PC_BWD_GEMM,
             PC_DW_GEMM, PC_OPT, PC_ALLREDUCE, PC_COUNT };

// RAII: records an event pair around the launches issued in its scope when profiling is on.
struct ProfScope {
  minppo_ctx* c; cudaStream_t s; size_t idx; bool on;
  ProfScope(minppo_ctx* ctx, int cls, cudaStream_t stream) : c(ctx), s(stream), idx(0), on(ctx->profiling) {
    if (!on) return;
    if (c->prof_used + 2 > c->prof_events.size()) {
      cudaEvent_t a, b;
      cudaEventCreate(&a); cudaEventCreate(&b);
      c->prof_events.push_back(a); c->prof_events.push_back(b);
      c->prof_class.push_back(cls);
    } else {
      c->prof_class[c->prof_used / 2] = cls;
    }
    idx = c->prof_used;
    c->prof_used += 2;
    cudaEventRecord(c->prof_events[idx], s);
  }
  ~ProfScope() { if (on) cudaEventRecord(c->prof_events[idx + 1], s); }
};
#define PROF(cls) ProfScope prof_scope_(c, cls, stream)

namespace minppo {

template <typename T>
static int dev_alloc(minppo_ctx* c, T** p, size_t n, bool zero = true) {
  void* q = nullptr;
  const size_t bytes = (n * sizeof(T) + 255) & ~static_cast<size_t>(255);
  CK(cudaMalloc(&q, bytes));
  if (zero) CK(cudaMemset(q, 0, bytes));
  c->allocs.push_back(q);
  *p = reinterpret_cast<T*>(q);
  return 0;
}

__global__ void fill_u32_kernel(uint32_t* p, size_t n, uint32_t v) {
  for (size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x; i < n; i += static_cast<size_t>(gridDim.x) * blockDim.x) p[i] = v;
}

static const LeafInfo& find_leaf(const minppo_ctx* c, int net, int layer, int is_kernel) {
  for (const auto& l : c->leaves)
    if (l.net == net && l.layer == layer && l.is_kernel == is_kernel) return l;
  return c->leaves[0];
}

// Column range j of a hidden layer split into n groups: n == 1 is the whole of H; n == 2 puts H / 2 rounded up to a whole
// 64-column panel first (512 -> 256 + 256, 448 -> 256 + 192, 320 -> 192 + 128): both widths are multiples of 64 and <= 256.
static void col_group(int H, int n, int j, int* n_off, int* N) {
  const int first = n == 1 ? H : (H / 2 + 63) / 64 * 64;
  *n_off = j == 0 ? 0 : first;
  *N = j == 0 ? first : H - first;
}

static int act_kind(const minppo_ctx* c, int net) {
  if (net == 1 || !c->cfg.use_tanh) return ACT_RELU;        // critic is relu always (train.py:82)
  return c->cfg.fast_tanh ? ACT_TANH_FAST : ACT_TANH;
}

// cudaFuncSetAttribute applies to the CURRENT device: set on every context creation (a process may hold contexts on
// several GPUs; the calls are cheap and idempotent).
static int init_kernel_attrs() {
  CK(cudaFuncSetAttribute(umma_gemm_kernel<EPI_ACT>, cudaFuncAttributeMaxDynamicSharedMemorySize, GEMM_SMEM_BYTES));
  CK(cudaFuncSetAttribute(umma_gemm_kernel<EPI_DACT>, cudaFuncAttributeMaxDynamicSharedMemorySize, GEMM_SMEM_BYTES));
  CK(cudaFuncSetAttribute(umma_gemm_kernel<EPI_PARTIAL>, cudaFuncAttributeMaxDynamicSharedMemorySize, GEMM_SMEM_BYTES));
  if (head_loss_init()) { set_error("head_loss_init failed"); return MINPPO_ERR_CUDA; }
  if (policy_head_init()) { set_error("policy_head_init failed"); return MINPPO_ERR_CUDA; }
  CK(cudaFuncSetAttribute(fused_step_kernel<16>, cudaFuncAttributeMaxDynamicSharedMemorySize, FsLayout<16>::BYTES));
  CK(cudaFuncSetAttribute(fused_step_kernel<32>, cudaFuncAttributeMaxDynamicSharedMemorySize, FsLayout<32>::BYTES));
  CK(cudaFuncSetAttribute(dwopt_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, GEMM_SMEM_BYTES));
  CK(cudaFuncSetAttribute(dwopt_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, GEMM_SMEM_BYTES));
  CK(cudaFuncSetAttribute(dwopt_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, GEMM_SMEM_BYTES));
  CK(policy_fused_init_attrs());
  return 0;
}

template <int EPI>
static int launch_gemm(const GemmParams& p_in, int ctas, cudaStream_t stream, bool pdl = false) {
  GemmParams p = p_in;
  gemm_finalize(p);
  const cudaError_t e = launch_kernel(umma_gemm_kernel<EPI>, ctas, GEMM_THREADS, GEMM_SMEM_BYTES, stream, pdl, p);
  if (e != cudaSuccess) { set_error("umma_gemm launch failed: %s", cudaGetErrorString(e)); return MINPPO_ERR_CUDA; }
  return 0;
}

// ---- optimizer argument block ---------------------------------------------------------------
static void fill_opt_args(const minppo_ctx* c, const UpdatePtrs& u, OptArgs* o) {
  memset(o, 0, sizeof(*o));
  const minppo_config& cfg = c->cfg;
  const int L = c->L, H = c->H;
  const int head_parts = c->plan.fused ? c->m_tiles : c->tiles64;   // head partials per minibatch
  int n = 0;
  for (const auto& lf : c->leaves) {
    OptLeaf& ol = o->leaf[n++];
    ol.offset = static_cast<int>(lf.offset);
    ol.cols = static_cast<int>(lf.cols);
    if (lf.net == 2) {                         // log_std
      ol.grad_src = c->head_part; ol.src_offset = c->po_logstd; ol.nparts = head_parts; ol.part_stride = c->head_stride;
      ol.grad_bias = cfg.rank == 0 ? -static_cast<float>(cfg.ent_coef) : 0.f;
    } else if (lf.layer == L) {                // output heads
      ol.grad_src = c->head_part; ol.nparts = head_parts; ol.part_stride = c->head_stride;
      if (lf.is_kernel) { ol.src_offset = lf.net == 0 ? c->po_w3a : c->po_w3c; ol.img_w2 = c->plan.fused ? c->net[lf.net].w2img : nullptr; ol.ap = c->plan.ap; }
      else ol.src_offset = lf.net == 0 ? c->po_b3a : c->po_b3c;
    } else if (lf.is_kernel) {                 // hidden kernels: split-K partials of the dW GEMM
      const int in_l = lf.layer == 0 ? c->D : H;
      ol.grad_src = c->net[lf.net].dw_part[lf.layer]; ol.src_offset = 0; ol.nparts = c->plan.S; ol.part_stride = in_l * H; ol.late = 1;
      ol.img_n = c->net[lf.net].wn[lf.layer];
    } else if (c->plan.fused) {                // hidden biases, fused path: per-tile column sums of dz[l+1] from the fused step kernel
      ol.grad_src = c->head_part; ol.src_offset = c->po_db[lf.net][lf.layer]; ol.nparts = head_parts; ol.part_stride = c->head_stride;
    } else {                                   // hidden biases: column sums of dz[l+1], computed by the dW GEMM (ones x dz)
      ol.grad_src = c->net[lf.net].dbias[lf.layer]; ol.src_offset = 0; ol.nparts = c->plan.S;
      ol.part_stride = H; ol.late = 1;
    }
  }
  o->nleaves = n;
  o->n_early = 0;
  for (int i = 0; i < n; ++i) {
    o->leaf[i].size = (i + 1 < n ? o->leaf[i + 1].offset : static_cast<int>(c->P)) - o->leaf[i].offset;
    if (!o->leaf[i].late) o->n_early += o->leaf[i].size;
  }
  o->P = static_cast<int>(c->P);
  o->A = c->A;
  o->gflat = c->gflat;
  o->loss_src = c->head_part; o->loss_src_offset = c->po_loss; o->loss_nparts = head_parts; o->loss_part_stride = c->head_stride;
  o->params = u.params; o->mu = u.mu; o->nu = u.nu; o->count = u.count;
  o->block_ss = c->block_ss; o->barrier = c->barrier; o->err_flag = c->err_flag;
  o->off_logstd = c->head.logstd;
  o->anneal = cfg.anneal_lr ? 1 : 0;
  o->anneal_div = c->mb * c->E;                                                     // train.py:100
  const long long nu = cfg.total_timesteps / cfg.num_steps / cfg.num_envs;          // train.py:93
  o->num_updates = static_cast<int>(nu > 0x7fffffffLL ? 0x7fffffffLL : nu);
  o->lr = static_cast<float>(cfg.anneal_lr ? cfg.training_lr : cfg.opt_lr);
  o->max_norm = static_cast<float>(cfg.max_grad_norm);
  o->b1 = static_cast<float>(cfg.adam_b1); o->b2 = static_cast<float>(cfg.adam_b2);
  o->one_minus_b1 = static_cast<float>(1.0 - cfg.adam_b1); o->one_minus_b2 = static_cast<float>(1.0 - cfg.adam_b2);
  o->eps = static_cast<float>(cfg.adam_eps); o->eps_root = static_cast<float>(cfg.adam_eps_root);
  o->inv_mb = static_cast<float>(1.0 / c->mb);
  o->vf_coef = static_cast<float>(cfg.vf_coef); o->ent_coef = static_cast<float>(cfg.ent_coef);
  o->entropy_const = static_cast<float>(c->A * (0.5 + 0.5 * log(2.0 * M_PI)));
}

static int nccl_allreduce(minppo_ctx* c, float* buf, size_t n, cudaStream_t stream) {
  NcclApi* api = nccl_api();
  ncclResult_t r = api->AllReduce(buf, buf, n, ncclFloat, ncclSum, c->comm, stream);
  if (r != ncclSuccess) { set_error("ncclAllReduce failed: %s", api->GetErrorString(r)); return MINPPO_ERR_NCCL; }
  return 0;
}

// ---- parameter blocks of the per-minibatch kernels ----
static void fill_loss_operands(const minppo_ctx* c, const UpdatePtrs& u, int s, LossOperands* lo) {
  lo->rowidx = c->rowidx; lo->count = c->counts; lo->cap = c->plan.row_cap; lo->step = s;
  lo->adv_sum = c->stats; lo->adv_sq = c->stats + c->E * c->M;
  lo->action = u.action; lo->v_old = u.value; lo->logp_old = u.log_prob; lo->adv = c->adv; lo->tgt = c->tgt;
  lo->inv_mb = static_cast<float>(1.0 / c->mb);
  lo->clip_eps = static_cast<float>(c->cfg.clip_eps); lo->vf_coef = static_cast<float>(c->cfg.vf_coef);
}

static void fill_fused_params(minppo_ctx* c, const UpdatePtrs& u, int s, FusedParams* pp) {
  FusedParams& p = *pp;
  memset(&p, 0, sizeof(p));
  const int H = c->H;
  for (int net = 0; net < 2; ++net) {
    FusedNet& g = p.net[net];
    NetBufs& nb = c->net[net];
    g.tm_w0 = nb.m_wn_h[0]; g.tm_w1 = nb.m_wn_h[1]; g.tm_w1k = nb.m_w1k_h;
    g.tm_h1 = nb.m_act_k[1]; g.tm_dz2 = nb.m_dz_k[2]; g.tm_dz1 = nb.m_dz_k[1];
    g.b0 = u.params + find_leaf(c, net, 0, 0).offset;
    g.b1 = u.params + find_leaf(c, net, 1, 0).offset;
    g.w2img = reinterpret_cast<const uint4*>(nb.w2img);
    g.b2 = u.params + (net == 0 ? c->head.b3a : c->head.b3c);
    g.act = act_kind(c, net);
    g.aout = net == 0 ? c->A : 1;
    g.po_w2 = net == 0 ? c->po_w3a : c->po_w3c;
    g.po_b2 = net == 0 ? c->po_b3a : c->po_b3c;
    g.po_loss = c->po_loss + (net == 0 ? 1 : 0);          // [0] = sum max(vl, vlc), [1] = sum min(l1, l2)
    g.po_stat = c->po_loss + (net == 0 ? 3 : 2);          // [2] value-clip count; [3] approx-KL sum, [4] ratio-clip count
    g.po_db0 = c->po_db[net][0]; g.po_db1 = c->po_db[net][1];
  }
  fill_loss_operands(c, u, s, &p.loss);
  p.obs_img = c->obs_img; p.tm_xg = c->m_xg_k;
  p.log_std = u.params + c->head.logstd;
  p.part = c->head_part; p.part_stride = c->head_stride; p.po_logstd = c->po_logstd;
  p.H = H; p.A = c->A; p.Dp = c->Dp; p.m_tiles = c->m_tiles;
  p.trace = c->trace_on ? c->trace : nullptr;
}

// weight-gradient GEMM groups + optimizer block + per-update arrays
static void fill_dwopt_params(minppo_ctx* c, const UpdatePtrs& u, DwOptParams* dpp) {
  DwOptParams& dp = *dpp;
  memset(&dp, 0, sizeof(dp));
  const int L = c->L, H = c->H;
  GemmParams& p = dp.gemm;
  int cta = 0, ng = 0;
  int tile_first[2][4], tile_count[2][4], tile_split[2][4];   // split-K output tiles of each (net, layer): dwopt.cuh counters
  for (int net = 0; net < 2; ++net) {
    NetBufs& nb = c->net[net];
    for (int l = 0; l < L; ++l) {
      tile_first[net][l] = cta / c->plan.S;
      tile_count[net][l] = 0;
      for (int nh = 0; nh < c->plan.dw_nsplit; ++nh) {
      GemmGroup& g = p.g[ng++];
      g.cta_begin = cta;
      const int in_l = l == 0 ? c->D : H;
      const int in_pad = l == 0 ? c->Dp : H;
      if (l == 0 && c->plan.fused) { g.amode = A_TMA_MN; g.tmA = c->m_xg_mn; }   // rows gathered by the fused kernel
      else if (l == 0) { g.amode = A_GATHER_MN; g.rowidx = c->rowidx; g.gimage = c->obs_img; g.ldg = c->Dp; }      // row list: per step
      else { g.amode = A_TMA_MN; g.tmA = nb.m_act_mn[l]; }
      g.bmode = B_TMA_MN; g.tmB = nb.m_dz_mn[l + 1];
      g.kb_total = c->plan.row_cap / 64;
      g.k_count = nullptr;                                    // per step (counts[] below)
      g.tmC = nb.m_dw[l];
      g.colsum_out = c->plan.fused ? nullptr : nb.dbias[l]; // fused path: the bias gradients come from the fused step kernel
      col_group(H, c->plan.dw_nsplit, nh, &g.n_off, &g.N);
      g.ldc = H;
      g.m_tiles = (in_pad + 127) / 128; g.splits = c->plan.S; g.m_store = in_l;
      cta += g.m_tiles * g.splits;
      tile_count[net][l] += g.m_tiles;
      if (nh == 0) tile_split[net][l] = g.N;
      }
    }
  }
  p.ngroups = ng;
  gemm_finalize(p);
  fill_opt_args(c, u, &dp.opt);
  // A GEMM grid past one CTA per SM runs as a launch of its own in front of dwopt (enqueue_step): dwopt then has no GEMM
  // CTAs, and its late leaves wait for no counter (tile fields 0), since their partials are complete when it starts.
  dp.gemm_ctas = c->plan.two_launch ? 0 : c->plan.dw_gemm_ctas;
  for (size_t i = 0; i < c->leaves.size() && dp.gemm_ctas; ++i) {
    OptLeaf& ol = dp.opt.leaf[i];
    const LeafInfo& lf = c->leaves[i];
    if (!ol.late) continue;                                  // hidden kernels (and, layer-wise path, hidden biases)
    ol.tile0 = 1 + tile_first[lf.net][lf.layer];             // counter 0: the small-leaf pre-reducers
    ol.tile_n = tile_count[lf.net][lf.layer];
    ol.tile_split = lf.is_kernel ? tile_split[lf.net][lf.layer] : 0;
  }
  dp.done = c->dw_done;
  dp.opt.losses_out = u.losses_out ? u.losses_out : c->losses_scratch;
  dp.losses_stride = u.losses_out ? 4 : 0;
  dp.opt.gnorm_out = c->gnorms;
  dp.opt.stats_out = u.stats_out;
  dp.ridx_base = c->rowidx; dp.counts = c->counts; dp.cap = c->plan.row_cap; dp.EM = c->E * c->M;
  dp.padded = c->plan.padded;
  dp.part_rows = c->plan.fused ? 128 : 64;
  dp.obs_img = c->obs_img; dp.obs_ld = c->Dp;
  dp.trace = c->trace_on ? c->trace2 : nullptr;
}

// The NCCL fallback's second dwopt launch, which only applies the all-reduced gradient: gflat holds it (P floats, then the
// LOSS_SUMS loss sums), and it becomes the single partial of every leaf and of the loss sums.  The reduction phase then copies
// gflat onto itself and forms the global norm; phase 3 runs clip + Adam and writes the weight images as usual.  Every leaf
// is "early": the late path issues 16-byte loads, and gflat + a leaf offset is only 4-byte aligned.  grad_bias is 0
// because rank 0 added -ent_coef to the log_std gradient before the all-reduce, and padded is 0 because the live-tile
// cap counts per-tile partials, which gflat is not.
static void fill_apply_only(const minppo_ctx* c, DwOptParams* dpp) {
  DwOptParams& dp = *dpp;
  OptArgs& o = dp.opt;
  for (int i = 0; i < o.nleaves; ++i) {
    OptLeaf& ol = o.leaf[i];
    ol.late = 0; ol.grad_src = c->gflat; ol.src_offset = ol.offset; ol.nparts = 1; ol.grad_bias = 0.f;
  }
  o.n_early = o.P;
  o.loss_src = c->gflat; o.loss_src_offset = o.P; o.loss_nparts = 1;
  o.do_apply = 1;
  dp.gemm_ctas = 0;
  dp.padded = 0;
}

// One net's operands in the forward GEMM of one hidden layer
struct FwdOperands {
  const int32_t* rowidx;        // A gathered by index from the observation image (layer 0 of a minibatch), or null:
  const CUtensorMap* a_map;     //   A through this K-major map [rows][in]
  __nv_bfloat16* out;           // [m_tiles * 128][H]
};
// Forward GEMM of hidden layer l, out = f(A W_l + b_l), for nets first_net..1 (the critic-only bootstrap value starts at
// net 1): one group per (net, column group) over m_tiles 128-row tiles.
static void fill_forward_gemm(const minppo_ctx* c, int l, const float* params, int first_net, int m_tiles,
                              const FwdOperands (&op)[2], GemmParams* pp) {
  GemmParams& p = *pp;
  memset(&p, 0, sizeof(p));
  const int H = c->H;
  int ng = 0;
  for (int i = first_net * c->plan.hsplit; i < 2 * c->plan.hsplit; ++i, ++ng) {
    const int net = i / c->plan.hsplit;
    GemmGroup& g = p.g[ng];
    g.cta_begin = ng * m_tiles;
    col_group(H, c->plan.hsplit, i % c->plan.hsplit, &g.n_off, &g.N);
    g.bmode = B_TMA_MN;                   // kernel image as stored [in = k][out = n]
    g.tmB = c->net[net].m_wn_mn[l];
    if (op[net].rowidx) { g.amode = A_GATHER_K; g.rowidx = op[net].rowidx; g.gimage = c->obs_img; g.ldg = c->Dp; }
    else { g.amode = A_TMA_K; g.tmA = *op[net].a_map; }
    g.kb_total = (l == 0 ? c->Dp : H) / 64;
    g.out = op[net].out; g.ldo = H;
    g.bias = params + find_leaf(c, net, l, 0).offset;
    g.act = act_kind(c, net);
    g.m_tiles = m_tiles; g.splits = 1; g.m_store = m_tiles * 128;
  }
  p.ngroups = ng;
}

// bf16 weight images of the fp32 arena `params` (what the GEMMs and the fused kernels read)
static int enqueue_weight_images(const minppo_ctx* c, const float* params, cudaStream_t stream) {
  UpdatePtrs u;
  memset(&u, 0, sizeof(u));
  u.params = const_cast<float*>(params);               // weight_images only reads the arena
  OptArgs o;
  fill_opt_args(c, u, &o);
  return weight_images_launch(o, stream);
}

// ---- one minibatch step --------------------------------------------------------------------
static int enqueue_step(minppo_ctx* c, const UpdatePtrs& u, int s, cudaStream_t stream) {
  const int L = c->L, H = c->H;
  const int32_t* ridx = c->rowidx + static_cast<size_t>(s) * c->plan.row_cap;
  // programmatic dependent launch between the per-minibatch kernels (fused path only; common.cuh)
  const bool pdl = c->plan.fused && !c->profiling;
  if (c->plan.fused) {
    // forward + heads + loss + backward-to-dZ of both nets in one launch (fused_step.cuh)
    FusedParams p;
    fill_fused_params(c, u, s, &p);
    PROF(PC_FWD_GEMM);
    const cudaError_t e = c->plan.ap == 16
        ? launch_kernel(fused_step_kernel<16>, 2 * c->m_tiles, FS_THREADS, FsLayout<16>::BYTES, stream, pdl, p)
        : launch_kernel(fused_step_kernel<32>, 2 * c->m_tiles, FS_THREADS, FsLayout<32>::BYTES, stream, pdl, p);
    if (e != cudaSuccess) { set_error("fused_step launch failed: %s", cudaGetErrorString(e)); return MINPPO_ERR_CUDA; }
    c->launches++;
  } else {
  // forward
  for (int l = 0; l < L; ++l) {
    FwdOperands op[2];
    for (int net = 0; net < 2; ++net)
      op[net] = {l == 0 ? ridx : nullptr, &c->net[net].m_act_k[l], c->net[net].act[l + 1]};
    GemmParams p;
    fill_forward_gemm(c, l, u.params, 0, c->m_tiles, op, &p);
    PROF(PC_FWD_GEMM);
    RET(launch_gemm<EPI_ACT>(p, p.ngroups * c->m_tiles, stream));
    c->launches++;
  }
  // heads + loss + dz[L]
  {
    HeadLossArgs a;
    memset(&a, 0, sizeof(a));
    a.h_a = c->net[0].act[L]; a.h_c = c->net[1].act[L];
    a.dz_a = c->net[0].dz[L]; a.dz_c = c->net[1].dz[L];
    a.params = u.params;
    fill_loss_operands(c, u, s, &a.loss);
    a.partials = c->head_part; a.partial_stride = c->head_stride;
    a.po_w3a = c->po_w3a; a.po_b3a = c->po_b3a; a.po_w3c = c->po_w3c; a.po_b3c = c->po_b3c;
    a.po_logstd = c->po_logstd; a.po_loss = c->po_loss;
    a.off = c->head;
    a.H = H; a.A = c->A; a.ldh = H;
    a.act_a = act_kind(c, 0) == ACT_RELU ? ACTK_RELU : ACTK_TANH; a.act_c = ACTK_RELU;
    PROF(PC_HEAD_LOSS);
    RET(head_loss_launch(a, c->tiles64, stream));
    c->launches++;
  }
  // backward through hidden layers: dz[l] = (dz[l+1] W_l^T) * f'(act[l])
  for (int l = L - 1; l >= 1; --l) {
    GemmParams p;
    memset(&p, 0, sizeof(p));
    p.ngroups = 2 * c->plan.hsplit;
    for (int i = 0; i < p.ngroups; ++i) {
      const int net = i / c->plan.hsplit, j = i % c->plan.hsplit;
      GemmGroup& g = p.g[i];
      NetBufs& nb = c->net[net];
      g.cta_begin = i * c->m_tiles;
      col_group(H, c->plan.hsplit, j, &g.n_off, &g.N);
      g.amode = A_TMA_K; g.tmA = nb.m_dz_k[l + 1];
      g.bmode = B_TMA_K; g.tmB = nb.m_wn[2 * l + j];
      g.kb_total = H / 64;
      g.out = nb.dz[l]; g.ldo = H;
      g.hprev = nb.act[l]; g.ldh = H;
      g.act = act_kind(c, net);
      g.m_tiles = c->m_tiles; g.splits = 1; g.m_store = c->plan.row_cap;
    }
    PROF(PC_BWD_GEMM);
    RET(launch_gemm<EPI_DACT>(p, p.ngroups * c->m_tiles, stream));
    c->launches++;
  }
  }  // !fused
  // weight gradients dW_l = act[l]^T dz[l+1] (split-K over minibatch rows), then the optimizer: ONE dwopt launch
  // (dwopt.cuh) when the GEMM grid fits one CTA per SM; otherwise the stand-alone GEMM kernel, then dwopt without GEMM
  // CTAs.  Env-sharded ranks without the peer-memory exchange then all-reduce the gradient sums over NCCL and apply them
  // with a second dwopt launch.
  DwOptParams dp;
  fill_dwopt_params(c, u, &dp);
  dp.step = s;
  const bool sharded = c->cfg.world_size > 1;
  const bool px_on = sharded && c->peers_set && c->plan.peer_exchange;   // all-reduce fused into the dwopt launch
  const bool nccl = sharded && !px_on;
  if (px_on) dp.px = c->px;
  dp.opt.do_apply = nccl ? 0 : 1;
  auto launch_dwopt = [&]() -> int {
    PROF(dp.gemm_ctas ? PC_DW_GEMM : PC_OPT);
    const cudaError_t e = dwopt_launch(dp, c->sm_count, stream, pdl, c->plan.maxu);
    if (e != cudaSuccess) { set_error("dwopt launch failed: %s", cudaGetErrorString(e)); return MINPPO_ERR_CUDA; }
    c->launches++;
    return 0;
  };
  if (c->plan.two_launch) {
    GemmParams p = dp.gemm;                                  // this step's row list and row count go into the groups
    for (int i = 0; i < p.ngroups; ++i) {
      if (p.g[i].rowidx) p.g[i].rowidx = ridx;
      p.g[i].k_count = c->plan.padded ? c->counts + s : nullptr;
    }
    PROF(PC_DW_GEMM);
    RET(launch_gemm<EPI_PARTIAL>(p, c->plan.dw_gemm_ctas, stream, pdl));
    c->launches++;
  }
  RET(launch_dwopt());
  if (nccl) {
    { PROF(PC_ALLREDUCE); RET(nccl_allreduce(c, c->gflat, static_cast<size_t>(c->P) + LOSS_SUMS, stream)); }
    c->launches++;
    fill_apply_only(c, &dp);
    RET(launch_dwopt());
  }
  return 0;
}

static int enqueue_update(minppo_ctx* c, const UpdatePtrs& u, cudaStream_t stream) {
  const minppo_config& cfg = c->cfg;
  c->launches = 0;
  const float gamma = static_cast<float>(cfg.gamma);
  const float gl = static_cast<float>(cfg.gamma * cfg.gae_lambda);      // python-float product, then f32 (train.py:194)
  c->prof_used = 0;
  // Fork: the bf16 images of the observations and of the weights depend on nothing the GAE -> permutation -> row-list
  // chain produces (and vice versa) until the first minibatch step, so they run on a side branch (captured as a
  // parallel branch of the graph).  The permutation chain is 25+ tiny dependent launches, the observation image one
  // bandwidth-bound pass over the trajectory: side by side they cost the longer of the two.  Eager profiling runs keep
  // everything on one stream so that the per-class event times stay attributable.
  const bool fork = !c->profiling;
  if (fork) {
    CK(cudaEventRecord(c->ev_fork, stream));
    CK(cudaStreamWaitEvent(c->side_stream, c->ev_fork, 0));
    RET(obs_image_launch(u.obs, c->obs_img, c->Bl, c->D, c->Dp, c->side_stream));
    RET(enqueue_weight_images(c, u.params, c->side_stream));
    CK(cudaEventRecord(c->ev_join, c->side_stream));
    c->launches += 2;
  }
  {
    PROF(PC_GAE);
    RET(gae_launch(u.reward, u.value, u.done, u.last_val, c->adv, c->tgt, c->T, c->Nl, gamma, gl, c->sm_count, 0, stream));
    c->launches++;
  }
  if (cfg.world_size > 1) {
    // The permutations depend only on the key chain, so the ranks split the sorting work by epoch (rank e % W sorts
    // epoch e) and broadcast: every rank still ends up with the same GLOBAL permutations, bit for bit.
    PROF(PC_PERM);
    const int W = cfg.world_size, R = cfg.rank;
    const int mine = R < c->E ? (c->E - R + W - 1) / W : 0;
    RET(perm_launch(u.key_in, u.key_out, cfg.prng_mode, mine, c->B, c->perm_tmp, c->perm_ws, c->perm_ws_bytes, stream, R, W, c->E));
    NcclApi* api = nccl_api();
    ncclResult_t r = api->GroupStart();
    for (int e = 0; e < c->E && r == ncclSuccess; ++e) {
      const int root = e % W;
      int32_t* dst = c->perms + static_cast<size_t>(e) * c->B;
      const int32_t* src = root == R ? c->perm_tmp + static_cast<size_t>(e / W) * c->B : dst;
      r = api->Broadcast(src, dst, static_cast<size_t>(c->B), ncclInt32, root, c->comm, stream);
    }
    const ncclResult_t r2 = api->GroupEnd();
    if (r == ncclSuccess) r = r2;
    if (r != ncclSuccess) { set_error("ncclBroadcast (permutations) failed: %s", api->GetErrorString(r)); return MINPPO_ERR_NCCL; }
    c->launches += (mine > 0 ? perm_launch_count(c->B) : 0) + (u.key_out ? 1 : 0);
  } else {
    PROF(PC_PERM);
    RET(perm_launch(u.key_in, u.key_out, cfg.prng_mode, c->E, c->B, c->perms, c->perm_ws, c->perm_ws_bytes, stream));
    c->launches += perm_launch_count(c->B) + (u.key_out ? 1 : 0);
  }
  const int EM = c->E * c->M;
  {
    PROF(PC_PREP);
    RET(compact_rows_launch(c->perms, c->rowidx, c->counts, c->E, c->M, c->B, c->mb, c->plan.row_cap, c->N, c->n0, c->Nl, c->err_flag, stream));
    RET(adv_stats_launch(c->adv, c->rowidx, c->counts, c->stats, EM, c->plan.row_cap, c->mb, 0, stream));
    if (cfg.world_size > 1) RET(nccl_allreduce(c, c->stats, EM, stream));
    RET(adv_stats_launch(c->adv, c->rowidx, c->counts, c->stats, EM, c->plan.row_cap, c->mb, 1, stream));
    if (cfg.world_size > 1) RET(nccl_allreduce(c, c->stats + EM, EM, stream));
    c->launches += 3 + (cfg.world_size > 1 ? 2 : 0);
  }
  if (fork) {
    CK(cudaStreamWaitEvent(stream, c->ev_join, 0));              // join
  } else {
    {
      PROF(PC_OBS_IMAGE);
      RET(obs_image_launch(u.obs, c->obs_img, c->Bl, c->D, c->Dp, stream));
      c->launches++;
    }
    // the weight images must match the caller's params at entry (they may have been replaced)
    {
      PROF(PC_WEIGHT_IMAGES);
      RET(enqueue_weight_images(c, u.params, stream));
      c->launches++;
    }
  }
  for (int s = 0; s < EM; ++s) RET(enqueue_step(c, u, s, stream));
  return 0;
}

}  // namespace minppo

// ==========================================================================================
// C ABI
// ==========================================================================================
extern "C" {

const char* minppo_last_error(void) { return g_err; }
int minppo_version(void) { return 100; }

int minppo_gae_chunked(const float* reward, const float* value, const uint8_t* done, const float* last_val,
                       float* adv_out, float* tgt_out, int32_t T, int64_t N, double gamma, double gae_lambda,
                       int32_t chunks, void* stream) {
  if (!reward || !value || !done || !last_val || !adv_out || !tgt_out || T <= 0 || N <= 0) {
    set_error("minppo_gae: null pointer or non-positive size");
    return MINPPO_ERR_ARG;
  }
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  int r = gae_launch(reward, value, done, last_val, adv_out, tgt_out, T, N, static_cast<float>(gamma),
                     static_cast<float>(gamma * gae_lambda), sms, chunks, static_cast<cudaStream_t>(stream));
  if (r) { set_error("gae launch failed: %s", cudaGetErrorString(cudaGetLastError())); return MINPPO_ERR_CUDA; }
  return 0;
}
int minppo_gae(const float* reward, const float* value, const uint8_t* done, const float* last_val, float* adv_out,
               float* tgt_out, int32_t T, int64_t N, double gamma, double gae_lambda, void* stream) {
  return minppo_gae_chunked(reward, value, done, last_val, adv_out, tgt_out, T, N, gamma, gae_lambda, 0, stream);
}

size_t minppo_permutation_workspace_size(int32_t epochs, int64_t B) { return perm_workspace_bytes(epochs, B); }

int minppo_permutation(const uint32_t* key_in, uint32_t* key_out, int32_t prng_mode, int32_t epochs, int64_t B,
                       int32_t* perm_out, void* workspace, size_t workspace_bytes, void* stream) {
  if (!key_in || !perm_out || !workspace) { set_error("minppo_permutation: null pointer"); return MINPPO_ERR_ARG; }
  if (prng_mode != MINPPO_PRNG_LEGACY && prng_mode != MINPPO_PRNG_PARTITIONABLE) { set_error("bad prng_mode"); return MINPPO_ERR_ARG; }
  int r = perm_launch(key_in, key_out, prng_mode, epochs, B, perm_out, workspace, workspace_bytes,
                      static_cast<cudaStream_t>(stream));
  if (r == MINPPO_ERR_ARG) set_error("minppo_permutation: bad size");
  else if (r == MINPPO_ERR_WORKSPACE) set_error("minppo_permutation: workspace too small");
  else if (r) set_error("minppo_permutation: launch failed: %s", cudaGetErrorString(cudaGetLastError()));
  return r;
}

int64_t minppo_param_layout(const minppo_config* cfg, int32_t* nleaves, int64_t* offsets, int64_t* rows,
                            int64_t* cols) {
  if (!cfg) { set_error("null config"); return MINPPO_ERR_ARG; }
  std::vector<LeafInfo> lv;
  const long long P = build_layout(*cfg, &lv);
  if (nleaves) *nleaves = static_cast<int32_t>(lv.size());
  for (size_t i = 0; i < lv.size(); ++i) {
    if (offsets) offsets[i] = lv[i].offset;
    if (rows) rows[i] = lv[i].rows;
    if (cols) cols[i] = lv[i].cols;
  }
  return P;
}

int minppo_nccl_unique_id(void* id128_host) {
  NcclApi* api = nccl_api();
  if (!api) { set_error("libnccl.so.2 could not be loaded"); return MINPPO_ERR_NCCL; }
  ncclUniqueId id;
  ncclResult_t r = api->GetUniqueId(&id);
  if (r != ncclSuccess) { set_error("ncclGetUniqueId: %s", api->GetErrorString(r)); return MINPPO_ERR_NCCL; }
  static_assert(sizeof(ncclUniqueId) == 128, "ncclUniqueId is 128 bytes");
  memcpy(id128_host, &id, 128);
  return 0;
}

// Every choice of the kernel path (include/minppo_b200.h); minppo_ctx_create keeps the result as c->plan.
int minppo_plan(const minppo_config* cfg, int32_t sm_count, struct minppo_plan* out) {
  if (!cfg || !out || sm_count < 1) { set_error("minppo_plan: null argument or sm_count %d", sm_count); return MINPPO_ERR_ARG; }
  RET(validate_config(*cfg));
  const minppo_config& c = *cfg;
  const int L = c.num_layers, H = c.hidden_size, A = c.act_dim, Dp = (c.obs_dim + 63) / 64 * 64;
  const long long Bl = static_cast<long long>(c.num_steps) * (c.num_envs / c.world_size);   // this rank's transitions
  const int mb = static_cast<int>(static_cast<long long>(c.num_steps) * c.num_envs / c.num_minibatches);
  struct minppo_plan p = {};
  p.num_params = build_layout(c, nullptr);
  // row lists: the whole minibatch, or on env-sharded ranks 1.5 x the mean share + 256 rows
  p.padded = c.world_size > 1;
  int cap = mb;
  if (p.padded) cap = static_cast<int>(std::min<long long>({(3LL * mb / c.world_size + 1) / 2 + 256, mb, Bl}));
  // test hook (tests/test_gpu_update.py): an undersized row list, to exercise the overflow path on one GPU
  const int force_cap = getenv("MINPPO_FORCE_CAP") ? atoi(getenv("MINPPO_FORCE_CAP")) : 0;
  if (force_cap > 0) { p.padded = 1; cap = force_cap; }
  p.row_cap = (cap + 127) / 128 * 128;                 // row lists are padded to whole GEMM tiles
  // wider hidden layers or heads than the fused step kernel holds run layer-wise, whatever learner.fused says
  p.fused = !c.disable_fused && L == 2 && H <= GEMM_MAXN && A <= FS_MAX_AP;
  p.ap = A <= 16 ? 16 : 32;
  p.head_amax = head_amax(A);
  p.hsplit = H > GEMM_MAXN ? 2 : 1;
  const long long P = p.num_params;
  p.maxu = P <= dwopt_fast_capacity(sm_count, 1) ? 1 : (P <= dwopt_fast_capacity(sm_count, 2) ? 2 : 4);
  // split-K of the dW GEMMs: fill the SMs once
  // N-halved dW tiles (fused path, H a multiple of 128): half the split-K factor for the same number of GEMM CTAs
  // (only with TMA-fed A operands: groups that gather their rows by index would gather every row twice).
  // H > GEMM_MAXN needs the two column groups of col_group whatever the path; there the first layer's groups gather
  // their observation rows by index (A_GATHER_MN), so every row is gathered once per column group: twice the
  // observation-image reads of that layer's A operand.
  p.dw_nsplit = H > GEMM_MAXN ? 2 : (p.fused && H % 128 == 0 && 2 * 2 * L <= GEMM_MAX_GROUPS) ? 2 : 1;
  int per_split = 0;
  for (int l = 0; l < L; ++l) per_split += 2 * p.dw_nsplit * (((l == 0 ? Dp : H) + 127) / 128);
  // leave ~16 of the one-CTA-per-SM grid as spare CTAs: they sum the per-tile partials of the small leaves while the GEMM
  // runs (D = 415 / A = 20 with 4 spare CTAs: 6,441 elements x 64 partials on 2,048 threads outlasted the GEMM itself)
  const int gemm_budget = sm_count > 48 ? sm_count - 16 : sm_count;
  int S = c.dw_splits > 0 ? c.dw_splits : (gemm_budget / (per_split > 0 ? per_split : 1));
  // k-blocks (64 minibatch rows each) the splits share.  Padded row lists (env-sharded ranks): size the split for the
  // rows a minibatch is EXPECTED to have on this rank (mean + 3 sigma of the hypergeometric count), not for the
  // worst-case capacity -- the kernel splits the live k-blocks at run time, an over-sized S only removes spare CTAs.
  int kb_total = p.row_cap / 64;
  if (p.padded) {
    const double mean = static_cast<double>(mb) / c.world_size;
    const long long rows = static_cast<long long>(mean + 3.0 * sqrt(mean)) + 1;
    kb_total = std::max(1, static_cast<int>(std::min<long long>(p.row_cap, rows + 63) / 64));
  }
  S = std::max(1, std::min({S, kb_total, 32}));
  // no empty splits: ceil(kb_total / S) * (S - 1) < kb_total
  while (S > 1 && ((kb_total + S - 1) / S) * (S - 1) >= kb_total) --S;
  p.S = S;
  p.dw_gemm_ctas = per_split * S;
  // a GEMM grid past one CTA per SM runs as a launch of its own in front of dwopt
  p.two_launch = p.dw_gemm_ctas > sm_count;
  // dwopt_kernel decides its register-resident path on the device from the leaf table, `n_units <= G * NT * MAXU`
  // (dwopt.cuh), n_units = the 4-element units of the late leaves that fill_opt_args marks: the hidden kernels and, on
  // the layer-wise path, the hidden biases whose column sums the dW GEMM computes.  The same condition on the host:
  long long late_units = 0;                            // both nets: hidden kernel (+ bias)
  for (int l = 0; l < L; ++l) late_units += 2 * ((l == 0 ? c.obs_dim : H) * (H / 4LL) + (p.fused ? 0 : H / 4));
  p.dwopt_fast = 4 * late_units <= dwopt_fast_capacity(sm_count, p.maxu);
  // the all-reduce fused into the dwopt launch needs the kernel's register-resident path and the GEMM in the same launch
  p.peer_exchange = P <= dwopt_fast_capacity(sm_count, p.maxu) && !p.two_launch;
  *out = p;
  return 0;
}

static void drop_graphs(minppo_ctx* c) {
  for (auto& g : c->graphs) { cudaGraphExecDestroy(g.exec); cudaGraphDestroy(g.graph); }
  c->graphs.clear();
}

int minppo_ctx_destroy(minppo_ctx* c) {
  if (!c) return 0;
  drop_graphs(c);
  for (cudaEvent_t e : c->prof_events) cudaEventDestroy(e);
  if (c->cap_stream) cudaStreamDestroy(c->cap_stream);
  if (c->side_stream) cudaStreamDestroy(c->side_stream);
  if (c->ev_fork) cudaEventDestroy(c->ev_fork);
  if (c->ev_join) cudaEventDestroy(c->ev_join);
  if (c->have_comm) nccl_api()->CommDestroy(c->comm);
  for (int r = 0; r < MINPPO_MAX_RANKS; ++r) if (c->peer_ptr[r]) cudaIpcCloseMemHandle(c->peer_ptr[r]);
  for (void* p : c->allocs) cudaFree(p);
  delete c;
  return 0;
}

int minppo_ctx_create(const minppo_config* cfg, const void* nccl_unique_id_host, minppo_ctx** out) {
  if (!cfg || !out) { set_error("null argument"); return MINPPO_ERR_ARG; }
  RET(validate_config(*cfg));
  minppo_ctx* c = new minppo_ctx();
  c->cfg = *cfg;
  c->have_comm = false; c->cap_stream = nullptr; c->launches = 0;
  c->side_stream = nullptr; c->ev_fork = nullptr; c->ev_join = nullptr;
  c->profiling = false; c->prof_used = 0;
  int rc = 0;
  auto fail = [&](int code) { minppo_ctx_destroy(c); return code; };
  if (cudaGetDevice(&c->device) != cudaSuccess) { set_error("no CUDA device"); return fail(MINPPO_ERR_CUDA); }
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, c->device) != cudaSuccess) { set_error("cudaGetDeviceProperties failed"); return fail(MINPPO_ERR_CUDA); }
  if (prop.major != 10) {
    set_error("minppo_b200 requires an sm_100a (B200) device; found sm_%d%d", prop.major, prop.minor);
    return fail(MINPPO_ERR_UNSUPPORTED);
  }
  c->sm_count = prop.multiProcessorCount;
  if ((rc = init_kernel_attrs())) return fail(rc);

  c->T = cfg->num_steps; c->N = cfg->num_envs; c->Nl = c->N / cfg->world_size; c->n0 = cfg->rank * c->Nl;
  c->M = cfg->num_minibatches; c->E = cfg->update_epochs; c->L = cfg->num_layers; c->H = cfg->hidden_size;
  c->D = cfg->obs_dim; c->Dp = (c->D + 63) / 64 * 64; c->A = cfg->act_dim;
  c->B = static_cast<long long>(c->T) * c->N; c->Bl = static_cast<long long>(c->T) * c->Nl;
  c->mb = static_cast<int>(c->B / c->M);
  if ((rc = minppo_plan(cfg, c->sm_count, &c->plan))) return fail(rc);
  c->m_tiles = c->plan.row_cap / 128;
  c->tiles64 = c->plan.row_cap / 64;
  c->P = build_layout(*cfg, &c->leaves);
  c->head.w3a = static_cast<int>(find_leaf(c, 0, c->L, 1).offset);
  c->head.b3a = static_cast<int>(find_leaf(c, 0, c->L, 0).offset);
  c->head.w3c = static_cast<int>(find_leaf(c, 1, c->L, 1).offset);
  c->head.b3c = static_cast<int>(find_leaf(c, 1, c->L, 0).offset);
  c->head.logstd = static_cast<int>(c->leaves.back().offset);
  const int H = c->H, L = c->L, A = c->A;
  // head partial layout
  {
    int o = 0;                                       // (the head-kernel gradients start 16-byte aligned: the fused step writes
    c->po_w3a = o; o += H * A;                       //  each of them with one bulk copy)
    c->po_b3a = o; o += A;
    o = (o + 3) / 4 * 4;
    c->po_w3c = o; o += H;
    c->po_b3c = o; o += 1;
    c->po_logstd = o; o += A;
    for (int net = 0; net < 2; ++net)
      for (int l = 0; l < 2; ++l) { c->po_db[net][l] = o; o += H; }
    c->po_loss = o; o += LOSS_SUMS;
    c->head_stride = (o + 3) / 4 * 4;
  }
  const int EM = c->E * c->M;
#define ALLOC(ptr, n) if ((rc = dev_alloc(c, &(ptr), (n)))) return fail(rc)
  ALLOC(c->adv, static_cast<size_t>(c->Bl));
  ALLOC(c->tgt, static_cast<size_t>(c->Bl));
  ALLOC(c->stats, static_cast<size_t>(2 * EM));
  c->xchg = nullptr; c->peers_set = false; memset(&c->px, 0, sizeof(c->px)); memset(c->peer_ptr, 0, sizeof(c->peer_ptr));
  if (cfg->world_size > 1) {
    // the local gradient buffer lives inside the exchange allocation so that peers can read it (own cudaMalloc:
    // CUDA IPC exports whole allocations)
    const int np = static_cast<int>((c->P + LOSS_SUMS + 3) / 4 * 4);
    const size_t floats = 2 * static_cast<size_t>(cfg->world_size) * np + static_cast<size_t>(cfg->world_size) * 256 + 2 * static_cast<size_t>(np);
    ALLOC(c->xchg, floats);
    // staging / result words start as the "not yet written" sentinel -0.0f of the Lamport-style exchange (dwopt.cuh)
    fill_u32_kernel<<<296, 256>>>(reinterpret_cast<uint32_t*>(c->xchg), floats, 0x80000000u);
    ALLOC(c->xseq, 1);
    c->px.np = np; c->px.world = 0; c->px.rank = cfg->rank; c->px.seq = c->xseq;
  }
  ALLOC(c->gflat, static_cast<size_t>(c->P) + 8);
  ALLOC(c->block_ss, static_cast<size_t>(c->sm_count));
  ALLOC(c->head_part, static_cast<size_t>(c->tiles64) * c->head_stride);
  ALLOC(c->gnorms, static_cast<size_t>(EM));
  ALLOC(c->losses_scratch, 4);
  ALLOC(c->trace, static_cast<size_t>(2 * c->m_tiles) * FS_TRACE_SLOTS);
  ALLOC(c->trace2, static_cast<size_t>(c->sm_count) * 16);
  c->trace_on = getenv("MINPPO_TRACE") != nullptr;
  ALLOC(c->perms, static_cast<size_t>(c->E) * c->B);
  c->perm_tmp = nullptr;
  if (cfg->world_size > 1) ALLOC(c->perm_tmp, static_cast<size_t>((c->E + cfg->world_size - 1) / cfg->world_size) * c->B);
  ALLOC(c->rowidx, static_cast<size_t>(EM) * c->plan.row_cap);
  ALLOC(c->counts, static_cast<size_t>(EM));
  c->perm_ws_bytes = perm_workspace_bytes(c->E, c->B);
  { uint8_t* p; ALLOC(p, c->perm_ws_bytes); c->perm_ws = p; }
  ALLOC(c->obs_img, static_cast<size_t>(c->Bl) * c->Dp + 256);   // slack: MN gather may read one chunk past Dp
  ALLOC(c->xg, static_cast<size_t>(c->plan.row_cap) * c->Dp);
  if ((rc = make_tmap(&c->m_xg_k, c->xg, c->Dp, c->plan.row_cap, c->Dp, 64, 128))) return fail(rc);
  if ((rc = make_tmap(&c->m_xg_mn, c->xg, c->Dp, c->plan.row_cap, c->Dp, 64, 64))) return fail(rc);
  ALLOC(c->barrier, 1);
  ALLOC(c->dw_done, static_cast<size_t>(c->sm_count + 2) * DWOPT_DONE_STRIDE);   // zeroed: dwopt_kernel expects 0 at launch
  ALLOC(c->err_flag, 1);
  for (int net = 0; net < 2; ++net) {
    NetBufs& nb = c->net[net];
    nb.act.assign(L + 1, nullptr); nb.dz.assign(L + 1, nullptr); nb.wn.assign(L, nullptr);
    nb.dw_part.assign(L, nullptr); nb.dbias.assign(L, nullptr);
    ALLOC(nb.w2img, static_cast<size_t>(H) * FS_MAX_AP * 4);       // H/64 panels of [2 AP rows][128 B]
    nb.m_act_k.resize(L + 1); nb.m_act_mn.resize(L + 1); nb.m_dz_k.resize(L + 1); nb.m_dz_mn.resize(L + 1);
    nb.m_wn_mn.resize(L); nb.m_wn.resize(2 * L); nb.m_dw.resize(L); nb.m_wn_h.resize(L);
    for (int l = 1; l <= L; ++l) {
      ALLOC(nb.act[l], static_cast<size_t>(c->plan.row_cap) * H);
      ALLOC(nb.dz[l], static_cast<size_t>(c->plan.row_cap) * H);
      if ((rc = make_tmap(&nb.m_act_k[l], nb.act[l], H, c->plan.row_cap, H, 64, 128))) return fail(rc);
      if ((rc = make_tmap(&nb.m_act_mn[l], nb.act[l], H, c->plan.row_cap, H, 64, 64))) return fail(rc);
      if ((rc = make_tmap(&nb.m_dz_k[l], nb.dz[l], H, c->plan.row_cap, H, 64, 128))) return fail(rc);
      if ((rc = make_tmap(&nb.m_dz_mn[l], nb.dz[l], H, c->plan.row_cap, H, 64, 64))) return fail(rc);
    }
    for (int l = 0; l < L; ++l) {
      const int kp = l == 0 ? c->Dp : H;
      const int in_l = l == 0 ? c->D : H;
      ALLOC(nb.wn[l], static_cast<size_t>(kp) * H);
      if ((rc = make_tmap(&nb.m_wn_mn[l], nb.wn[l], H, kp, H, 64, 64))) return fail(rc);
      if ((rc = make_tmap(&nb.m_wn_h[l], nb.wn[l], H, kp, H, 64, 32))) return fail(rc);
      if (l == 1 && (rc = make_tmap(&nb.m_w1k_h, nb.wn[l], H, H, H, 64, H / 2))) return fail(rc);
      if (l >= 1) {
        for (int j = 0; j < c->plan.hsplit; ++j) {
          int n_off, n;
          col_group(H, c->plan.hsplit, j, &n_off, &n);
          if ((rc = make_tmap(&nb.m_wn[2 * l + j], nb.wn[l], H, H, H, 64, n))) return fail(rc);
        }
      }
      ALLOC(nb.dw_part[l], static_cast<size_t>(c->plan.S) * in_l * H);
      ALLOC(nb.dbias[l], static_cast<size_t>(c->plan.S) * H);
      if ((rc = make_tmap_f32_3d(&nb.m_dw[l], nb.dw_part[l], H, in_l, c->plan.S))) return fail(rc);
    }
  }
  c->pol_tiles = (c->Nl + 127) / 128;
  {
    const size_t prow = static_cast<size_t>(c->pol_tiles) * 128;
    ALLOC(c->pol_img, prow * c->Dp);
    if ((rc = make_tmap(&c->m_pol_img_k, c->pol_img, c->Dp, prow, c->Dp, 64, 128))) return fail(rc);
    for (int net = 0; net < 2; ++net)
      for (int l = 1; l <= L; ++l) {
        ALLOC(c->pol_act[net][l], prow * H);
        if ((rc = make_tmap(&c->m_pol_act_k[net][l], c->pol_act[net][l], H, prow, H, 64, 128))) return fail(rc);
      }
  }
#undef ALLOC
  if (cfg->world_size > 1) {
    NcclApi* api = nccl_api();
    if (!api) { set_error("libnccl.so.2 could not be loaded"); return fail(MINPPO_ERR_NCCL); }
    if (!nccl_unique_id_host) { set_error("world_size > 1 requires a NCCL unique id"); return fail(MINPPO_ERR_ARG); }
    ncclUniqueId id;
    memcpy(&id, nccl_unique_id_host, 128);
    ncclResult_t r = api->CommInitRank(&c->comm, cfg->world_size, id, cfg->rank);
    if (r != ncclSuccess) { set_error("ncclCommInitRank: %s", api->GetErrorString(r)); return fail(MINPPO_ERR_NCCL); }
    c->have_comm = true;
  }
  if (cudaStreamCreateWithFlags(&c->side_stream, cudaStreamNonBlocking) != cudaSuccess ||
      cudaEventCreateWithFlags(&c->ev_fork, cudaEventDisableTiming) != cudaSuccess ||
      cudaEventCreateWithFlags(&c->ev_join, cudaEventDisableTiming) != cudaSuccess) {
    set_error("side stream / event creation failed");
    return fail(MINPPO_ERR_CUDA);
  }
  if (cudaStreamCreateWithFlags(&c->cap_stream, cudaStreamNonBlocking) != cudaSuccess) {
    set_error("cudaStreamCreate failed");
    return fail(MINPPO_ERR_CUDA);
  }
  if (cudaDeviceSynchronize() != cudaSuccess) { set_error("context initialisation failed: %s", cudaGetErrorString(cudaGetLastError())); return fail(MINPPO_ERR_CUDA); }
  *out = c;
  return 0;
}

int minppo_update_with_stats(minppo_ctx* c, float* params, float* mu, float* nu, int32_t* count, const float* obs,
                             const float* action, const float* value, const float* reward, const float* log_prob,
                             const uint8_t* done, const float* last_val, const uint32_t* key_in, uint32_t* key_out,
                             float* losses_out, float* stats_out, int32_t use_graph, void* stream_v) {
  if (!c || !params || !mu || !nu || !count || !obs || !action || !value || !reward || !log_prob || !done ||
      !last_val || !key_in) {
    set_error("minppo_update: null pointer");
    return MINPPO_ERR_ARG;
  }
  cudaStream_t stream = static_cast<cudaStream_t>(stream_v);
  UpdatePtrs u;
  memset(&u, 0, sizeof(u));
  u.params = params; u.mu = mu; u.nu = nu; u.count = count; u.obs = obs; u.action = action; u.value = value;
  u.reward = reward; u.log_prob = log_prob; u.done = done; u.last_val = last_val; u.key_in = key_in;
  u.key_out = key_out; u.losses_out = losses_out; u.stats_out = stats_out;
  if (!use_graph) return enqueue_update(c, u, stream);
  const bool was_profiling = c->profiling;
  c->profiling = false;                         // event records are not captured; profile in eager mode
  struct Restore { minppo_ctx* c; bool v; ~Restore() { c->profiling = v; } } restore{c, was_profiling};
  size_t hit = c->graphs.size();
  for (size_t i = 0; i < c->graphs.size(); ++i)
    if (c->graphs[i].ptrs == u) { hit = i; break; }
  if (hit == c->graphs.size()) {
    constexpr size_t kMaxGraphs = 4;
    if (c->graphs.size() >= kMaxGraphs) {
      // evict the least recently used set; the exec may still be running on the caller's stream: CUDA defers the release
      // of an executable graph's resources until its in-flight launches have completed
      cudaGraphExecDestroy(c->graphs.front().exec); cudaGraphDestroy(c->graphs.front().graph);
      c->graphs.erase(c->graphs.begin());
    }
    CK(cudaStreamBeginCapture(c->cap_stream, cudaStreamCaptureModeThreadLocal));
    int r = enqueue_update(c, u, c->cap_stream);
    cudaGraph_t g = nullptr;
    cudaError_t e = cudaStreamEndCapture(c->cap_stream, &g);
    if (r != 0) { if (g) cudaGraphDestroy(g); return r; }
    if (e != cudaSuccess) { set_error("graph capture failed: %s", cudaGetErrorString(e)); return MINPPO_ERR_CUDA; }
    cudaGraphExec_t ge = nullptr;
    if (cudaGraphInstantiate(&ge, g, 0) != cudaSuccess) { cudaGraphDestroy(g); set_error("cudaGraphInstantiate failed: %s", cudaGetErrorString(cudaGetLastError())); return MINPPO_ERR_CUDA; }
    c->graphs.push_back({g, ge, u, c->launches});
  } else if (hit + 1 != c->graphs.size()) {
    const minppo_ctx::CachedGraph cg = c->graphs[hit];         // most recently used goes last
    c->graphs.erase(c->graphs.begin() + hit);
    c->graphs.push_back(cg);
  }
  c->launches = c->graphs.back().launches;
  CK(cudaGraphLaunch(c->graphs.back().exec, stream));
  return 0;
}

int minppo_update(minppo_ctx* c, float* params, float* mu, float* nu, int32_t* count, const float* obs,
                  const float* action, const float* value, const float* reward, const float* log_prob,
                  const uint8_t* done, const float* last_val, const uint32_t* key_in, uint32_t* key_out,
                  float* losses_out, int32_t use_graph, void* stream_v) {
  return minppo_update_with_stats(c, params, mu, nu, count, obs, action, value, reward, log_prob, done, last_val, key_in,
                                  key_out, losses_out, nullptr, use_graph, stream_v);
}

int minppo_policy_step(minppo_ctx* c, const float* params, const float* obs, const uint32_t* key_in, uint32_t* key_out,
                       float* action, float* log_prob, float* value, float* mean, int32_t flags, void* stream_v) {
  if (!c || !params || !obs) { set_error("minppo_policy_step: null pointer"); return MINPPO_ERR_ARG; }
  if (key_in && key_out == key_in) { set_error("minppo_policy_step: key_out must not alias key_in"); return MINPPO_ERR_ARG; }
  const bool actor = action || log_prob || mean;
  if (!actor && !value) { set_error("minppo_policy_step: no output requested"); return MINPPO_ERR_ARG; }
  cudaStream_t stream = static_cast<cudaStream_t>(stream_v);
  const int L = c->L, H = c->H;
  if (!(flags & MINPPO_POLICY_WEIGHTS_CURRENT)) RET(enqueue_weight_images(c, params, stream));
  if (c->plan.fused) {
    // 2-hidden-layer nets: ONE launch (policy_fused.cuh) -- observation conversion, both hidden layers, heads, sampler
    PolicyParams pp;
    memset(&pp, 0, sizeof(pp));
    for (int net = 0; net < 2; ++net) {
      PolicyNet& g = pp.net[net];
      NetBufs& nb = c->net[net];
      g.tm_w0 = nb.m_wn_h[0]; g.tm_w1 = nb.m_wn_h[1];
      g.b0 = params + find_leaf(c, net, 0, 0).offset;
      g.b1 = params + find_leaf(c, net, 1, 0).offset;
      g.w2img = reinterpret_cast<const uint4*>(nb.w2img);
      g.b2 = params + (net == 0 ? c->head.b3a : c->head.b3c);
      g.act = act_kind(c, net);
      g.aout = net == 0 ? c->A : 1;
    }
    pp.obs = obs; pp.log_std = params + c->head.logstd;
    pp.key_in = actor ? key_in : nullptr; pp.key_out = actor ? key_out : nullptr;
    pp.action = action; pp.log_prob = log_prob; pp.value = value; pp.mean_out = mean;
    pp.n0 = c->n0; pp.n_total = static_cast<long long>(c->N) * c->A;
    pp.rows = c->Nl; pp.D = c->D; pp.Dp = c->Dp; pp.H = H; pp.A = c->A; pp.mode = c->cfg.prng_mode;
    pp.net_first = actor ? 0 : 1;
    const cudaError_t e = policy_fused_launch(pp, c->pol_tiles, stream, c->plan.ap);
    if (e != cudaSuccess) { set_error("policy_fused launch failed: %s", cudaGetErrorString(e)); return MINPPO_ERR_CUDA; }
    return 0;
  }
  // bf16 image of last_obs, zero padded to Dp columns (rows >= Nl of the image stay zero from allocation)
  RET(obs_image_launch(obs, c->pol_img, c->Nl, c->D, c->Dp, stream));
  const int first = actor ? 0 : 1;                        // critic only: the bootstrap value (train.py:182-183)
  for (int l = 0; l < L; ++l) {
    FwdOperands op[2];
    for (int net = 0; net < 2; ++net)
      op[net] = {nullptr, l == 0 ? &c->m_pol_img_k : &c->m_pol_act_k[net][l], c->pol_act[net][l + 1]};
    GemmParams p;
    fill_forward_gemm(c, l, params, first, c->pol_tiles, op, &p);
    RET(launch_gemm<EPI_ACT>(p, p.ngroups * c->pol_tiles, stream));
  }
  PolicyHeadArgs a;
  memset(&a, 0, sizeof(a));
  a.h_a = actor ? c->pol_act[0][L] : nullptr;
  a.h_c = c->pol_act[1][L];
  a.params = params;
  a.off = c->head;
  a.H = H; a.A = c->A; a.ldh = H; a.rows = c->Nl;
  a.n0 = c->n0; a.n_total = static_cast<long long>(c->N) * c->A;
  a.key_in = actor ? key_in : nullptr; a.key_out = actor ? key_out : nullptr; a.mode = c->cfg.prng_mode;
  a.action = action; a.log_prob = log_prob; a.value = value; a.mean_out = mean;
  return policy_head_launch(a, stream);
}

int minppo_ctx_ipc_handle(minppo_ctx* c, void* handle64_host) {
  if (!c || !handle64_host) { set_error("null argument"); return MINPPO_ERR_ARG; }
  if (!c->xchg) { set_error("minppo_ctx_ipc_handle: context has world_size == 1"); return MINPPO_ERR_ARG; }
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "cudaIpcMemHandle_t is 64 bytes");
  cudaIpcMemHandle_t h;
  CK(cudaIpcGetMemHandle(&h, c->xchg));
  memcpy(handle64_host, &h, 64);
  return 0;
}

int minppo_ctx_set_peers(minppo_ctx* c, const void* handles_host) {
  if (!c || !handles_host) { set_error("null argument"); return MINPPO_ERR_ARG; }
  if (!c->xchg) { set_error("minppo_ctx_set_peers: context has world_size == 1"); return MINPPO_ERR_ARG; }
  const int W = c->cfg.world_size;
  if (W > MINPPO_MAX_RANKS) { set_error("peer exchange supports up to %d ranks", MINPPO_MAX_RANKS); return MINPPO_ERR_UNSUPPORTED; }
  for (int r = 0; r < W; ++r) {
    if (r == c->cfg.rank) { c->px.base[r] = reinterpret_cast<char*>(c->xchg); continue; }
    cudaIpcMemHandle_t h;
    memcpy(&h, static_cast<const char*>(handles_host) + 64 * r, 64);
    void* ptr = nullptr;
    CK(cudaIpcOpenMemHandle(&ptr, h, cudaIpcMemLazyEnablePeerAccess));
    c->peer_ptr[r] = ptr;
    c->px.base[r] = static_cast<char*>(ptr);
  }
  c->px.world = W;
  // one-shot push for small worlds (one NVLink latency), reduce-at-owner + result push for W >= 4 (2 (W-1)/W of a
  // gradient per rank on the links instead of W - 1 gradients); MINPPO_PX_TWO_PHASE=0/1 forces either
  c->px.two_phase = getenv("MINPPO_PX_TWO_PHASE") ? (atoi(getenv("MINPPO_PX_TWO_PHASE")) != 0) : (W >= 4);
  c->peers_set = true;
  drop_graphs(c);
  return 0;
}

int minppo_ctx_check(minppo_ctx* c, void* stream_v) {
  if (!c) return MINPPO_ERR_ARG;
  cudaStream_t stream = static_cast<cudaStream_t>(stream_v);
  CK(cudaStreamSynchronize(stream));
  int flag = 0;
  CK(cudaMemcpy(&flag, c->err_flag, sizeof(int), cudaMemcpyDeviceToHost));
  if (flag) { set_error("device-side error flag %d", flag); return flag; }
  const int EM = c->E * c->M;
  std::vector<int32_t> counts(EM);
  CK(cudaMemcpy(counts.data(), c->counts, EM * sizeof(int32_t), cudaMemcpyDeviceToHost));
  for (int s = 0; s < EM; ++s)
    if (counts[s] > c->plan.row_cap) { set_error("minibatch %d: %d local rows exceed capacity %d", s, counts[s], c->plan.row_cap); return MINPPO_ERR_WORKSPACE; }
  std::vector<float> gn(EM);
  CK(cudaMemcpy(gn.data(), c->gnorms, EM * sizeof(float), cudaMemcpyDeviceToHost));
  for (int s = 0; s < EM; ++s)
    if (!isfinite(gn[s])) { set_error("non-finite gradient norm at minibatch step %d", s); return MINPPO_ERR_NONFINITE; }
  return 0;
}

int64_t minppo_update_launch_count(const minppo_ctx* c) { return c ? c->launches : 0; }

int minppo_ctx_profile(minppo_ctx* c, int32_t enable) {
  if (!c) return MINPPO_ERR_ARG;
  c->profiling = enable != 0;
  c->prof_used = 0;
  return 0;
}

int minppo_ctx_profile_read(minppo_ctx* c, float* ms_per_class_host, int32_t* launches_per_class_host, int32_t nclasses) {
  if (!c || !ms_per_class_host || !launches_per_class_host) { set_error("null argument"); return MINPPO_ERR_ARG; }
  CK(cudaDeviceSynchronize());
  for (int i = 0; i < nclasses; ++i) { ms_per_class_host[i] = 0.f; launches_per_class_host[i] = 0; }
  for (size_t i = 0; i + 1 < c->prof_used; i += 2) {
    float ms = 0.f;
    CK(cudaEventElapsedTime(&ms, c->prof_events[i], c->prof_events[i + 1]));
    const int cls = c->prof_class[i / 2];
    if (cls < nclasses) { ms_per_class_host[cls] += ms; launches_per_class_host[cls] += 1; }
  }
  return 0;
}

int minppo_ctx_read(minppo_ctx* c, int32_t what, void* dst, size_t bytes, void* stream_v) {
  if (!c || !dst) { set_error("null argument"); return MINPPO_ERR_ARG; }
  const void* src = nullptr;
  size_t have = 0;
  const size_t EM = static_cast<size_t>(c->E) * c->M;
  switch (what) {
    case 0: src = c->adv; have = c->Bl * 4; break;
    case 1: src = c->tgt; have = c->Bl * 4; break;
    case 2: src = c->perms; have = static_cast<size_t>(c->E) * c->B * 4; break;
    case 3: src = c->gflat; have = (c->P + 4) * 4; break;
    case 4: src = c->gnorms; have = EM * 4; break;
    case 5: src = c->counts; have = EM * 4; break;
    case 6: src = c->stats; have = 2 * EM * 4; break;
    case 7: src = c->trace; have = static_cast<size_t>(2 * c->m_tiles) * FS_TRACE_SLOTS * 8; break;
    case 8: src = c->trace2; have = static_cast<size_t>(c->sm_count) * 16 * 8; break;
    default: set_error("minppo_ctx_read: unknown buffer %d", what); return MINPPO_ERR_ARG;
  }
  if (bytes > have) { set_error("minppo_ctx_read: %zu bytes requested, buffer has %zu", bytes, have); return MINPPO_ERR_ARG; }
  CK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToDevice, static_cast<cudaStream_t>(stream_v)));
  return 0;
}

int minppo_debug_gemm(int32_t mode, const void* a_bf16, const void* b_bf16, const int32_t* rowidx, float* cmat,
                      int32_t M, int32_t N, int32_t K, int32_t lda, int32_t splits, void* stream_v) {
  if (!a_bf16 || !b_bf16 || !cmat || M % 128 || K % 64 || N % 64 || N > 256 || N <= 0 || splits < 1 || mode < 0 ||
      mode > 3 || ((mode >= 2) && !rowidx)) {
    set_error("minppo_debug_gemm: bad argument");
    return MINPPO_ERR_ARG;
  }
  RET(init_kernel_attrs());
  GemmParams p;
  memset(&p, 0, sizeof(p));
  p.ngroups = 1;
  GemmGroup& g = p.g[0];
  g.cta_begin = 0; g.N = N; g.m_tiles = M / 128; g.splits = splits; g.kb_total = K / 64; g.m_store = M;
  RET(make_tmap_f32_3d(&g.tmC, cmat, N, M, splits));
  switch (mode) {
    case 0:
      g.amode = A_TMA_K; g.bmode = B_TMA_K;
      RET(make_tmap(&g.tmA, a_bf16, K, M, lda ? lda : K, 64, 128));
      RET(make_tmap(&g.tmB, b_bf16, K, N, K, 64, N));
      break;
    case 1:
      g.amode = A_TMA_MN; g.bmode = B_TMA_MN;
      RET(make_tmap(&g.tmA, a_bf16, M, K, lda ? lda : M, 64, 64));
      RET(make_tmap(&g.tmB, b_bf16, N, K, N, 64, 64));
      break;
    case 2:
      g.amode = A_GATHER_K; g.bmode = B_TMA_K; g.rowidx = rowidx;
      g.gimage = reinterpret_cast<const __nv_bfloat16*>(a_bf16); g.ldg = lda;
      RET(make_tmap(&g.tmB, b_bf16, K, N, K, 64, N));
      break;
    case 3:
      g.amode = A_GATHER_MN; g.bmode = B_TMA_MN; g.rowidx = rowidx;
      g.gimage = reinterpret_cast<const __nv_bfloat16*>(a_bf16); g.ldg = lda;
      RET(make_tmap(&g.tmB, b_bf16, N, K, N, 64, 64));
      break;
  }
  return launch_gemm<EPI_PARTIAL>(p, g.m_tiles * splits, static_cast<cudaStream_t>(stream_v));
}

}  // extern "C"
