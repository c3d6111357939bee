// minppo_b200 -- grouped BF16 GEMM on tcgen05 tensor cores (sm_100a) with fused epilogues.
//
// One CTA computes one 128 x N (N <= 256) fp32 accumulator tile in TMEM over a K range:
//   warp 0      : TMA producer (cp.async.bulk.tensor, SWIZZLE_128B boxes) for A and/or B
//   warp 1      : TMEM allocator + single-thread tcgen05.mma issuer
//   warps 2..5  : optional row-gather producer for A (cp.async by index, software swizzle),
//                 then the epilogue (tcgen05.ld -> registers -> fused math -> global)
// Operands are staged in a 4-deep shared-memory ring (mbarrier full/empty pairs).
// A layer wider than 256 columns runs as several groups of one launch, each on its own column range (GemmGroup::n_off,
// widths multiples of 64 and <= 256); B_TMA_K groups then carry a tensor map whose box is their own width.
//
// Operand modes (what the learner's layers need, /root/reference/minppo/train.py:56-83, 246):
//   A_TMA_K     A[m][k] row-major in HBM (activations)            -> K-major tile
//   A_GATHER_K  A[m][k] = image[rowidx[m]][k]  (minibatch gather, train.py:261, done on the fly)
//   A_TMA_MN    A[m][k] = act[k][m]  (dW = act^T * dZ; act stored [rows][features])
//   A_GATHER_MN A[m][k] = image[rowidx[k]][m]  (dW of the first layer)
//   B_TMA_K     B[n][k] row-major (weight images, dZ)             -> K-major tile
//   B_TMA_MN    B[n][k] = dz[k][n]
#pragma once

#include "common.cuh"

namespace minppo {

constexpr int GEMM_BM = 128;
constexpr int GEMM_BK = 64;
constexpr int GEMM_MAXN = 256;
constexpr int GEMM_STAGES = 4;
constexpr int GEMM_A_BYTES = GEMM_BM * GEMM_BK * 2;      // 16 KB
constexpr int GEMM_B_BYTES = GEMM_MAXN * GEMM_BK * 2;    // 32 KB
constexpr int GEMM_STAGE_BYTES = GEMM_A_BYTES + GEMM_B_BYTES;
constexpr int GEMM_THREADS = 192;
constexpr int GEMM_EPI_THREADS = 128;
constexpr int GEMM_ONES_BYTES = 16384;                   // all-ones bf16 [128][64] tile: A operand of the bias-gradient MMAs
constexpr int GEMM_SMEM_BYTES = GEMM_STAGES * GEMM_STAGE_BYTES + GEMM_ONES_BYTES + 1024 /*align*/ + 4 * GEMM_MAXN * 4 /*colsum*/ + 256;
constexpr int GEMM_MAX_GROUPS = 8;

enum : int { A_TMA_K = 0, A_GATHER_K = 1, A_TMA_MN = 2, A_GATHER_MN = 3 };
enum : int { B_TMA_K = 0, B_TMA_MN = 2 };
enum : int { EPI_ACT = 0, EPI_DACT = 1, EPI_PARTIAL = 2 };
enum : int { ACT_TANH = 0, ACT_RELU = 1, ACT_TANH_FAST = 2 };

struct alignas(64) GemmGroup {
  CUtensorMap tmA;                 // A_TMA_*
  CUtensorMap tmB;                 // B_TMA_*
  CUtensorMap tmC;                 // EPI_PARTIAL: fp32 [splits][m_store][N] store map, box {32, 128, 1}
  const int32_t* rowidx;           // A_GATHER_*: flat row index per minibatch row (all entries valid)
  const __nv_bfloat16* gimage;     // A_GATHER_*: bf16 image [rows][ldg]
  void* out;                       // EPI_ACT/EPI_DACT: bf16 [M][ldo]
  const float* bias;               // EPI_ACT: fp32 [N]
  const __nv_bfloat16* hprev;      // EPI_DACT: layer output h (for f'(z) from h), bf16 [M][ldh]
  float* colsum;                   // EPI_DACT: fp32 [m_tiles][ldc] per-tile column sums (bias grads)
  float* colsum_out;               // EPI_PARTIAL + B_TMA_MN: fp32 [splits][ldc] column sums of B over this CTA's K range
                                   // (= bias gradient partials), computed on the tensor core as ones x B; or null
  int ldg, ldo, ldh;
  int amode, bmode;                // A_* / B_* operand modes
  int cta_begin;                   // first blockIdx.x of this group
  int act;                         // ACT_*
  int N;                           // accumulator width (multiple of 16, <= 256)
  int m_tiles;                     // 128-row tiles
  int splits;                      // split-K factor (EPI_PARTIAL)
  int kb_total;                    // number of 64-wide k-blocks over the whole K
  int m_store;                     // EPI_PARTIAL: rows m < m_store are stored
  int n_off;                       // first column of this group's N range inside B, C, bias, out, hprev and the column sums
                                   // (N-split groups: a layer wider than GEMM_MAXN runs as several groups of <= 256 columns)
  int ldc;                         // row stride of colsum / colsum_out in floats (the full width of an N-split layer); 0 = N
  const int32_t* k_count;          // optional: number of valid K rows (device side); k-blocks beyond it are skipped
};

// 512 bytes: GEMM_MAX_GROUPS of them sit in every GEMM / dwopt parameter block
static_assert(sizeof(GemmGroup) == 512, "GemmGroup grew: the kernel parameter blocks grow with it");

struct alignas(64) GemmParams {
  int ngroups;                     // groups occupy consecutive blockIdx.x ranges starting at cta_begin
  int grp_begin[GEMM_MAX_GROUPS];  // copy of g[i].cta_begin, unused entries INT_MAX (gemm_finalize): one constant-bank line
                                   // instead of a dependent walk over the 512-byte group records at the head of every launch
  GemmGroup g[GEMM_MAX_GROUPS];
};
inline void gemm_finalize(GemmParams& p) {
  for (int i = 0; i < GEMM_MAX_GROUPS; ++i) p.grp_begin[i] = i < p.ngroups ? p.g[i].cta_begin : 0x7fffffff;
}

// ---- row-gather of one 128-byte line into a swizzled tile --------------------------------
MINPPO_DEVINL void gather_line(uint32_t tile_base, int line, const __nv_bfloat16* src) {
  const uint32_t dst = tile_base + line * 128;
  const int sw = line & 7;
#pragma unroll
  for (int j = 0; j < 8; ++j) cp_async_16(dst + ((j ^ sw) << 4), reinterpret_cast<const char*>(src) + j * 16);
}

// ---- 32x32 transpose-reduce: lane j ends with the sum over lanes of v[j] --------------------
MINPPO_DEVINL float warp_colsum32(float (&v)[32]) {
  const uint32_t lane = lane_id();
#pragma unroll
  for (int half = 16; half >= 1; half >>= 1) {
    const bool upper = (lane & half) != 0;
#pragma unroll
    for (int i = 0; i < half; ++i) {
      // keep the half of the columns selected by this lane's bit, send the other half
      float keep = upper ? v[i + half] : v[i];
      float send = upper ? v[i] : v[i + half];
      v[i] = keep + __shfl_xor_sync(0xffffffffu, send, half);
    }
  }
  return v[0];   // column index == lane (bit b of lane selected the upper half at step b)
}

// The whole CTA (GEMM_THREADS threads) calls this; it returns after the TMEM columns are released.
// Warps 0..5 carry the roles; a caller may run with more warps per CTA (dwopt.cuh): they only take part
// in the two CTA-wide barriers.
struct GemmNoIdle { MINPPO_DEVINL void operator()() const {} };
// `idle` runs on the helper warps (warps >= 6, if the caller has any) while the GEMM is in flight.
// Persistent callers (ppo_steps.cuh) pass the TMEM base they allocated once (`ext_tmem`; 0xFFFFFFFF = allocate and free
// here), per-step overrides of the gather row list / valid-row count, and get the mbarriers re-initialised on every call.
constexpr uint32_t GEMM_NO_TMEM = 0xFFFFFFFFu;
template <int EPI, typename IdleFn = GemmNoIdle>
MINPPO_DEVINL void umma_gemm_body(const GemmParams& p, uint8_t* smem_raw, long long* trace = nullptr, IdleFn idle = IdleFn(),
                                  uint32_t ext_tmem = GEMM_NO_TMEM, const int32_t* step_rowidx = nullptr,
                                  const int32_t* step_kcount = nullptr) {
#define GEMM_STAMP(slot) do { if (trace) trace[(slot)] = clock64(); } while (0)
  const uint32_t raw = smem_u32(smem_raw);
  const uint32_t base = (raw + 1023u) & ~1023u;                      // SWIZZLE_128B: 1024-B aligned tiles
  uint8_t* aligned = smem_raw + (base - raw);
  const uint32_t ones = base + GEMM_STAGES * GEMM_STAGE_BYTES;                             // 1024-byte aligned
  float* colsum_s = reinterpret_cast<float*>(aligned + GEMM_STAGES * GEMM_STAGE_BYTES + GEMM_ONES_BYTES);   // [4][MAXN]
  uint64_t* bars = reinterpret_cast<uint64_t*>(aligned + GEMM_STAGES * GEMM_STAGE_BYTES + GEMM_ONES_BYTES + 4 * GEMM_MAXN * 4);
  uint64_t* full_bar = bars;                       // [STAGES]
  uint64_t* empty_bar = bars + GEMM_STAGES;        // [STAGES]
  uint64_t* tmem_full_bar = bars + 2 * GEMM_STAGES;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * GEMM_STAGES + 1);
  uint64_t* chunk_bar = bars + 2 * GEMM_STAGES + 2;   // [8] EPI_PARTIAL: 32-column chunk c of the tile staged by its four warps

  const int warp = threadIdx.x >> 5;
  int grp = 0;
#pragma unroll
  for (int i = 1; i < GEMM_MAX_GROUPS; ++i) grp += static_cast<int>(blockIdx.x) >= p.grp_begin[i] ? 1 : 0;
  const GemmGroup& G = p.g[grp];
  const int rem = static_cast<int>(blockIdx.x) - G.cta_begin;
  const int AMODE = G.amode, BMODE = G.bmode;
  const int m_tile = rem / G.splits;
  const int split = rem % G.splits;
  // K extent: all of it, or only the k-blocks holding valid rows (env-sharded minibatches are padded to a worst-case
  // capacity; the count is device data and identical for every CTA of the launch)
  const int32_t* kcount = step_kcount ? step_kcount : G.k_count;
  const int kb_total = kcount ? min(G.kb_total, (max(*kcount, 0) + GEMM_BK - 1) / GEMM_BK) : G.kb_total;
  const int kb_per = (kb_total + G.splits - 1) / G.splits;
  const int kb0 = split * kb_per;
  const int kb1 = min(kb_total, kb0 + kb_per);
  const int nkb = max(0, kb1 - kb0);
  const int N = G.N;
  const bool kGather = (AMODE == A_GATHER_K || AMODE == A_GATHER_MN);
  const bool kTmaA = !kGather;
  // bias-gradient columns of this CTA: the m-tiles of one (group, split) share the N columns between them when
  // the shares are whole 64-column panels, otherwise m-tile 0 takes all of them
  const bool cs_even = (N % G.m_tiles) == 0 && ((N / G.m_tiles) % 64) == 0;
  const int cs_nc = cs_even ? N / G.m_tiles : (m_tile == 0 ? N : 0);
  const int cs_c0 = cs_even ? m_tile * cs_nc : 0;
  const bool kColsum = EPI == EPI_PARTIAL && G.colsum_out != nullptr && BMODE == B_TMA_MN && cs_nc > 0;
  constexpr uint32_t kTmemCols = EPI == EPI_PARTIAL ? 512 : 256;
  if (kColsum) {
    for (int i = threadIdx.x; i < GEMM_ONES_BYTES / 16; i += blockDim.x)
      sts128(ones + i * 16, make_uint4(0x3F803F80u, 0x3F803F80u, 0x3F803F80u, 0x3F803F80u));       // bf16 1.0
    fence_proxy_async_smem();
  }

  if (threadIdx.x == 0) {
    GEMM_STAMP(13);
    // tensor maps into the descriptor cache first: a cold descriptor fetch sits in front of the first operand load otherwise
    if (kTmaA) tma_prefetch_desc(&G.tmA);
    tma_prefetch_desc(&G.tmB);
    if (EPI == EPI_PARTIAL) tma_prefetch_desc(&G.tmC);
    for (int s = 0; s < GEMM_STAGES; ++s) {
      mbar_init(&full_bar[s], 1 + (kGather ? GEMM_EPI_THREADS : 0));
      mbar_init(&empty_bar[s], 1);
    }
    mbar_init(tmem_full_bar, 1);
    for (int c = 0; c < GEMM_MAXN / 32; ++c) mbar_init(&chunk_bar[c], 4);
    fence_mbar_init();
    GEMM_STAMP(15);
  }
  if (warp == 1 && ext_tmem == GEMM_NO_TMEM) {
    tmem_alloc(tmem_slot, kTmemCols);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = ext_tmem == GEMM_NO_TMEM ? *tmem_slot : ext_tmem;
  if (threadIdx.x == 64) GEMM_STAMP(6);                 // prologue done

  // EPI_PARTIAL: warps beyond the six role warps (a caller running more warps per CTA, dwopt.cuh) help draining the
  // accumulator: the 32-column chunks of a TMEM lane quadrant are dealt round-robin to the warps sharing it.
  const int nwarps = static_cast<int>(blockDim.x) >> 5;
  const int pq = warp & 3;
  const int first_helper = 6 + ((pq - 2) & 3);
  const int helpers_q = (EPI == EPI_PARTIAL && first_helper < nwarps) ? (nwarps - 1 - first_helper) / 4 + 1 : 0;
  const int drain_members = 1 + helpers_q;
  const int drain_idx = warp < 6 ? 0 : 1 + (warp - first_helper) / 4;

  if (warp == 0) {
    // ===================== TMA producer =====================
    if (elect_one()) {
      griddep_wait();                  // PDL (common.cuh): operands are written by the preceding kernel
      griddep_launch();
      if (ext_tmem != GEMM_NO_TMEM)    // persistent callers: the operands were published through a grid barrier (generic-proxy
        fence_proxy_async_global();    // acquire) -- order the TMA (async-proxy) reads below after it
      GEMM_STAMP(7);                   // dependency wait passed
      const uint32_t a_bytes = kTmaA ? GEMM_A_BYTES : 0;
      const uint32_t b_bytes = static_cast<uint32_t>(N) * GEMM_BK * 2;
      for (int i = 0; i < nkb; ++i) {
        const int s = i % GEMM_STAGES;
        const uint32_t ph = (i / GEMM_STAGES) & 1;
        mbar_wait(&empty_bar[s], ph ^ 1);
        const uint32_t sa = base + s * GEMM_STAGE_BYTES;
        const uint32_t sb = sa + GEMM_A_BYTES;
        mbar_arrive_expect_tx(&full_bar[s], a_bytes + b_bytes);
        const int kb = kb0 + i;
        if (AMODE == A_TMA_K) {
          tma_load_2d(sa, &G.tmA, &full_bar[s], kb * GEMM_BK, m_tile * GEMM_BM);           // box {64 k, 128 m}
        } else if (AMODE == A_TMA_MN) {
          tma_load_2d(sa, &G.tmA, &full_bar[s], m_tile * GEMM_BM, kb * GEMM_BK);           // box {64 m, 64 k}
          tma_load_2d(sa + 8192, &G.tmA, &full_bar[s], m_tile * GEMM_BM + 64, kb * GEMM_BK);
        }
        if (BMODE == B_TMA_K) {
          tma_load_2d(sb, &G.tmB, &full_bar[s], kb * GEMM_BK, G.n_off);                    // box {64 k, N}
        } else {
          for (int c = 0; c < N / 64; ++c)
            tma_load_2d(sb + c * 8192, &G.tmB, &full_bar[s], G.n_off + c * 64, kb * GEMM_BK);   // box {64 n, 64 k}
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    if (elect_one()) {
      const uint32_t idesc = umma_idesc_bf16(GEMM_BM, static_cast<uint32_t>(N),
                                             (AMODE == A_TMA_MN || AMODE == A_GATHER_MN) ? 1u : 0u,
                                             (BMODE == B_TMA_MN) ? 1u : 0u);
      for (int i = 0; i < nkb; ++i) {
        const int s = i % GEMM_STAGES;
        const uint32_t ph = (i / GEMM_STAGES) & 1;
        mbar_wait(&full_bar[s], ph);
        tc_fence_after();
        if (i == 0) GEMM_STAMP(8);     // first operands landed
        const uint32_t sa = base + s * GEMM_STAGE_BYTES;
        const uint32_t sb = sa + GEMM_A_BYTES;
#pragma unroll
        for (int j = 0; j < GEMM_BK / 16; ++j) {
          uint64_t da, db;
          if (AMODE == A_TMA_K || AMODE == A_GATHER_K) da = umma_smem_desc(sa + j * 32, 16, 1024);
          else da = umma_smem_desc(sa + j * 2048, 8192, 1024);
          if (BMODE == B_TMA_K) db = umma_smem_desc(sb + j * 32, 16, 1024);
          else db = umma_smem_desc(sb + j * 2048, 8192, 1024);
          umma_bf16(tmem_base, da, db, idesc, (i > 0 || j > 0) ? 1u : 0u);
          if (kColsum)         // D[:, c] += sum_k 1 * B[k][c]: every accumulator row holds the column sums
            umma_bf16(tmem_base + 256, umma_smem_desc(ones + j * 32, 16, 1024),
                      umma_smem_desc(sb + j * 2048 + (cs_c0 >> 6) * 8192, 8192, 1024),
                      umma_idesc_bf16(GEMM_BM, static_cast<uint32_t>(cs_nc), 0u, 1u), (i > 0 || j > 0) ? 1u : 0u);
        }
        umma_commit(&empty_bar[s]);          // frees the smem slot once these MMAs retire
      }
      umma_commit(tmem_full_bar);            // accumulator complete
      GEMM_STAMP(9);                         // all MMAs issued
      if (EPI == EPI_PARTIAL) {
        // This thread is idle from here on: it TMA-stores each 32-column chunk of the fp32 tile as soon as the four
        // warps draining it have staged it (tmC: fp32 [splits][m_store][N], box {32, 128, 1}; rows >= m_store are
        // clipped by the TMA unit), so the store overlaps the rest of the drain.
        for (int c = 0; c < N / 32; ++c) {
          mbar_wait(&chunk_bar[c], 0);
          if (c == 0) GEMM_STAMP(11);          // first chunk staged
          tma_store_3d(base + c * 16384, &G.tmC, G.n_off + c * 32, m_tile * GEMM_BM, split);
        }
        tma_store_commit();
        tma_store_wait_all0();
        fence_proxy_async_global();
        GEMM_STAMP(12);                        // partial tile written
      }
    }
  } else if (warp < GEMM_THREADS / 32) {
    // ===================== gather producer (optional) + epilogue =====================
    const int et = threadIdx.x - 64;         // 0..127
    if (kGather) {
      // Row indices are prefetched 8 k-blocks at a time (one dependent global load per batch, not
      // per k-block) and up to GEMM_STAGES - 1 cp.async groups stay in flight before publishing.
      const int32_t* ridx = step_rowidx ? step_rowidx : G.rowidx;
      constexpr int LAG = GEMM_STAGES - 1;
      const int c = et >> 6, kr = et & 63;
      const int row_k = (AMODE == A_GATHER_K) ? ridx[m_tile * GEMM_BM + et] : 0;
      int rows[8];
      for (int i = 0; i < nkb; ++i) {
        if ((i & 7) == 0 && AMODE == A_GATHER_MN) {
#pragma unroll
          for (int u = 0; u < 8; ++u) rows[u] = (i + u < nkb) ? ridx[(kb0 + i + u) * GEMM_BK + kr] : 0;
        }
        const int s = i % GEMM_STAGES;
        const uint32_t ph = (i / GEMM_STAGES) & 1;
        mbar_wait(&empty_bar[s], ph ^ 1);
        const uint32_t sa = base + s * GEMM_STAGE_BYTES;
        const int kb = kb0 + i;
        if (AMODE == A_GATHER_K) {
          gather_line(sa, et, G.gimage + static_cast<size_t>(row_k) * G.ldg + kb * GEMM_BK);
        } else {
          int row = rows[0];
#pragma unroll
          for (int u = 1; u < 8; ++u) row = ((i & 7) == u) ? rows[u] : row;
          gather_line(sa + c * 8192, kr, G.gimage + static_cast<size_t>(row) * G.ldg + m_tile * GEMM_BM + c * 64);
        }
        cp_async_commit();
        if (i >= LAG) {
          cp_async_wait<LAG>();
          fence_proxy_async_smem();
          mbar_arrive(&full_bar[(i - LAG) % GEMM_STAGES]);
        }
      }
      for (int j = max(0, nkb - LAG); j < nkb; ++j) {          // drain: publish the last groups in order
        const int left = nkb - 1 - j;                          // groups that may still be in flight
        if (left >= 2) cp_async_wait<2>();
        else if (left == 1) cp_async_wait<1>();
        else cp_async_wait<0>();
        fence_proxy_async_smem();
        mbar_arrive(&full_bar[j % GEMM_STAGES]);
      }
    }

    // ---- epilogue ----
    const int q = warp & 3;                                   // TMEM lane quadrant of this warp
    const int row = m_tile * GEMM_BM + q * 32 + static_cast<int>(lane_id());
    if (nkb > 0) {
      mbar_wait(tmem_full_bar, 0);
      tc_fence_after();
    }
    if (et == 0) GEMM_STAMP(10);                // accumulator complete
    const uint32_t taddr = tmem_base + (static_cast<uint32_t>(q * 32) << 16);
    const int ldc = G.ldc ? G.ldc : N;
    for (int c0 = 32 * drain_idx; c0 < N; c0 += 32 * drain_members) {
      float v[32];
      if (nkb > 0) {
        tmem_ld_32x32(taddr + c0, v);
        tmem_ld_wait();
      } else {
#pragma unroll
        for (int j = 0; j < 32; ++j) v[j] = 0.f;
      }
      if (EPI == EPI_ACT) {
        const float* bp = G.bias + G.n_off + c0;   // leaf offsets in the arena are only 4-byte aligned
        uint32_t w[16];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          float x0 = v[4 * j] + __ldg(bp + 4 * j), x1 = v[4 * j + 1] + __ldg(bp + 4 * j + 1);
          float x2 = v[4 * j + 2] + __ldg(bp + 4 * j + 2), x3 = v[4 * j + 3] + __ldg(bp + 4 * j + 3);
          if (G.act == ACT_RELU) {
            x0 = fmaxf(x0, 0.f); x1 = fmaxf(x1, 0.f); x2 = fmaxf(x2, 0.f); x3 = fmaxf(x3, 0.f);
          } else if (G.act == ACT_TANH_FAST) {
            x0 = fast_tanh(x0); x1 = fast_tanh(x1); x2 = fast_tanh(x2); x3 = fast_tanh(x3);
          } else {
            x0 = exp_tanh(x0); x1 = exp_tanh(x1); x2 = exp_tanh(x2); x3 = exp_tanh(x3);
          }
          w[2 * j] = pack_bf16x2(x0, x1);
          w[2 * j + 1] = pack_bf16x2(x2, x3);
        }
        uint4* o = reinterpret_cast<uint4*>(reinterpret_cast<__nv_bfloat16*>(G.out) + static_cast<size_t>(row) * G.ldo + G.n_off + c0);
#pragma unroll
        for (int j = 0; j < 4; ++j) o[j] = make_uint4(w[4 * j], w[4 * j + 1], w[4 * j + 2], w[4 * j + 3]);
      } else if (EPI == EPI_DACT) {
        const uint4* h4 = reinterpret_cast<const uint4*>(G.hprev + static_cast<size_t>(row) * G.ldh + G.n_off + c0);
        uint32_t w[16];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const uint4 hh = __ldg(h4 + j);
          const uint32_t hw[4] = {hh.x, hh.y, hh.z, hh.w};
#pragma unroll
          for (int t = 0; t < 4; ++t) {
            const float h0 = bf16_lo(hw[t]), h1 = bf16_hi(hw[t]);
            float d0, d1;
            if (G.act == ACT_RELU) { d0 = h0 > 0.f ? 1.f : 0.f; d1 = h1 > 0.f ? 1.f : 0.f; }
            else { d0 = 1.f - h0 * h0; d1 = 1.f - h1 * h1; }
            const int e = 8 * j + 2 * t;
            v[e] *= d0; v[e + 1] *= d1;
            w[4 * j + t] = pack_bf16x2(v[e], v[e + 1]);
            // bias gradient sums what the dW GEMM will see: the bf16-rounded dZ
            v[e] = bf16_lo(w[4 * j + t]); v[e + 1] = bf16_hi(w[4 * j + t]);
          }
        }
        uint4* o = reinterpret_cast<uint4*>(reinterpret_cast<__nv_bfloat16*>(G.out) + static_cast<size_t>(row) * G.ldo + G.n_off + c0);
#pragma unroll
        for (int j = 0; j < 4; ++j) o[j] = make_uint4(w[4 * j], w[4 * j + 1], w[4 * j + 2], w[4 * j + 3]);
        const float cs = warp_colsum32(v);
        colsum_s[q * GEMM_MAXN + c0 + lane_id()] = cs;
      } else {  // EPI_PARTIAL: stage the fp32 tile in the (now idle) operand ring, SW128, then TMA-store it
        const int r = q * 32 + static_cast<int>(lane_id());
        const uint32_t dst = base + (c0 >> 5) * 16384 + r * 128;      // chunk tile: [128 rows][32 floats]
#pragma unroll
        for (int j = 0; j < 8; ++j)
          sts128(dst + ((j ^ (r & 7)) << 4),
                 make_uint4(__float_as_uint(v[4 * j]), __float_as_uint(v[4 * j + 1]), __float_as_uint(v[4 * j + 2]),
                            __float_as_uint(v[4 * j + 3])));
        fence_proxy_async_smem();
        __syncwarp();
        if (lane_id() == 0) mbar_arrive(&chunk_bar[c0 >> 5]);
      }
    }
    if (kColsum) {
      // all 128 accumulator rows are equal: warp q picks 32-column chunks q, q + 4, ..., lane i keeps column i
      for (int ch = q; ch < cs_nc / 32; ch += 4) {
        float v[32];
        if (nkb > 0) {
          tmem_ld_32x32(taddr + 256 + ch * 32, v);
          tmem_ld_wait();
        } else {
#pragma unroll
          for (int j = 0; j < 32; ++j) v[j] = 0.f;
        }
        float out = v[0];
#pragma unroll
        for (int j = 1; j < 32; ++j) out = (static_cast<int>(lane_id()) == j) ? v[j] : out;
        G.colsum_out[static_cast<size_t>(split) * ldc + G.n_off + cs_c0 + ch * 32 + lane_id()] = out;
      }
    }
    if (EPI == EPI_DACT) {
      asm volatile("bar.sync 1, 128;" ::: "memory");
      for (int c = et; c < N; c += GEMM_EPI_THREADS) {
        const float s = (colsum_s[c] + colsum_s[GEMM_MAXN + c]) + (colsum_s[2 * GEMM_MAXN + c] + colsum_s[3 * GEMM_MAXN + c]);
        G.colsum[static_cast<size_t>(m_tile) * ldc + G.n_off + c] = s;
      }
    }
  }

  else if (EPI == EPI_PARTIAL) {
    // ===================== helper warps: drain their share of the accumulator =====================
    const int r = pq * 32 + static_cast<int>(lane_id());
    idle();
    if (nkb > 0) {
      mbar_wait(tmem_full_bar, 0);
      tc_fence_after();
    }
    const uint32_t taddr = tmem_base + (static_cast<uint32_t>(pq * 32) << 16);
    for (int c0 = 32 * drain_idx; c0 < N; c0 += 32 * drain_members) {
      float v[32];
      if (nkb > 0) {
        tmem_ld_32x32(taddr + c0, v);
        tmem_ld_wait();
      } else {
#pragma unroll
        for (int j = 0; j < 32; ++j) v[j] = 0.f;
      }
      const uint32_t dst = base + (c0 >> 5) * 16384 + r * 128;
#pragma unroll
      for (int j = 0; j < 8; ++j)
        sts128(dst + ((j ^ (r & 7)) << 4),
               make_uint4(__float_as_uint(v[4 * j]), __float_as_uint(v[4 * j + 1]), __float_as_uint(v[4 * j + 2]),
                          __float_as_uint(v[4 * j + 3])));
      fence_proxy_async_smem();
      __syncwarp();
      if (lane_id() == 0) mbar_arrive(&chunk_bar[c0 >> 5]);
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1 && ext_tmem == GEMM_NO_TMEM) tmem_dealloc(tmem_base, kTmemCols);
}

template <int EPI>
__global__ void __launch_bounds__(GEMM_THREADS, 1) umma_gemm_kernel(const __grid_constant__ GemmParams p) {
  extern __shared__ uint8_t smem_raw[];
  umma_gemm_body<EPI>(p, smem_raw);
}

}  // namespace minppo
