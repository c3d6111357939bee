// minppo_b200 -- weight-gradient GEMMs + gradient reduction + global-norm clip + Adam in ONE launch
// (replaces jax.value_and_grad's dW contractions, optax.chain(clip_by_global_norm, adam) and
//  TrainState.apply_gradients: /root/reference/minppo/train.py:98-124, 246-248).
//
// Grid = one CTA per SM, all co-resident (one grid barrier):
//   phase 1  CTAs [0, gemm_ctas): split-K tcgen05 GEMM dW_l = act_l^T dZ_{l+1} for every hidden layer of both
//            nets (umma_gemm_body<EPI_PARTIAL>), fp32 partial tiles -> L2 by TMA store; then each CTA counts its
//            output tile's completion counter up (S CTAs per tile).
//            CTAs [gemm_ctas, grid): meanwhile sum the per-tile partials of the SMALL leaves (biases, output
//            heads, log_std: one partial per 128-row tile of the fused step kernel) and the loss sums -> gflat,
//            then count the small-leaf counter up.
//   phase 2  fixed-order sum of the split-K partials of the hidden kernels -> gflat (bitwise reproducible, no
//            atomics; 16-byte loads, 16 partials in flight per thread), sum of squares -> per-block partial.
//            Every thread first waits for the counter(s) of the tile(s) its units lie in: it depends on the S CTAs
//            of that tile only, not on the whole grid.
//   barrier
//   phase 3  clip scale, Adam, params / mu / nu in place, bf16 weight images for the next step's GEMMs.
// The counters are reset to zero after the barrier, when every wait of the launch has been satisfied; the next
// launch's producers run behind this launch's end (griddepcontrol.wait), so the counters need no generations.
// The phases are plain strided loops (no per-element unrolling): an earlier fully unrolled version was
// 15k SASS instructions and spent a third of its time on instruction-cache misses.
// Launched without GEMM CTAs (gemm_ctas == 0), every CTA is a spare CTA: after a stand-alone dW GEMM launch when the GEMM
// grid does not fit one CTA per SM, and to apply an all-reduced gradient (learner.cu fill_apply_only).
// With env-sharded ranks that do not exchange over peer memory (do_apply == 0) the kernel stops after phase 2 and the
// barrier (the counter reset needs it) with the local gradient SUM in gflat; the NCCL all-reduce and that apply-only
// launch follow.
#pragma once

#include "opt_common.cuh"
#include "umma_gemm.cuh"

namespace minppo {

// 16 warps per CTA: warps 0..5 run the GEMM roles in phase 1, all of them the element-wise phases (one CTA
// per SM: with 6 warps the dependent divide / sqrt chains of the Adam phase had nothing to hide behind)
constexpr int DWOPT_THREADS = 512;

// Gradient exchange over NVLink peer memory, Lamport style.  ONE-SHOT variant: every rank pushes its local gradient sums into
// a staging slot on every OTHER rank; the staging words themselves are the arrival flags (sentinel -0.0f until written),
// so an exchange costs one NVLink one-way latency -- no release/acknowledge round and no flag round.  Every rank then
// sums the W contributions in rank order (same values, same order: bit-identical gradients on all ranks with no
// broadcast), resets the words it consumed to the sentinel and continues with the norm and Adam like a single GPU.
// TWO-PHASE variant (W >= 4): see the exchange code in dwopt_kernel.
// Exchange allocation of one rank (exported by CUDA IPC):
//   stage [2][W][np] f32   slot (n & 1, q): rank q's local gradient of exchange n (all words start as the sentinel).
//                          Inside a slot: the 4-element units of the late leaves (16-byte aligned), then the early
//                          elements and the LOSS_SUMS loss sums (dwopt job numbering).  The element -> (CTA, thread)
//                          mapping is the same on every rank: a thread only ever waits for its own unit.
//   (pad)  [W][256] u32    unused (was: the arrival flags of the earlier release/acquire protocol).
//   result [2][np] f32     two-phase variant: the reduced gradient of exchange n, pushed by the owners of its units.
struct PeerXchg {
  char* base[MINPPO_MAX_RANKS];  // rank r's allocation as mapped on THIS device
  unsigned int* seq;             // local exchange counter (device memory): exchanges completed so far
  int world, rank;
  int np;                        // floats per staging slot (multiple of 4)
  int two_phase;                 // 0: one-shot push to every rank; 1: reduce at rank (CTA index % W), result pushed back
};
MINPPO_DEVINL float* px_stage(const PeerXchg& x, int r, unsigned int par, int q) {
  return reinterpret_cast<float*>(x.base[r]) + (static_cast<size_t>(par) * x.world + q) * x.np;
}
// result slots of the two-phase exchange: [2][np] f32 behind the flags
MINPPO_DEVINL float* px_result(const PeerXchg& x, int r, unsigned int par) {
  return reinterpret_cast<float*>(x.base[r]) + 2 * static_cast<size_t>(x.world) * x.np + static_cast<size_t>(x.world) * 256 +
         static_cast<size_t>(par) * x.np;
}
// system-scope accesses for memory another GPU reads or writes
MINPPO_DEVINL float4 ld_sys_v4(const float* p) {
  float4 v;
  asm volatile("ld.relaxed.sys.global.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p) : "memory");
  return v;
}
MINPPO_DEVINL void st_sys_f32(float* p, float v) { asm volatile("st.relaxed.sys.global.f32 [%0], %1;" ::"l"(p), "f"(v) : "memory"); }
MINPPO_DEVINL void st_sys_v4(float* p, float4 v) {
  asm volatile("st.relaxed.sys.global.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}
MINPPO_DEVINL unsigned int ld_relaxed_sys_u32(const unsigned int* p) {
  unsigned int v;
  asm volatile("ld.relaxed.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
// Split-K completion counters (DwOptParams::done), one per 128-byte line: ~2k warps poll them in phase 2, and counters
// sharing a line would put all of that on one L2 slice.
constexpr int DWOPT_DONE_STRIDE = 32;
MINPPO_DEVINL void red_release_add(unsigned int* p, unsigned int v) {
  asm volatile("red.release.gpu.global.add.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
// wait until *p >= target; bounded like grid_barrier: past the bound the error flag goes up instead of a hang
MINPPO_DEVINL void wait_count(const unsigned int* p, unsigned int target, int* err_flag) {
  const long long t0 = clock64();
  for (;;) {
    unsigned int v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    if (v >= target) break;
    if (clock64() - t0 > 4000000000LL) { atomicExch(err_flag, MINPPO_ERR_BARRIER); break; }
  }
}
// Wait until the split-K partials of the 4-element unit at element e of late leaf L are complete: the counter of the dW
// GEMM tile that wrote them reaches S (the layer-wise path's bias leaves: every tile of the layer, each writes some columns).
MINPPO_DEVINL void wait_late_unit(const unsigned int* done, const OptLeaf& L, int e, unsigned int S, int* err_flag) {
  int k = L.tile0, n = L.tile_n;
  if (L.tile_split) {                                    // hidden kernel [in][out]: column group, then 128-row m-tile
    const int i = e / L.cols, j = e - i * L.cols;
    k += (j >= L.tile_split ? n >> 1 : 0) + (i >> 7);
    n = 1;
  }
  for (const int end = k + n; k < end; ++k) wait_count(done + k * DWOPT_DONE_STRIDE, S, err_flag);
}

// four consecutive fp32 of an arena (L2-coherent: ld.cg / plain st), by the widest access the address allows
MINPPO_DEVINL void ld_unit(const float* p, float (&v)[4]) {
  const uintptr_t a = reinterpret_cast<uintptr_t>(p);
  if ((a & 15u) == 0) { const float4 q = __ldcg(reinterpret_cast<const float4*>(p)); v[0] = q.x; v[1] = q.y; v[2] = q.z; v[3] = q.w; }
  else if ((a & 7u) == 0) {
    const float2 q0 = __ldcg(reinterpret_cast<const float2*>(p)), q1 = __ldcg(reinterpret_cast<const float2*>(p) + 1);
    v[0] = q0.x; v[1] = q0.y; v[2] = q1.x; v[3] = q1.y;
  } else {
#pragma unroll
    for (int e = 0; e < 4; ++e) v[e] = __ldcg(p + e);
  }
}
MINPPO_DEVINL void st_unit(float* p, const float (&v)[4]) {
  const uintptr_t a = reinterpret_cast<uintptr_t>(p);
  if ((a & 15u) == 0) *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2], v[3]);
  else if ((a & 7u) == 0) { reinterpret_cast<float2*>(p)[0] = make_float2(v[0], v[1]); reinterpret_cast<float2*>(p)[1] = make_float2(v[2], v[3]); }
  else {
#pragma unroll
    for (int e = 0; e < 4; ++e) p[e] = v[e];
  }
}

struct alignas(64) DwOptParams {
  GemmParams gemm;               // the per-step row list / valid-row count of the groups come from the arrays below
  OptArgs opt;                   // losses_out / gnorm_out: bases of the per-step arrays (losses_stride floats apart / 1 apart)
  int gemm_ctas;                 // CTAs [0, gemm_ctas) run the GEMM; the others pre-reduce the small leaves (gemm.g[0].splits
                                 // >= 1 also at 0: the counter reset divides by it)
  long long* trace;              // debug: [grid][16] clock64 stamps (null = off)
  unsigned int* done;            // [1 + gemm_ctas / S][DWOPT_DONE_STRIDE] completion counters (zero at launch, reset at its end):
                                 // [0] small-leaf CTAs done, [1 + b / S] split-K tile of GEMM CTA b: S partials stored
  // Gradient exchange over NVLink peer memory (env-sharded ranks; world == 0: not configured).  Every rank exports
  // one allocation [stage | pad | result] (PeerXchg above); base[r] is rank r's copy as mapped HERE.
  PeerXchg px;
  // per-update arrays, indexed by the minibatch step s = e * M + k
  const int32_t* ridx_base;      // [EM][cap] row lists (gather groups of the GEMM; L2 prefetch of the NEXT step's rows)
  const int32_t* counts;         // [EM] rows of each minibatch on this rank
  int cap, EM;
  int padded;                    // 1: row lists are sized for a worst case, counts[] bound the per-minibatch work
  int losses_stride;             // floats between the losses of consecutive steps (4; 0 = every step writes the scratch slot)
  int part_rows;                 // minibatch rows per early-leaf partial (128: fused step kernel, 64: head_loss kernel)
  const __nv_bfloat16* obs_img;  // [Bl][obs_ld]
  int obs_ld;
  int step;                      // the minibatch step of this launch
};

template <int NTHREADS_MAX = 1024>
MINPPO_DEVINL float block_sum_dyn(float v, float* scratch /*[32]*/) {
  const int nw = static_cast<int>(blockDim.x) >> 5;
  v = warp_sum(v);
  if ((threadIdx.x & 31) == 0) scratch[threadIdx.x >> 5] = v;
  __syncthreads();
  float s = 0.f;
  if (threadIdx.x < 32) {
    s = static_cast<int>(threadIdx.x) < nw ? scratch[threadIdx.x] : 0.f;
    s = warp_sum(s);
  }
  __syncthreads();
  return s;                                   // valid in warp 0
}

// MAXU = 4-element units of the hidden kernels a thread may own (fast path: reduced gradient and optimizer state stay in
// registers across the grid barrier).  MAXU = 1 covers P_late <= 4 * grid * 512 (303k parameters on 148 SMs: the
// stand-in shape); larger observation widths take MAXU = 2 or 4.
template <int MAXU>
__global__ void __launch_bounds__(DWOPT_THREADS, 1) dwopt_kernel(const __grid_constant__ DwOptParams p) {
  extern __shared__ uint8_t smem_raw[];
  __shared__ float scratch[32];
  __shared__ float s_bcast[4];
  __shared__ LeafTab T;
  const OptArgs& a = p.opt;
  const int P = a.P, step = p.step;
  const int G = static_cast<int>(gridDim.x), NT = static_cast<int>(blockDim.x);
  const int32_t* row_count = p.padded ? p.counts + step : nullptr;          // rows of this minibatch on this rank
  const int32_t* next_ridx = step + 1 < p.EM ? p.ridx_base + static_cast<size_t>(step + 1) * p.cap : nullptr;
  const int32_t* next_count = p.padded ? p.counts + step + 1 : nullptr;
  float* losses_out = a.losses_out ? a.losses_out + static_cast<size_t>(step) * p.losses_stride : nullptr;
  float* gnorm_out = a.gnorm_out ? a.gnorm_out + step : nullptr;
  const int b = static_cast<int>(blockIdx.x), t = static_cast<int>(threadIdx.x);
  const bool has_extra = p.gemm_ctas < G;
#define DW_STAMP(slot) do { if (p.trace && t == 0) p.trace[static_cast<size_t>(b) * 16 + (slot)] = clock64(); } while (0)
  float ss = 0.f;
  DW_STAMP(0);
  __shared__ unsigned int s_seq;
  __shared__ int s_dead;                                  // error flag already up when this launch started
  __shared__ unsigned long long s_waited;                 // trace: when this CTA's last counter wait was satisfied (clock64)
  const bool px_on = p.px.world > 1;                     // gradient exchange over peer memory fused into this launch
  if (p.trace && t == 0) s_waited = 0ull;
  if (px_on && t == 0) {
    s_seq = __ldcg(p.px.seq) + 1u;                       // number of this exchange
    s_dead = __ldcg(a.err_flag) != 0;
  }
  // The leaf table (kernel parameters -> shared memory: cold constant-bank misses, ~2k cycles at the head of a launch) is first
  // read in phase 2.  GEMM CTAs: the helper warps copy it while the GEMM is in flight (the CTA-wide barrier at the end of the GEMM
  // body orders it); spare CTAs need it at once.
  const bool gemm_cta = b < p.gemm_ctas;
  if (!gemm_cta) {
    leaf_tab_build(T, a, t, NT);
    __syncthreads();
  }
  DW_STAMP(14);

  // Per-step scalars (two powf, A exp/log): computed by the last thread, whose warp has no GEMM role, while the
  // GEMM is in flight (GEMM CTAs) or up front (spare CTAs) -- never in phase 2, never in front of the
  // CTA-wide barrier of the GEMM prologue.
  const bool scal_thread = t == NT - 1;
  int count = 0;
  float ent = a.entropy_const;                           // A * (0.5 + 0.5 log 2pi) + sum log|scale|
  auto scalars = [&]() {
    if (scal_thread && a.do_apply) {
      count = __ldcg(a.count);                           // Adam step count BEFORE this step
      step_scalars(a, count, s_bcast[1], s_bcast[2], s_bcast[3]);
      if (b == 0 && losses_out) {
        // train.py:240 -- evaluated with the PRE-update log_std (nothing is updated before the grid barrier)
        for (int j = 0; j < a.A; ++j) ent += logf(fabsf(expf(__ldcg(a.params + a.off_logstd + j))));
      }
    }
  };

  // ---- phase 1 ----------------------------------------------------------------------------------
  if (gemm_cta) {
    // Helper warps (idle until the accumulator is complete): the per-step scalars, and this CTA's share of the L2
    // prefetch of the NEXT minibatch's observation rows (row lists and the observation image are static during an
    // update: no dependency on the preceding kernel).  Spread over all GEMM CTAs so that it never rides on the few
    // spare CTAs, whose number depends on the split-K factor.
    auto idle_work = [&]() {
      leaf_tab_build(T, a, t - GEMM_THREADS, NT - GEMM_THREADS);
      scalars();
      if (next_ridx) {
        const int HELPERS = NT - GEMM_THREADS;
        const int h = t - GEMM_THREADS;
        const int lines = (p.obs_ld * 2) >> 7;
        const int nrows = next_count ? min(p.cap, __ldcg(next_count)) : p.cap;
        for (int j = b * HELPERS + h; j < nrows * lines; j += p.gemm_ctas * HELPERS) {
          const char* row = reinterpret_cast<const char*>(p.obs_img + static_cast<size_t>(next_ridx[j / lines]) * p.obs_ld);
          asm volatile("prefetch.global.L2 [%0];" ::"l"(row + (j % lines) * 128));
        }
      }
    };
    umma_gemm_body<EPI_PARTIAL>(p.gemm, smem_raw, p.trace ? p.trace + static_cast<size_t>(b) * 16 : nullptr, idle_work,
                                p.ridx_base + static_cast<size_t>(step) * p.cap, row_count);   // PDL wait / trigger inside
  } else {
    scalars();
    griddep_wait();                                      // the small-leaf partials come from the fused step kernel
    if (t == 0) griddep_launch();
    const int e = b - p.gemm_ctas, ne = G - p.gemm_ctas;
    const int live_tiles = row_count ? (max(__ldcg(row_count), 0) + p.part_rows - 1) / p.part_rows : 0x7fffffff;
    ss = reduce_leaves<false>(a, T, e * NT + t, ne * NT, live_tiles);
  }
  // Publish this CTA's phase-1 output: one count on its tile's counter (GEMM CTAs) or on the small-leaf counter.  The GEMM's
  // partial tile is an async-proxy (TMA) write that phase 2 reads with generic loads: the storing thread waited for it with
  // cp.async.bulk.wait_group 0 (the writes done, not only the shared-memory reads that .read waits for) and then issued
  // fence.proxy.async.global, which orders those writes before its later generic operations.  This CTA barrier carries them,
  // and every other thread's plain stores (small-leaf gflat, the layer-wise path's bias column sums), to thread 0, whose
  // release add makes all of it visible to a consumer's acquire load of the counter.  (The barrier also keeps the phase-2
  // set-up from being scheduled into phase 1: without it the kernel spills at MAXU = 2 and 4.)
  const unsigned int S = static_cast<unsigned int>(p.gemm.g[0].splits);
  __syncthreads();
  if (t == 0) red_release_add(p.done + (gemm_cta ? (1 + b / S) * DWOPT_DONE_STRIDE : 0), 1u);
  DW_STAMP(1);
  auto wait_unit = [&](const OptLeaf& L, int e) {
    wait_late_unit(p.done, L, e, S, a.err_flag);
    if (p.trace) atomicMax(&s_waited, static_cast<unsigned long long>(clock64()));
  };

  // ---- phase 2 ----------------------------------------------------------------------------------
  // Fast path: at most MAXU 4-element units of a hidden kernel per thread, so the reduced gradient and the optimizer
  // state of those elements stay in registers across the grid barrier and only the small leaves go through gflat.
  int n_units = 0;
  for (int l = 0; l < T.nleaves; ++l)
    if (T.leaf[l].late) n_units += T.size[l] >> 2;
  const int GT_ = G * NT;
  const bool fast = n_units <= GT_ * MAXU;
  // job number of this thread for the per-element work on the SMALL leaves (reduction, exchange, Adam).  (Dealing the jobs
  // round-robin over the CTAs instead -- t * G + b -- was measured: every CTA's Adam phase then carries one more dependent
  // load -> divide chain, 6.5k -> 12.5k cycles; concentrated on the first CTAs the chain hides behind the grid barrier.)
  const int gtid = b * NT + t;
  float4 g4[MAXU];
  float pv[MAXU][4], mv[MAXU][4], nv[MAXU][4];
  int ul[MAXU], ui[MAXU];                                // leaf and first arena index of each of this thread's units
  if (!has_extra) ss += reduce_leaves<false>(a, T, gtid, GT_, row_count ? (max(__ldcg(row_count), 0) + p.part_rows - 1) / p.part_rows : 0x7fffffff);
  // units dealt to warps round-robin over the CTAs (balanced, 512 contiguous bytes per warp and partial)
  const int unit0 = (((t >> 5) * G + b) << 5) + (t & 31);
#pragma unroll
  for (int u = 0; u < MAXU; ++u) { ul[u] = -1; ui[u] = 0; g4[u] = make_float4(0.f, 0.f, 0.f, 0.f); }
  if (fast) {
#pragma unroll
    for (int u = 0; u < MAXU; ++u) {
      const int unit = unit0 + u * GT_;
      if (unit < n_units) {
        int x = unit, l = 0;
        for (; l < T.nleaves; ++l) {
          if (!T.leaf[l].late) continue;
          const int n = T.size[l] >> 2;
          if (x < n) break;
          x -= n;
        }
        const OptLeaf& L = T.leaf[l];
        ul[u] = l; ui[u] = L.offset + 4 * x;
        if (a.do_apply) {
          // the arena offset of a leaf is only 4-byte aligned in general (act_dim is arbitrary): widest aligned access.
          // Issued before the counter wait: phase 1 does not write them.
          ld_unit(a.params + ui[u], pv[u]); ld_unit(a.mu + ui[u], mv[u]); ld_unit(a.nu + ui[u], nv[u]);
        }
        wait_unit(L, 4 * x);
        g4[u] = sum_partials16_v4<8>(L.grad_src + L.src_offset + 4 * x, L.nparts, L.part_stride);
        if (!px_on) {
          const float gq[4] = {g4[u].x, g4[u].y, g4[u].z, g4[u].w};
          st_unit(a.gflat + ui[u], gq);
          ss = fmaf(g4[u].x, g4[u].x, ss); ss = fmaf(g4[u].y, g4[u].y, ss); ss = fmaf(g4[u].z, g4[u].z, ss); ss = fmaf(g4[u].w, g4[u].w, ss);
        }
      }
    }
  } else {
    ss += reduce_leaves<true>(a, T, gtid, GT_, 0x7fffffff, wait_unit);
  }

  if (px_on) {
    // ---- one-shot all-reduce over NVLink peer memory (PeerXchg above; requires the fast path) -----------------
    const PeerXchg& X = p.px;
    const int R = X.rank;
    const int W = X.world;
    // Once the error flag is up (a peer never delivered within the bound, or any earlier device-side guard fired) the
    // exchange stops waiting: the update is already lost (minppo_ctx_check reports it), and 128 steps x the spin bound
    // must not turn one dead peer into a quarter of an hour of hung GPUs.
    const bool nowait = s_dead != 0;
    const unsigned int n = s_seq, par = n & 1u;
    const int n_late4 = 4 * n_units;
    // early element (or loss sum) of this thread: same job numbering as apply_adam_class<false>
    int eidx = -1;
    if (gtid < T.n_early + LOSS_SUMS) {
      if (gtid >= T.n_early) eidx = P + (gtid - T.n_early);
      else {
        int x = gtid, l = 0;
        for (; l < T.nleaves; ++l) {
          if (T.leaf[l].late) continue;
          if (x < T.size[l]) break;
          x -= T.size[l];
        }
        eidx = T.leaf[l].offset + x;
      }
    }
    // Lamport-style exchange: the data is its own flag.  Every staging word holds the sentinel -0.0f until a peer's
    // push lands (a gradient that is exactly -0.0 is sent as +0.0: same sums); the reader polls its own unit of each
    // peer's slot until all four words are real, sums the W contributions in rank order (its own from registers) and
    // puts the sentinel back.  One NVLink one-way latency per exchange: no release/acknowledge round, no flag round.
    // Slot reuse (parity of n) is safe without a fence: a peer can only push exchange n + 2 after it has completed
    // n + 1, which needed this rank's pushes of n + 1, which were issued by a later launch than this one's clears.
    constexpr unsigned int SENT = 0x80000000u;
    auto canon = [](float x) { return x == 0.f ? 0.f : x; };
    auto is_real4 = [](const float4& v) {
      return __float_as_uint(v.x) != SENT && __float_as_uint(v.y) != SENT && __float_as_uint(v.z) != SENT && __float_as_uint(v.w) != SENT;
    };
    const float4 sent4 = make_float4(-0.f, -0.f, -0.f, -0.f);
    float gl = 0.f;
    if (eidx >= 0) {
      // written by the small-leaf CTAs (or, without them, by this thread in phase 2)
      if (has_extra) {
        wait_count(p.done, static_cast<unsigned int>(G - p.gemm_ctas), a.err_flag);
        if (p.trace) atomicMax(&s_waited, static_cast<unsigned long long>(clock64()));
      }
      gl = canon(__ldcg(a.gflat + eidx));
    }
    // TWO-PHASE (X.two_phase, used for W >= 4): the units of warp w of CTA b are reduced by rank (b + w) % W only (dealt per warp,
    // not per CTA: the owner's W - 1 polls and W - 1 result pushes per unit then spread over all SMs).  A non-owner pushes its
    // unit to the owner (one store instead of W - 1) and polls the result slot; the owner polls the W - 1 contributions,
    // sums in rank order and pushes the result to everybody.  Two NVLink latencies instead of one, but (W - 1) / W of a
    // gradient sent and received per rank instead of W - 1 gradients -- and the same sums, bit for bit, as ONE-SHOT.
    const bool two = X.two_phase != 0;
    const int owner = two ? (b + (t >> 5)) % W : R;        // per warp: every CTA holds NT / 32 / W owner warps of each rank
    const bool reduce_here = owner == R;
    // ---- pushes (all units first: every store is in flight before the first poll) ----
#pragma unroll
    for (int u = 0; u < MAXU; ++u) {
      if (ul[u] < 0) continue;
      const int unit = unit0 + u * GT_;
      g4[u].x = canon(g4[u].x); g4[u].y = canon(g4[u].y); g4[u].z = canon(g4[u].z); g4[u].w = canon(g4[u].w);
      if (reduce_here) {
        if (!two) {
#pragma unroll
          for (int r = 0; r < MINPPO_MAX_RANKS; ++r) if (r < W && r != R) st_sys_v4(px_stage(X, r, par, R) + 4 * unit, g4[u]);
        }
      } else {
        st_sys_v4(px_stage(X, owner, par, R) + 4 * unit, g4[u]);
      }
    }
    if (eidx >= 0) {
      if (reduce_here) {
        if (!two) {
#pragma unroll
          for (int r = 0; r < MINPPO_MAX_RANKS; ++r) if (r < W && r != R) st_sys_f32(px_stage(X, r, par, R) + n_late4 + gtid, gl);
        }
      } else {
        st_sys_f32(px_stage(X, owner, par, R) + n_late4 + gtid, gl);
      }
    }
    DW_STAMP(13);
    ss = 0.f;
    const long long t0 = clock64();
#pragma unroll
    for (int u = 0; u < MAXU; ++u) {
      if (ul[u] < 0) continue;
      const int unit = unit0 + u * GT_;
      if (reduce_here) {
        float4 v[MINPPO_MAX_RANKS];
        unsigned int pending = nowait ? 0u : ((1u << W) - 1u) & ~(1u << R);
#pragma unroll
        for (int q = 0; q < MINPPO_MAX_RANKS; ++q) v[q] = g4[u];
        while (pending) {
#pragma unroll
          for (int q = 0; q < MINPPO_MAX_RANKS; ++q) {
            if ((pending >> q) & 1u) {
              v[q] = ld_sys_v4(px_stage(X, R, par, q) + 4 * unit);
              if (is_real4(v[q])) pending &= ~(1u << q);
            }
          }
          if (pending && clock64() - t0 > 8000000000LL) { atomicExch(a.err_flag, MINPPO_ERR_BARRIER); break; }
        }
        const float4 own = g4[u];
        float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int q = 0; q < MINPPO_MAX_RANKS; ++q) {
          if (q < W) {
            const float4 c = q == R ? own : v[q];
            acc.x += c.x; acc.y += c.y; acc.z += c.z; acc.w += c.w;
            if (q != R) st_sys_v4(px_stage(X, R, par, q) + 4 * unit, sent4);
          }
        }
        g4[u] = acc;
        if (two) {
          const float4 res = make_float4(canon(acc.x), canon(acc.y), canon(acc.z), canon(acc.w));
#pragma unroll
          for (int r = 0; r < MINPPO_MAX_RANKS; ++r) if (r < W && r != R) st_sys_v4(px_result(X, r, par) + 4 * unit, res);
        }
      } else {
        float* src = px_result(X, R, par) + 4 * unit;
        float4 v = g4[u];
        while (!nowait) {
          v = ld_sys_v4(src);
          if (is_real4(v)) break;
          if (clock64() - t0 > 8000000000LL) { atomicExch(a.err_flag, MINPPO_ERR_BARRIER); break; }
        }
        g4[u] = v;
        st_sys_v4(src, sent4);
      }
      const float gq[4] = {g4[u].x, g4[u].y, g4[u].z, g4[u].w};
      st_unit(a.gflat + ui[u], gq);
      ss = fmaf(g4[u].x, g4[u].x, ss); ss = fmaf(g4[u].y, g4[u].y, ss); ss = fmaf(g4[u].z, g4[u].z, ss); ss = fmaf(g4[u].w, g4[u].w, ss);
    }
    if (eidx >= 0) {
      float ge = 0.f;
      auto poll1 = [&](float* src, float fallback) {
        unsigned int w = __float_as_uint(fallback);
        while (!nowait && (w = ld_relaxed_sys_u32(reinterpret_cast<const unsigned int*>(src))) == SENT) {
          if (clock64() - t0 > 8000000000LL) { atomicExch(a.err_flag, MINPPO_ERR_BARRIER); break; }
        }
        st_sys_f32(src, -0.f);
        return __uint_as_float(w);
      };
      if (reduce_here) {
        // all W - 1 contributions polled together (one L2 round trip per sweep, not one per rank)
        float ev[MINPPO_MAX_RANKS];
        unsigned int pending = nowait ? 0u : ((1u << W) - 1u) & ~(1u << R);
#pragma unroll
        for (int q = 0; q < MINPPO_MAX_RANKS; ++q) ev[q] = gl;
        while (pending) {
#pragma unroll
          for (int q = 0; q < MINPPO_MAX_RANKS; ++q) {
            if ((pending >> q) & 1u) {
              const unsigned int w = ld_relaxed_sys_u32(reinterpret_cast<const unsigned int*>(px_stage(X, R, par, q) + n_late4 + gtid));
              if (w != SENT) { ev[q] = __uint_as_float(w); pending &= ~(1u << q); }
            }
          }
          if (pending && clock64() - t0 > 8000000000LL) { atomicExch(a.err_flag, MINPPO_ERR_BARRIER); break; }
        }
#pragma unroll
        for (int q = 0; q < MINPPO_MAX_RANKS; ++q) {
          if (q < W) {
            ge += ev[q];
            if (q != R) st_sys_f32(px_stage(X, R, par, q) + n_late4 + gtid, -0.f);
          }
        }
        if (two) {
          const float res = canon(ge);
#pragma unroll
          for (int r = 0; r < MINPPO_MAX_RANKS; ++r) if (r < W && r != R) st_sys_f32(px_result(X, r, par) + n_late4 + gtid, res);
        }
      } else {
        ge = poll1(px_result(X, R, par) + n_late4 + gtid, gl);
      }
      a.gflat[eidx] = ge;                                // read back by this same thread (small leaves) / after the barrier (losses)
      if (eidx < P) ss = fmaf(ge, ge, ss);
    }
    DW_STAMP(15);
    if (b == 0 && scal_thread) *X.seq = n;
  }
  const float bs = block_sum_dyn(ss, scratch);           // (its CTA barriers also order the s_waited updates)
  if (t == 0) a.block_ss[b] = bs;
  // trace slot 2: this CTA's last counter wait satisfied (the end of phase 1 if it had none)
  if (p.trace && t == 0) p.trace[static_cast<size_t>(b) * 16 + 2] = max(static_cast<long long>(s_waited), p.trace[static_cast<size_t>(b) * 16 + 1]);
  DW_STAMP(3);
  grid_barrier(a.barrier, a.err_flag);
  DW_STAMP(4);
  // every counter wait of this launch is behind the barrier: back to zero for the next launch
  if (b == 0 && t <= p.gemm_ctas / static_cast<int>(S)) p.done[t * DWOPT_DONE_STRIDE] = 0u;
  if (!a.do_apply) return;                               // NCCL fallback: gflat = the local gradient sum; applied by a later launch

  // ---- phase 3 ----------------------------------------------------------------------------------
  // This thread's element of the SMALL leaves (at most one when they fit one sweep of the grid): gradient and optimizer state
  // are requested first, so that the L2 round trip runs under the norm reduction and the register-resident units below --
  // the launch ends with its slowest CTA, and the CTAs that carry the small leaves are those (phase 3: 4.4k cycles mean,
  // 8.8k on them).  Same job numbering and the same arithmetic as apply_adam_class<false>.
  const bool early_one = fast && !px_on && T.n_early <= GT_;   // (sharded ranks keep the loop below: measured at 2 / 8 ranks as is)
  int el = -1, ei = 0;
  float eg = 0.f, ep = 0.f, em = 0.f, en = 0.f;
  if (early_one && gtid < T.n_early) {
    int x = gtid, l = 0;
    for (; l < T.nleaves; ++l) {
      if (T.leaf[l].late) continue;
      if (x < T.size[l]) break;
      x -= T.size[l];
    }
    el = l; ei = T.leaf[l].offset + x;
    eg = __ldcg(a.gflat + ei); ep = __ldcg(a.params + ei); em = __ldcg(a.mu + ei); en = __ldcg(a.nu + ei);
  }
  {
    // one load per thread (G <= DWOPT_THREADS): a serial loop over the per-block sums cost five dependent
    // L2 round trips on lines every SM is hammering at the same time
    const float v = t < G ? __ldcg(a.block_ss + t) : 0.f;
    const float tot = block_sum_dyn(v, scratch);
    if (t == 0) s_bcast[0] = sqrtf(tot);
  }
  __syncthreads();
  AdamScalars sc;
  sc.gnorm = s_bcast[0]; sc.lr = s_bcast[1]; sc.c1 = s_bcast[2]; sc.c2 = s_bcast[3];
  sc.trigger = sc.gnorm < a.max_norm;                    // optax.clip_by_global_norm
  if (fast) {
#pragma unroll
    for (int u = 0; u < MAXU; ++u) {
      if (ul[u] < 0) continue;
      const OptLeaf& L = T.leaf[ul[u]];
      const float gv[4] = {g4[u].x, g4[u].y, g4[u].z, g4[u].w};
#pragma unroll
      for (int e = 0; e < 4; ++e) adam_element(a, sc, gv[e], pv[u][e], mv[u][e], nv[u][e]);
      st_unit(a.params + ui[u], pv[u]); st_unit(a.mu + ui[u], mv[u]); st_unit(a.nu + ui[u], nv[u]);
      if (L.img_n)             // 4 consecutive bf16 of the kernel image (unit index is a multiple of 4: 8-byte aligned)
        *reinterpret_cast<uint2*>(L.img_n + (ui[u] - L.offset)) = make_uint2(pack_bf16x2(pv[u][0], pv[u][1]), pack_bf16x2(pv[u][2], pv[u][3]));
    }
    if (early_one) {
      if (el >= 0) {
        adam_element(a, sc, eg, ep, em, en);
        a.params[ei] = ep; a.mu[ei] = em; a.nu[ei] = en;
        write_images(T.leaf[el], ei, ep);
      }
    } else {
      apply_adam_class<false>(a, T, sc, gtid, GT_);
    }
  } else {
    apply_adam(a, T, sc, gtid, GT_);
  }
  __syncthreads();
  DW_STAMP(5);
  if (b == 0 && scal_thread) {
    *a.count = count + 1;
    if (losses_out) {
      // gflat[P] = sum max(vl, vlc), gflat[P+1] = sum min(l1, l2) over the global minibatch
      const float value_loss = 0.5f * __ldcg(a.gflat + P) * a.inv_mb;
      const float actor_loss = -__ldcg(a.gflat + P + 1) * a.inv_mb;
      // a raised device-side error flag (row-list overflow, barrier / exchange timeout) poisons the reported losses:
      // the failure surfaces in the update's own result without a host round trip (minppo_ctx_check names the cause)
      const float poison = __ldcg(a.err_flag) != 0 ? __int_as_float(0x7fc00000) : 0.f;
      losses_out[0] = actor_loss + a.vf_coef * value_loss - a.ent_coef * ent + poison;
      losses_out[1] = value_loss + poison;
      losses_out[2] = actor_loss + poison;
      losses_out[3] = ent + poison;
      if (gnorm_out) *gnorm_out = sc.gnorm;
      if (a.stats_out) {
        // gflat[P+2] = value-clip count, gflat[P+3] = approx-KL sum, gflat[P+4] = ratio-clip count (LOSS_SUMS).  The
        // address is formed here, from the kernel parameters: a pointer live across the kernel adds to dwopt_kernel<4>'s spills
        float* stats_out = a.stats_out + static_cast<size_t>(p.step) * 4;
        stats_out[0] = __ldcg(a.gflat + P + 3) * a.inv_mb + poison;
        stats_out[1] = __ldcg(a.gflat + P + 4) * a.inv_mb + poison;
        stats_out[2] = __ldcg(a.gflat + P + 2) * a.inv_mb + poison;
        stats_out[3] = sc.gnorm + poison;
      }
    }
  }
}

// largest parameter count of the hidden kernels the register-resident fast path covers on a grid of `grid` CTAs
inline long long dwopt_fast_capacity(int grid, int maxu) { return 4LL * grid * DWOPT_THREADS * maxu; }

inline cudaError_t dwopt_launch(const DwOptParams& p, int grid, cudaStream_t stream, bool pdl, int maxu) {
  if (maxu <= 1) return launch_kernel(dwopt_kernel<1>, grid, DWOPT_THREADS, GEMM_SMEM_BYTES, stream, pdl, p);
  if (maxu == 2) return launch_kernel(dwopt_kernel<2>, grid, DWOPT_THREADS, GEMM_SMEM_BYTES, stream, pdl, p);
  return launch_kernel(dwopt_kernel<4>, grid, DWOPT_THREADS, GEMM_SMEM_BYTES, stream, pdl, p);
}

}  // namespace minppo
