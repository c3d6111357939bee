// minppo_b200 -- fused minibatch forward + PPO loss + backward-to-dZ for the 2-hidden-layer nets
// (the reference's default model.num_layers = 2, /root/reference/minppo/config.py:53).
//
// One CTA = one 128-row tile of the minibatch x one net (actor or critic).  Everything between
// the gathered observation rows and the layer gradients dZ stays on chip; every contraction runs
// on the tcgen05 tensor cores with accumulators in TMEM:
//
//   gather X k-blocks (cp.async by row index, SW128) -> 4 slots in R1 (streamed for obs_dim > 256)
//   L1   acc0 = X  W0    (W0 half-k-blocks streamed by TMA)     -> +b0, act, bf16 -> R0 (H1) -> TMA store
//   L2   acc1 = H1 W1                                           -> +b1, act, bf16 -> R1 (H2)
//   head out  = H2 W2    (N = 2 AP: bf16 hi | lo; in acc0, per k-block of epilogue 2) -> +b2 -> Gaussian log-prob / clipped
//        surrogate (actor CTA) or clipped value loss (critic CTA), train.py:218-243 -> g = dL/dout
//   bwd  dA2  = g W2^T   (K = AP),  dW2 = H2^T g (N = 2 AP)     -> dZ2 = dA2 * f'(H2) in place -> TMA store
//   dH1  acc1 = dZ2 W1^T (two N halves)                         -> * f'(H1), bf16 -> R0 (dZ1, over H1) -> TMA store
//   bias gradients: column sums of dZ2 / dZ1 as dZ^T x ones (N = 16) MMAs -> per-tile partials
//
// The output-head operands W2 and g are fp32 quantities: they enter the tensor cores as a bf16
// hi/lo pair (x = hi + lo to 2^-17), the cross terms hi*hi + hi*lo + lo*hi are accumulated in
// fp32, so the heads keep fp32-level accuracy while costing a few dozen tiny UMMAs.
//
// Shapes: any obs_dim (Dp = ceil(D / 64) * 64 columns, k-blocks streamed through 4 slots), act_dim <= 32
// (template AP = 16 or 32: padded head width), hidden_size a multiple of 64 up to 256 (two 128 x 256 fp32
// accumulators fill the 512 TMEM columns; 512-wide layers would need N-halved accumulators and are refused).
//
// Warp roles: warps 0..15 workers (gather, epilogues, loss), FOUR per TMEM lane quadrant -- a worker warp owns 16 of every
// 64 accumulator columns, so each scheduler has four epilogue warps to hide the tcgen05.ld / MUFU / st.shared latencies
// behind; warp 16 TMA producer (weight stages of 16 KB through a ring); warp 17 TMEM allocator + MMA issuer.
// H1, dZ2, dZ1 and (critic CTA) the gathered X rows are also written to HBM (bf16, TMA stores) for the split-K
// weight-gradient GEMM (dwopt.cuh), which runs as its own launch over all tiles.
//
// Scheduling rules this kernel follows (each one measured, DESIGN.md 3.4): global accesses with many lines per instruction
// (row gathers of the loss inputs, per-row partial stores) stay out of the epilogues -- issued by the warps that are done,
// they stall the shared-memory traffic of the warp that is not: the loss inputs are requested before griddepcontrol.wait,
// the head-kernel gradient leaves through shared memory and one bulk copy; the TMA unit is a FIFO whose stores drain at
// ~32 B/clk, so no store is queued in front of a weight load the MMAs are about to wait for.
#pragma once

#include "common.cuh"
#include "minppo_internal.h"
#include "ppo_math.cuh"
#include "umma_gemm.cuh"

namespace minppo {

constexpr int FS_THREADS = 576;
constexpr int FS_WORKERS = 512;                         // warps 0..15
constexpr int FS_NWW = 16;
constexpr int FS_TMA_WARP = 16;                         // weight producer
constexpr int FS_MMA_WARP = 17;                         // TMEM allocator + MMA issuer: the highest warp id wins the
                                                        // issue arbiter, so the single issuing thread is never starved
constexpr int FS_STAGE = 16384;                         // one weight stage: [32 k][H n] (forward, MN-major B: H/64 boxes of 4 KB)
                                                        // or [H/2 n][64 k] (dH1, K-major B)
constexpr int FS_XSLOTS = 4;                            // X k-block slots in R1 (16 KB each)
constexpr int FS_MAX_AP = 32;
constexpr int FS_STORE_THREAD = 480;                    // warp 15 lane 0 issues the H1 / dZ2 / dZ1 TMA stores: the highest-priority worker
                                                        // warp of a scheduler that hosts neither the TMA nor the MMA warp (a low-priority
                                                        // warp that starts an epilogue late finishes it last: measured +2k cycles on warp 1)

template <int AP>
struct FsLayout {
  static constexpr int NS = AP == 16 ? 4 : 2;           // ring stages (L2 / dH1 weight streams)
  static constexpr int NS1 = NS + 4;                    // L1 only: four more stages parked in R0 (free until epilogue 1)
  static constexpr int PG = 2 * AP * 128;               // bytes of one 64-column panel of W2T / GT: [2 AP rows][128 B], rows = hi | lo
  static constexpr int R0 = 0;                          // H1 / dZ1            64 KB
  static constexpr int R1 = 65536;                      // X / H2 / dZ2        64 KB
  static constexpr int RB = 131072;                     // weight ring
  static constexpr int W2T = RB + NS * FS_STAGE;        // head kernel^T bf16 hi / lo, SW128, 4 panels (H <= 256)
  static constexpr int GT = W2T + 4 * PG;               // g^T bf16 hi / lo, SW128, 2 panels (128 rows)
  static constexpr int ONES = GT + 2 * PG;              // all-ones bf16 [16 n][128 k] (K-major B of the bias-gradient MMAs)
  static constexpr int BIAS = ONES + 4096;              // [2][256] f32
  static constexpr int HB = BIAS + 2048;                // f32: head bias [AP], log_std [AP], 1/scale [AP], log-det [1]
  static constexpr int RS = 2 * AP + 8;                 // floats per loss warp in RED
  static constexpr int RED = HB + 512;                  // [4][RS] f32
  static constexpr int BARS = RED + 4 * RS * 4;         // mbarriers + tmem slot
  static constexpr int BYTES = BARS + 512 + 1024;       // + alignment slack
};
static_assert(FsLayout<16>::BYTES <= 232448 && FsLayout<32>::BYTES <= 232448, "fused step: shared memory budget");

struct alignas(64) FusedNet {
  CUtensorMap tm_w0;             // W0 image [Dp][H] (as stored: [in][out])  box {64 out, 32 in}: MN-major B of L1
  CUtensorMap tm_w1;             // W1 image [H][H]                          box {64 out, 32 in}: MN-major B of L2
  CUtensorMap tm_w1k;            // W1 image [H][H]                          box {64 out, H/2 in}: K-major B of dH1 (n = in, k = out)
  CUtensorMap tm_h1;             // act[1] [M_pad][H]    box {64, 128}  (TMA store)
  CUtensorMap tm_dz2;            // dz[2]
  CUtensorMap tm_dz1;            // dz[1]
  const float* b0;               // arena pointers
  const float* b1;
  const uint4* w2img;            // head kernel^T as bf16 hi / lo, the shared-memory image of FsLayout::W2T (written by the optimizer)
  const float* b2;               // head bias [aout]
  int act;                       // ACT_*
  int aout;                      // A (actor) or 1 (critic)
  int po_w2, po_b2, po_loss;     // offsets of this net's fields inside a per-tile partial
  int po_stat;                   // ... this net's statistics sums (LOSS_SUMS): actor 2 (KL, ratio clips), critic 1 (value clips)
  int po_db0, po_db1;            // ... hidden bias gradients (column sums of dZ1 / dZ2), H floats each
};

struct alignas(64) FusedParams {
  FusedNet net[2];
  CUtensorMap tm_xg;             // gathered observation rows [M_pad][Dp], box {64, 128}: TMA store by the critic CTAs,
                                 // the A operand of both nets' first-layer weight-gradient GEMM
  // (obs_img ahead of loss keeps the pointer pairs the compiler fetches with one 16-byte constant load, and the kernel's code)
  const __nv_bfloat16* obs_img;  // [Bl][Dp]
  LossOperands loss;             // its row lists also gather the observation rows
  const float* log_std;          // arena pointer
  float* part;                   // per-tile partials [m_tiles][part_stride]
  int part_stride, po_logstd;
  int H, A, Dp, m_tiles;
  long long* trace;              // debug: [ctas][32] clock64 stamps (null = off)
};

constexpr int FS_TRACE_SLOTS = 256;                     // clock64 stamps per unit: [0, 32) one thread per role, [64, 84) the MMA issuer
                                                        // inside the dH1 GEMM (k-block seen / stage landed / MMAs issued), [128, 256) every
                                                        // worker warp around the four big epilogues (128 + 32 e + warp: start, + 16: end)
#define FS_STAMP(slot) do { if (p.trace) p.trace[static_cast<size_t>(cta_id) * FS_TRACE_SLOTS + (slot)] = clock64(); } while (0)
#define FS_STAMP_W(e, end) do { if (p.trace && lane == 0) p.trace[static_cast<size_t>(cta_id) * FS_TRACE_SLOTS + 128 + 32 * (e) + 16 * (end) + warp] = clock64(); } while (0)

MINPPO_DEVINL void worker_bar() { asm volatile("bar.sync 1, 512;" ::: "memory"); }

MINPPO_DEVINL void sts_u16(uint32_t addr, uint32_t v) {
  asm volatile("st.shared.u16 [%0], %1;" ::"r"(addr), "h"(static_cast<uint16_t>(v)) : "memory");
}
// TMEM -> registers: 32 lanes x 16 consecutive fp32 columns
MINPPO_DEVINL void tmem_ld_32x16(uint32_t taddr, float (&v)[16]) {
  uint32_t* r = reinterpret_cast<uint32_t*>(v);
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
// TMEM -> registers: 32 lanes x 4 / 8 consecutive fp32 columns (the loss: a worker warp owns AP / 4 head columns)
MINPPO_DEVINL void tmem_ld_32xn(uint32_t taddr, float (&v)[4]) {
  uint32_t* r = reinterpret_cast<uint32_t*>(v);
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0, %1, %2, %3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(taddr) : "memory");
}
MINPPO_DEVINL void tmem_ld_32xn(uint32_t taddr, float (&v)[8]) {
  uint32_t* r = reinterpret_cast<uint32_t*>(v);
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "r"(taddr) : "memory");
}
// N x 32 transpose-reduce (N = 8, 16): lane l ends with the sum over the 32 lanes of v[l & (N - 1)]
template <int N>
MINPPO_DEVINL float warp_colsum_n(float (&v)[N]) {
  const uint32_t lane = lane_id();
#pragma unroll
  for (int half = N / 2; half >= 1; half >>= 1) {
    const bool upper = (lane & half) != 0;
#pragma unroll
    for (int i = 0; i < half; ++i) {
      const float keep = upper ? v[i + half] : v[i];
      const float send = upper ? v[i] : v[i + half];
      v[i] = keep + __shfl_xor_sync(0xffffffffu, send, half);
    }
  }
  float r = v[0];
#pragma unroll
  for (int o = N; o < 32; o <<= 1) r += __shfl_xor_sync(0xffffffffu, r, o);
  return r;
}
// TMEM -> registers: 32 lanes x 1 column
MINPPO_DEVINL float tmem_ld_32x1(uint32_t taddr) {
  uint32_t r;
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x1.b32 {%0}, [%1];" : "=r"(r) : "r"(taddr) : "memory");
  return __uint_as_float(r);
}
// byte offset of the 16-byte chunk holding column c of row r inside a [128][H] bf16 SW128 tile set
MINPPO_DEVINL uint32_t sw_off(int r, int c) {
  return static_cast<uint32_t>((c >> 6) * 16384 + r * 128 + ((((c & 63) >> 3) ^ (r & 7)) << 4));
}
// cp.async.wait_group with a run-time bound (waiting for fewer pending groups than allowed is always safe)
MINPPO_DEVINL void cp_async_wait_dyn(int n) {
  if (n <= 0) cp_async_wait<0>();
  else if (n == 1) cp_async_wait<1>();
  else if (n == 2) cp_async_wait<2>();
  else if (n == 3) cp_async_wait<3>();
  else cp_async_wait<4>();
}
template <int ACT>
MINPPO_DEVINL float act_apply(float x) {
  if (ACT == ACT_RELU) return fmaxf(x, 0.f);
  if (ACT == ACT_TANH_FAST) return fast_tanh(x);
  return exp_tanh(x);
}
template <int ACT>
MINPPO_DEVINL float act_deriv_t(float h) { return ACT == ACT_RELU ? (h > 0.f ? 1.f : 0.f) : (1.f - h * h); }
// The four epilogues walk `nchunks` 16-column chunks of an accumulator, chunk i at column col0 + i * cstride, and (bars != null)
// publish chunk i on bars[i] as soon as it is in shared memory.  The TMEM read of chunk i + 1 is issued before chunk i is
// processed (one tcgen05.ld outstanding at every tcgen05.wait::ld): with four warps per scheduler the read latency is
// otherwise exposed in every chunk, and the MUFU time of a tanh chunk (16 x 8 cycles per warp) adds to it instead of hiding it.
// (Not inlined: the epilogues share one copy of the code per activation -- the kernel's straight-line worker path is larger
//  than the instruction cache otherwise.)
// (Publishing the 64-column blocks in pairs where no GEMM is fed block by block -- epilogues 2 and 3 -- saves two of the four
//  generic -> async proxy fences per warp, ~130 cycles each in isolation, but measured no faster in the kernel: 5.287 vs 5.263 ms.)
MINPPO_DEVINL void chunk_publish(uint64_t* bar) {
  fence_proxy_async_smem();
  tc_fence_before();
  __syncwarp();
  if (lane_id() == 0) mbar_arrive(bar);
}
// one chunk: +bias, activation, bf16 -> swizzled smem tile
template <int ACT>
MINPPO_DEVINL void act_chunk(const float (&v)[16], uint32_t dst_base, const float* bias_s, int row, int c0) {
  const float4* b4 = reinterpret_cast<const float4*>(bias_s + c0);     // broadcast LDS.128
  float4 bb[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) bb[j] = b4[j];
#pragma unroll
  for (int j = 0; j < 2; ++j) {
    uint32_t w[4];
    const float bj[8] = {bb[2 * j].x, bb[2 * j].y, bb[2 * j].z, bb[2 * j].w,
                         bb[2 * j + 1].x, bb[2 * j + 1].y, bb[2 * j + 1].z, bb[2 * j + 1].w};
#pragma unroll
    for (int t = 0; t < 4; ++t) {
      const int e = 8 * j + 2 * t;
      const float x0 = act_apply<ACT>(v[e] + bj[2 * t]);
      const float x1 = act_apply<ACT>(v[e + 1] + bj[2 * t + 1]);
      w[t] = pack_bf16x2(x0, x1);
    }
    sts128(dst_base + sw_off(row, c0 + 8 * j), make_uint4(w[0], w[1], w[2], w[3]));
  }
}
template <int ACT>
__device__ __noinline__ void epilogue_act_t(uint32_t tmem_acc, uint32_t dst_base, const float* bias_s, int row, int q, int col0,
                                            int cstride, int nchunks, uint64_t* bars) {
  const uint32_t taddr = tmem_acc + (static_cast<uint32_t>(q * 32) << 16);
  float va[16], vb[16];
  tmem_ld_32x16(taddr + col0, va);
  for (int i = 0; i < nchunks; i += 2) {
    const int c0 = col0 + i * cstride;
    tmem_ld_wait();
    tmem_ld_32x16(taddr + (i + 1 < nchunks ? c0 + cstride : c0), vb);          // branch-free: the last chunk re-reads itself
    __syncwarp();
    act_chunk<ACT>(va, dst_base, bias_s, row, c0);
    if (bars) chunk_publish(bars + i);
    if (i + 1 < nchunks) {
      tmem_ld_wait();
      tmem_ld_32x16(taddr + (i + 2 < nchunks ? c0 + 2 * cstride : c0), va);
      __syncwarp();
      act_chunk<ACT>(vb, dst_base, bias_s, row, c0 + cstride);
      if (bars) chunk_publish(bars + i + 1);
    }
  }
  tmem_ld_wait();                                                  // the trailing read must have landed before the registers are reused
}
MINPPO_DEVINL void epilogue_act(uint32_t tmem_acc, uint32_t dst_base, const float* bias_s, int act, int row, int q,
                                int col0, int cstride, int nchunks, uint64_t* bars) {
  if (act == ACT_RELU) epilogue_act_t<ACT_RELU>(tmem_acc, dst_base, bias_s, row, q, col0, cstride, nchunks, bars);
  else if (act == ACT_TANH_FAST) epilogue_act_t<ACT_TANH_FAST>(tmem_acc, dst_base, bias_s, row, q, col0, cstride, nchunks, bars);
  else epilogue_act_t<ACT_TANH>(tmem_acc, dst_base, bias_s, row, q, col0, cstride, nchunks, bars);
}

// dZ = acc * f'(h): h read from `h_base`, bf16 result written to `dst_base` (may alias h_base:
// every thread touches only its own 16-byte chunks).  The bias gradients (column sums of dZ) are
// not formed here: they come from the tensor core as dZ^T x ones.
template <int ACT>
MINPPO_DEVINL void dact_chunk(const float (&v)[16], uint32_t h_base, uint32_t dst_base, int row, int c0) {
  uint4 hh[2];
#pragma unroll
  for (int j = 0; j < 2; ++j) hh[j] = lds128(h_base + sw_off(row, c0 + 8 * j));
#pragma unroll
  for (int j = 0; j < 2; ++j) {
    const uint32_t hw[4] = {hh[j].x, hh[j].y, hh[j].z, hh[j].w};
    uint32_t w[4];
#pragma unroll
    for (int t = 0; t < 4; ++t) {
      const int e = 8 * j + 2 * t;
      w[t] = pack_bf16x2(v[e] * act_deriv_t<ACT>(bf16_lo(hw[t])), v[e + 1] * act_deriv_t<ACT>(bf16_hi(hw[t])));
    }
    sts128(dst_base + sw_off(row, c0 + 8 * j), make_uint4(w[0], w[1], w[2], w[3]));
  }
}
template <int ACT>
__device__ __noinline__ void epilogue_dact_t(uint32_t tmem_acc, uint32_t h_base, uint32_t dst_base, int row, int q, int col0,
                                             int cstride, int nchunks, uint64_t* bars) {
  const uint32_t taddr = tmem_acc + (static_cast<uint32_t>(q * 32) << 16);
  float va[16], vb[16];
  tmem_ld_32x16(taddr + col0, va);
  for (int i = 0; i < nchunks; i += 2) {
    const int c0 = col0 + i * cstride;
    tmem_ld_wait();
    tmem_ld_32x16(taddr + (i + 1 < nchunks ? c0 + cstride : c0), vb);          // branch-free: the last chunk re-reads itself
    __syncwarp();
    dact_chunk<ACT>(va, h_base, dst_base, row, c0);
    if (bars) chunk_publish(bars + i);
    if (i + 1 < nchunks) {
      tmem_ld_wait();
      tmem_ld_32x16(taddr + (i + 2 < nchunks ? c0 + 2 * cstride : c0), va);
      __syncwarp();
      dact_chunk<ACT>(vb, h_base, dst_base, row, c0 + cstride);
      if (bars) chunk_publish(bars + i + 1);
    }
  }
  tmem_ld_wait();                                                  // the trailing read must have landed before the registers are reused
}
MINPPO_DEVINL void epilogue_dact(uint32_t tmem_acc, uint32_t h_base, uint32_t dst_base, int act, int row, int q,
                                 int col0, int cstride, int nchunks, uint64_t* bars) {
  if (act == ACT_RELU) epilogue_dact_t<ACT_RELU>(tmem_acc, h_base, dst_base, row, q, col0, cstride, nchunks, bars);
  else epilogue_dact_t<ACT_TANH>(tmem_acc, h_base, dst_base, row, q, col0, cstride, nchunks, bars);
}

// One (tile, net) unit of one minibatch step.  The whole CTA (FS_THREADS threads) calls this with the SAME arguments;
// `sm` / `base` = the 1024-byte aligned dynamic shared memory, `tmem_base` = 512 allocated TMEM columns.
template <int AP>
MINPPO_DEVINL void fused_tile(const FusedParams& p, int unit, int step, uint8_t* sm, uint32_t base, uint32_t tmem_base) {
  using LY = FsLayout<AP>;
  constexpr int NS = LY::NS, NS1 = LY::NS1, PG = LY::PG, RS = LY::RS;
  float* bias_s = reinterpret_cast<float*>(sm + LY::BIAS);      // [0..256) layer 0, [256..512) layer 1
  float* hb = reinterpret_cast<float*>(sm + LY::HB);            // [0, AP) head bias, [AP, 2AP) log_std,
                                                                // [2AP, 3AP) 1 / scale, [3AP] sum log|scale|
  float* red = reinterpret_cast<float*>(sm + LY::RED);
  float* qp = bias_s;                                           // [4 column groups][128 rows] partial quadratic forms of the actor loss:
                                                                // aliases the hidden biases, dead once every warp is past epilogue 2 (headf)
  uint64_t* bars = reinterpret_cast<uint64_t*>(sm + LY::BARS);
  uint64_t* l1_full = bars;             // [8] W0 half-k-block landed (TMA)
  uint64_t* l1_empty = bars + 8;        // [8] ... consumed (MMA commit)
  uint64_t* x_full = bars + 16;         // [4] X k-block gathered (16 worker warps)
  uint64_t* x_empty = bars + 20;        // [4] ... consumed (MMA commit)
  uint64_t* full_bar = bars + 24;       // [4] ring stage landed
  uint64_t* empty_bar = bars + 28;      // [4] ring stage consumed
  uint64_t* accf0 = bars + 32;          // L1 accumulator complete
  uint64_t* accf1 = bars + 33;          // L2 accumulator complete
  uint64_t* headf = bars + 34;          // head outputs complete
  uint64_t* bwdf = bars + 35;           // dA2 and dW2 complete
  uint64_t* dh1f = bars + 36;           // dH1 accumulator complete
  uint64_t* cs2f = bars + 37;           // column sums of dZ2 complete
  uint64_t* cs1f = bars + 38;           // column sums of dZ1 complete
  uint64_t* h2r = bars + 57;            // [4] H2 columns [64 b, 64 b + 64) in R1 (k-block b of the head GEMM); all: acc1 drained
  uint64_t* ldi = bars + 39;            // the TMA producer has issued its last weight load
  uint64_t* gr = bars + 40;             // g^T hi/lo written
  uint64_t* h1r = bars + 41;            // [4] H1 columns [64 b, 64 b + 64) in R0 (k-block b of the L2 GEMM)
  uint64_t* dz2r = bars + 45;           // [4] dZ2 columns [64 b, 64 b + 64) in R1 (k-block b of the dH1 GEMM)
  uint64_t* dz1r = bars + 49;           // [4] dZ1 columns [64 b, 64 b + 64) in R1
  uint64_t* x_stored = bars + 53;       // [4] the TMA store of the X k-block in slot s (for the dW GEMM) has read the slot
  const LossOperands& L = p.loss;
  const int32_t* rowidx_s = L.rowidx + static_cast<size_t>(step) * L.cap;   // this step's row list
  const int32_t* count_s = L.count + step;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // CTA order: (tile, net) with net fastest, so that the LIVE tiles of both nets are the lowest block indices and fit the
  // first wave even when the grid is sized for an env-sharded rank's worst-case row count (dead tiles come last)
  const int net = unit & 1;
  const int tile = unit >> 1;
  const int cta_id = net * p.m_tiles + tile;             // trace row (net-major, scripts/trace_fused.py)
  const FusedNet& G = p.net[net];
  const int H = p.H, nkH = H >> 6, nk0 = p.Dp >> 6;
  const int mtH = (H + 127) >> 7;                        // 128-column tiles of a hidden layer
  const uint32_t R0 = base + LY::R0, R1 = base + LY::R1, RB = base + LY::RB;
  const uint32_t W2T = base + LY::W2T, GT = base + LY::GT, ONES = base + LY::ONES;
  auto l1_stage = [&](int s) -> uint32_t { return s < NS ? RB + s * FS_STAGE : R0 + (s - NS) * FS_STAGE; };

  // Env-sharded ranks size the row lists for the worst case (learner.cu: 1.5 x the mean + 256 rows); the tiles
  // beyond this minibatch's actual row count have nothing to do except zeroing their partial sums.
  if (tile * 128 >= min(*count_s, L.cap)) {
    griddep_wait();                                     // the previous optimizer step may still be reading the partials
    float* part = p.part + static_cast<size_t>(tile) * p.part_stride;
    for (int i = threadIdx.x; i < H * G.aout; i += FS_THREADS) part[G.po_w2 + i] = 0.f;
    for (int i = threadIdx.x; i < H; i += FS_THREADS) { part[G.po_db0 + i] = 0.f; part[G.po_db1 + i] = 0.f; }
    if (static_cast<int>(threadIdx.x) < G.aout) part[G.po_b2 + threadIdx.x] = 0.f;
    if (net == 0 && static_cast<int>(threadIdx.x) < G.aout) part[p.po_logstd + threadIdx.x] = 0.f;
    if (threadIdx.x == 0) part[G.po_loss] = 0.f;
    if (static_cast<int>(threadIdx.x) < (net == 0 ? 2 : 1)) part[G.po_stat + threadIdx.x] = 0.f;
    return;
  }
  __syncthreads();
  if (threadIdx.x == FS_WORKERS) {
    FS_STAMP(16);
    // tensor maps into the descriptor cache first (weights: in front of the first L1 stage; stores: off any critical path)
    tma_prefetch_desc(&G.tm_w0); tma_prefetch_desc(&G.tm_w1); tma_prefetch_desc(&G.tm_w1k);
    tma_prefetch_desc(&G.tm_h1); tma_prefetch_desc(&G.tm_dz2); tma_prefetch_desc(&G.tm_dz1);
    if (net == 1) tma_prefetch_desc(&p.tm_xg);
    for (int s = 0; s < 8; ++s) { mbar_init(&l1_full[s], 1); mbar_init(&l1_empty[s], 1); }
    for (int s = 0; s < 4; ++s) {
      mbar_init(&x_full[s], FS_NWW); mbar_init(&x_empty[s], 1); mbar_init(&x_stored[s], 1);
      mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1);
      mbar_init(&h1r[s], FS_NWW); mbar_init(&h2r[s], FS_NWW); mbar_init(&dz2r[s], FS_NWW); mbar_init(&dz1r[s], FS_NWW);
    }
    mbar_init(accf0, 1); mbar_init(accf1, 1); mbar_init(headf, 1); mbar_init(bwdf, 1); mbar_init(dh1f, 1);
    mbar_init(cs2f, 1); mbar_init(cs1f, 1);
    mbar_init(gr, FS_NWW); mbar_init(ldi, 1);
    fence_mbar_init();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t acc0 = tmem_base, acc1 = tmem_base + 256;
  const uint32_t acc_head = acc0;               // [0, 2AP): head outputs, hi | lo halves (acc0 is free between epilogue 1 and dA2: the head
                                                // MMAs of k-block b run while epilogue 2 still drains acc1 for the later blocks)
  const uint32_t acc_dw = acc1 + 2 * AP;        // + 2AP per 128-column tile of H: head-kernel gradient, hi | lo halves
  const uint32_t acc_cs2 = acc0;                // + 16 per 128-column tile: column sums of dZ2 (after acc0 = dA2 is drained)
  const uint32_t acc_cs1 = acc0 + 32;           // + 16 per 128-column tile: column sums of dZ1

  if (warp == FS_TMA_WARP) {
    // ===================== weight producer ======================================================================
    if (elect_one()) {
      griddep_wait();                 // the weight images are rewritten by the previous optimizer step
      const uint32_t bytes = static_cast<uint32_t>(H) * 64u;
      // ---- L1: W0 half-k-blocks j = 0 .. 2 nk0 - 1 through NS1 stages (the ring + four stages parked in R0, which nothing
      //      touches before epilogue 1: for Dp <= 256 the whole L1 GEMM is fed up front)
      const int n1 = 2 * nk0;
      for (int j = 0; j < n1; ++j) {
        const int s = j % NS1;
        if (j >= NS1) mbar_wait(&l1_empty[s], ((j / NS1) - 1) & 1);
        mbar_arrive_expect_tx(&l1_full[s], bytes);
        const uint32_t dst = l1_stage(s);
        for (int c = 0; c < nkH; ++c) tma_load_2d(dst + c * 4096, &G.tm_w0, &l1_full[s], c * 64, j * 32);
      }
      // ---- ring: W1 half-k-blocks of L2 (MN-major), then W1 (k-block, N half) items of dH1 (K-major)
      const int n2 = 2 * nkH, total = 4 * nkH;
      for (int i = 0; i < total; ++i) {
        const int s = i % NS;
        if (i < NS) {
          // first pass over the ring: stage s may still hold a W0 half-k-block -- wait for L1's LAST use of it
          int jl = -1;
          for (int j = s; j < n1; j += NS1) jl = j;
          if (jl >= 0) mbar_wait(&l1_empty[s], (jl / NS1) & 1);
        } else {
          mbar_wait(&empty_bar[s], ((i / NS) - 1) & 1);
        }
        mbar_arrive_expect_tx(&full_bar[s], bytes);
        const uint32_t dst = RB + s * FS_STAGE;
        if (i < n2) {
          for (int c = 0; c < nkH; ++c) tma_load_2d(dst + c * 4096, &G.tm_w1, &full_bar[s], c * 64, i * 32);
        } else {
          const int ii = i - n2;
          tma_load_2d(dst, &G.tm_w1k, &full_bar[s], (ii >> 1) * 64, (ii & 1) * (H >> 1));
        }
        if (i == total - 1) mbar_arrive(ldi);
      }
    }
  } else if (warp == FS_MMA_WARP) {
    // ===================== MMA issuer ===========================================================================
    if (elect_one()) {
      const uint32_t idesc_bmn = umma_idesc_bf16(128, static_cast<uint32_t>(H), 0u, 1u);     // B as stored: MN-major
      FS_STAMP(17);
      // ---- L1: acc0 = X W0 -------------------------------------------------------------------------------------
      for (int kb = 0; kb < nk0; ++kb) {
        const int xs = kb & 3;
        mbar_wait_spin(&x_full[xs], (kb >> 2) & 1);
        if (kb == 0) FS_STAMP(18);
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
      FS_STAMP(19);
      // ---- L2: acc1 = H1 W1; the A k-blocks are published by epilogue 1 in 64-column blocks ---------------------------
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
      FS_STAMP(21);
      // ---- head forward: [out_hi | out_lo][128 x 2AP] = H2 [W2_hi | W2_lo]; A = H2 K-major, B = W2T K-major with the
      //      bf16 hi / lo halves stacked along N (the workers add the two halves); k-block b as soon as epilogue 2 has
      //      published it
      {
        const uint32_t idesc_h = umma_idesc_bf16(128, 2u * AP, 0u, 0u);
        uint32_t accum = 0;
        for (int kb = 0; kb < nkH; ++kb) {
          mbar_wait_spin(&h2r[kb], 0);
          tc_fence_after();
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            umma_bf16(acc_head, umma_smem_desc(R1 + kb * 16384 + j * 32, 16, 1024),
                      umma_smem_desc(W2T + kb * PG + j * 32, 16, 1024), idesc_h, accum);
            accum = 1;
          }
        }
        umma_commit(headf);
      }
      FS_STAMP(24);
      // ---- backward through the head ---------------------------------------------------------------------------------
      mbar_wait_spin(gr, 0);
      tc_fence_after();
      {
        // dA2[128 x H] = g W2^T, K = AP: A = g^T (MN-major, 64-row panels PG apart), B = W2T (MN-major, 64-column
        // panels PG apart); 16 rows of K per MMA (2 KB); the lo halves sit AP rows into each panel
        const uint32_t idesc_a = umma_idesc_bf16(128, static_cast<uint32_t>(H), 1u, 1u);
        uint32_t accum = 0;
#pragma unroll
        for (int ks = 0; ks < AP / 16; ++ks) {
          const uint32_t ghi = GT + ks * 2048, glo = GT + AP * 128 + ks * 2048;
          const uint32_t whi = W2T + ks * 2048, wlo = W2T + AP * 128 + ks * 2048;
          umma_bf16(acc0, umma_smem_desc(ghi, PG, 1024), umma_smem_desc(whi, PG, 1024), idesc_a, accum);       // hi * hi
          umma_bf16(acc0, umma_smem_desc(ghi, PG, 1024), umma_smem_desc(wlo, PG, 1024), idesc_a, 1u);          // hi * lo
          umma_bf16(acc0, umma_smem_desc(glo, PG, 1024), umma_smem_desc(whi, PG, 1024), idesc_a, 1u);          // lo * hi
          accum = 1;
        }
        // [dW2_hi | dW2_lo][c][j] = sum_r H2[r][c] g[r][j]: A = H2 (MN-major: M = c, K = rows), B = g^T (K-major, N = 2AP)
        const uint32_t idesc_w = umma_idesc_bf16(128, 2u * AP, 1u, 0u);
        for (int mh = 0; mh < mtH; ++mh) {
#pragma unroll
          for (int t = 0; t < 8; ++t)
            umma_bf16(acc_dw + 2 * AP * mh, umma_smem_desc(R1 + 2 * mh * 16384 + t * 2048, 16384, 1024),
                      umma_smem_desc(GT + (t >> 2) * PG + (t & 3) * 32, 16, 1024), idesc_w, t > 0 ? 1u : 0u);
        }
        umma_commit(bwdf);
      }
      FS_STAMP(25);
      // ---- dH1: acc1 = dZ2 W1^T in two N halves.  Accumulates into acc1: every worker warp has read the dW2
      //      columns of acc1 before its first arrival on dz2r[0], while acc0 (dA2) is still being drained by the dZ2 epilogue
      {
        const uint32_t idesc_h2 = umma_idesc_bf16(128, static_cast<uint32_t>(H >> 1), 0u, 0u);
        for (int kb = 0; kb < nkH; ++kb) {
          mbar_wait_spin(&dz2r[kb], 0);
          FS_STAMP(64 + kb);
          for (int nh = 0; nh < 2; ++nh, ++i) {
            const int s = i % NS;
            mbar_wait_spin(&full_bar[s], (i / NS) & 1);
            FS_STAMP(68 + 2 * kb + nh);
            tc_fence_after();
            const uint32_t sa = R1 + kb * 16384, sb = RB + s * FS_STAGE;
#pragma unroll
            for (int jj = 0; jj < 4; ++jj)
              umma_bf16(acc1 + nh * (H >> 1), umma_smem_desc(sa + jj * 32, 16, 1024), umma_smem_desc(sb + jj * 32, 16, 1024),
                        idesc_h2, (kb > 0 || jj > 0) ? 1u : 0u);
            umma_commit(&empty_bar[s]);
            FS_STAMP(76 + 2 * kb + nh);
          }
        }
        umma_commit(dh1f);
      }
      FS_STAMP(23);
      // ---- bias gradients: column sums of dZ as dZ^T x ones.  A = dZ (MN-major: M = 128 columns c, K = the 128 rows),
      //      B = ones [16 n][128 k] (K-major); every one of the 16 accumulator columns of row c holds sum_r dZ[r][c].
      //      dZ2: all of dz2r has been waited for above, so acc0 (dA2) is drained and dZ2 is complete in R1.
      const uint32_t idesc_cs = umma_idesc_bf16(128, 16u, 1u, 0u);
      for (int mh = 0; mh < mtH; ++mh)
#pragma unroll
        for (int t = 0; t < 8; ++t)
          umma_bf16(acc_cs2 + 16 * mh, umma_smem_desc(R1 + 2 * mh * 16384 + t * 2048, 16384, 1024),
                    umma_smem_desc(ONES + (t >> 2) * 2048 + (t & 3) * 32, 16, 1024), idesc_cs, t > 0 ? 1u : 0u);
      umma_commit(cs2f);
      // dZ1: epilogue 3 writes it over H1 in R0, block by block
      for (int mh = 0; mh < mtH; ++mh) {
        mbar_wait_spin(&dz1r[2 * mh], 0);
        if (2 * mh + 1 < nkH) mbar_wait_spin(&dz1r[2 * mh + 1], 0);
        tc_fence_after();
#pragma unroll
        for (int t = 0; t < 8; ++t)
          umma_bf16(acc_cs1 + 16 * mh, umma_smem_desc(R0 + 2 * mh * 16384 + t * 2048, 16384, 1024),
                    umma_smem_desc(ONES + (t >> 2) * 2048 + (t & 3) * 32, 16, 1024), idesc_cs, t > 0 ? 1u : 0u);
      }
      umma_commit(cs1f);
    }
  } else {
    // ===================== workers ================================================================================
    const int wt = static_cast<int>(threadIdx.x);               // 0..511
    const int q = warp & 3, sub = warp >> 2;                     // TMEM lane quadrant, column share
    const int erow = q * 32 + lane;                              // epilogue row == TMEM lane
    const int act = G.act, aout = G.aout;
    const int gchunk = wt & 7, grow0 = wt >> 3;                  // gather mapping: 8 lanes per 128-byte line, rows grow0 + 64 g
    if (wt == 0) FS_STAMP(0);

    // ---- gather the observation rows of this tile into the X slots of R1 ---------------------------------------
    int src_g[2];
#pragma unroll
    for (int g = 0; g < 2; ++g) src_g[g] = rowidx_s[tile * 128 + grow0 + 64 * g];
    const int lrow = tile * 128 + erow;                          // loss row of this thread (actor: the four warps of a lane
                                                                 // quadrant share a row, AP / 4 head columns each; critic: sub == 0)
    const int count = min(*count_s, L.cap);
    const bool live = (sub == 0 || net == 0) && (lrow < count);
    const int src_l = live ? rowidx_s[lrow] : 0;
    // one warp instruction copies 4 rows x 128 contiguous bytes (4 L1 wavefronts; a lane-per-row mapping needed 32)
    auto gather_block = [&](int kb) {
#pragma unroll
      for (int g = 0; g < 2; ++g) {
        const int row = grow0 + 64 * g;
        const __nv_bfloat16* src = p.obs_img + static_cast<size_t>(src_g[g]) * p.Dp + kb * 64 + gchunk * 8;
        cp_async_16(R1 + (kb & 3) * 16384 + row * 128 + ((gchunk ^ (row & 7)) << 4), src);
      }
      cp_async_commit();
    };
    const int nb0 = nk0 < FS_XSLOTS ? nk0 : FS_XSLOTS;
    for (int kb = 0; kb < nb0; ++kb) gather_block(kb);
    if (wt == 0) FS_STAMP(26);
    const float adv_sum = L.adv_sum[step], adv_sq = L.adv_sq[step];
    // per-row loss inputs (update-static: old log-prob / value, advantage / target, action), requested BEFORE the dependency
    // wait: under PDL this part of the kernel runs while the previous optimizer step drains, so the loads -- each touches 32
    // distinct lines -- are off the critical path.  Measured (configs[1], ms per update): here 5.48; after the X rows are
    // published, in the shadow of the L1 GEMM, 5.70; after epilogue 2, where the values are needed, 5.67 -- there the burst of the
    // warps that finish the epilogue first stalled the shared-memory traffic of the warp that finishes last by ~2k cycles.
    constexpr int CW = AP / 4;                                   // head columns of one actor loss warp: [sub CW, sub CW + CW)
    const int j0 = sub * CW;
    float in0 = 0.f, in1 = 0.f, zz[CW];
#pragma unroll
    for (int j = 0; j < CW; ++j) zz[j] = 0.f;
    if (live) {
      if (net == 0) {
        in0 = L.logp_old[src_l]; in1 = L.adv[src_l];
        const float* ap = L.action + static_cast<size_t>(src_l) * aout + j0;
        if ((aout & 1) == 0) {                                     // rows are 8-byte aligned: half the load wavefronts
#pragma unroll
          for (int j = 0; j < CW; j += 2)
            if (j0 + j < aout) { const float2 v = *reinterpret_cast<const float2*>(ap + j); zz[j] = v.x; zz[j + 1] = v.y; }
        } else {
#pragma unroll
          for (int j = 0; j < CW; ++j) if (j0 + j < aout) zz[j] = ap[j];
        }
      } else {
        in0 = L.v_old[src_l]; in1 = L.tgt[src_l];
      }
    }

    // ---- everything below reads what the previous optimizer step wrote (PDL: see common.cuh) -------
    griddep_wait();
    if (wt == 0) griddep_launch();
    if (wt == 0) FS_STAMP(28);
    // ---- small operands: biases, head bias / log_std, head kernel^T image (bf16 hi / lo, swizzled) --
    // (all global loads first: the st.shared wrappers are ordering barriers for the compiler)
    float bv = 0.f;
    if (wt < 256) bv = wt < H ? __ldcg(G.b0 + wt) : 0.f;
    else bv = wt - 256 < H ? __ldcg(G.b1 + wt - 256) : 0.f;
    float hbv = 0.f;
    if (wt < AP) hbv = wt < aout ? __ldcg(G.b2 + wt) : 0.f;
    else if (wt < 2 * AP) hbv = (net == 0 && wt - AP < aout) ? __ldcg(p.log_std + wt - AP) : 0.f;
    for (int i = wt; i < (H * AP) >> 2; i += FS_WORKERS) cp_async_16(W2T + i * 16, G.w2img + i);   // H/64 panels of PG bytes
    cp_async_commit();
    // the L1 GEMM needs only the gathered rows: publish them block by block, before the staging of the small operands;
    // for Dp > 256 the slots are refilled as the MMAs release them
    // The critic CTA (relu epilogues: the shorter chain) also TMA-stores every X k-block for the first-layer dW GEMM, straight
    // from its slot as soon as the block is complete; a slot is refilled only after that store has read it (x_stored).
    const bool x_store_cta = net == 1;
    const bool x_store = x_store_cta && wt == 0;
    {
      int issued = nb0 + 1;                                      // cp.async groups committed so far (X blocks, then W2T)
      for (int kb = 0; kb < nk0; ++kb) {
        const int idx = kb < FS_XSLOTS ? kb : kb + 1;            // commit order: X0..X3, W2T, X4, X5, ...
        cp_async_wait_dyn(issued - idx - 1);
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) mbar_arrive(&x_full[kb & 3]);
        if (x_store) {
          mbar_wait(&x_full[kb & 3], (kb >> 2) & 1);             // all 16 warps' parts of the block are in the slot
          tma_store_2d(R1 + (kb & 3) * 16384, &p.tm_xg, kb * 64, tile * 128);
          tma_store_commit();
        }
        // refill the slot of block kb - 1 (one block behind, so that publishing block kb never waits for an MMA)
        if (kb >= 1 && kb - 1 + FS_XSLOTS < nk0) {
          if (x_store) {                                         // the store of block kb - 1 (all but the newest group) has read its slot
            asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
            mbar_arrive(&x_stored[(kb - 1) & 3]);
          }
          mbar_wait(&x_empty[(kb - 1) & 3], ((kb - 1) >> 2) & 1);
          if (x_store_cta) mbar_wait(&x_stored[(kb - 1) & 3], ((kb - 1) >> 2) & 1);
          gather_block(kb - 1 + FS_XSLOTS);
          ++issued;
        }
      }
    }
    if (wt == 0) FS_STAMP(31);
    bias_s[wt] = bv;                                             // [0, 256) layer 0, [256, 512) layer 1
    if (wt < 2 * AP) hb[wt] = hbv;
    if (wt >= AP && wt < 2 * AP) hb[AP + wt] = 1.f / expf(hbv);   // 1 / scale (unused columns: 1)
    if (net == 0 && wt == 2 * AP) {
      // distrax: log|det| = sum log|scale|, scale = exp(log_std); summed in index order (train.py:223)
      float logdet = 0.f;
      for (int j = 0; j < aout; ++j) logdet += logf(fabsf(expf(__ldcg(p.log_std + j))));
      hb[3 * AP] = logdet;
    }
    if (wt >= 256) sts128(ONES + (wt - 256) * 16, make_uint4(0x3F803F80u, 0x3F803F80u, 0x3F803F80u, 0x3F803F80u));   // bf16 1.0
    // g^T starts as zeros: the loss below writes only the aout real columns (hi and lo rows), the padding rows stay 0
    for (int i = wt; i < (2 * PG) >> 4; i += FS_WORKERS) sts128(GT + i * 16, make_uint4(0u, 0u, 0u, 0u));
    if (wt == 0) FS_STAMP(30);
    cp_async_wait<0>();
    fence_proxy_async_smem();                                    // W2T / ones -> async proxy (UMMA)
    worker_bar();                                                // biases / hb / W2T visible to all workers; X complete
    if (wt == 0) FS_STAMP(1);
    // ---- epilogue 1: H1 = act(acc0 + b0) -> R0, then TMA store to HBM ------------------------------
    mbar_wait(accf0, 0);
    tc_fence_after();
    if (wt == 0) FS_STAMP(2);
    // the X store has read R1 before this warp's h1r arrivals let the L2 GEMM (and then epilogue 2, which
    // overwrites R1) proceed
    if (x_store) tma_store_wait_read0();
    FS_STAMP_W(0, 0);
    epilogue_act(acc0, R0, bias_s, act, erow, q, sub * 16, 64, nkH, h1r);   // 64-column block b published on h1r[b]
    FS_STAMP_W(0, 1);
    if (wt == 0) FS_STAMP(3);
    if (wt == FS_STORE_THREAD) {                                  // its own arrivals are done
      for (int b = 0; b < nkH; ++b) {
        mbar_wait(&h1r[b], 0);
        tma_store_2d(R0 + b * 16384, &G.tm_h1, b * 64, tile * 128);
      }
      tma_store_commit();
    }

    // ---- epilogue 2: H2 = act(acc1 + b1) -> R1 -------------------------------------------------------
    mbar_wait(accf1, 0);
    tc_fence_after();
    if (wt == 0) FS_STAMP(4);
    FS_STAMP_W(1, 0);
    epilogue_act(acc1, R1, bias_s + 256, act, erow, q, sub * 16, 64, nkH, h2r);   // 64-column block b published on h2r[b] (head MMAs)
    FS_STAMP_W(1, 1);
    if (wt == 0) FS_STAMP(5);

    // ---- loss and gradient seed g = dL/dout ------------------------------------------------------------------
    // actor: thread = (row, CW head columns) -- the four warps of a TMEM lane quadrant split the AP columns of a row and
    // combine the quadratic form through shared memory; critic: thread = row on the sub == 0 warps (one column)
    mbar_wait(headf, 0);
    tc_fence_after();
    if (wt == 0) FS_STAMP(6);
    // inputs of the statistics sums (LOSS_SUMS), reduced after g^T is published: actor log r and r, critic v - v_old
    float st_a = 0.f, st_b = 1.f;
    {
      const uint32_t th = acc_head + (static_cast<uint32_t>(q * 32) << 16);
      // g^T as bf16 hi/lo, [2AP j][128 rows] SW128 (the MN-major A of dA2 and the K-major B of dW2)
      const uint32_t gcol = GT + (erow >> 6) * PG + ((erow & 7) << 1);
      const int gch = (erow & 63) >> 3;
      auto put_g = [&](int j, float gj) {
        uint32_t hi, lo;
        split_bf16(gj, hi, lo);
        sts_u16(gcol + j * 128 + ((gch ^ (j & 7)) << 4), hi);
        sts_u16(gcol + (AP + j) * 128 + ((gch ^ ((AP + j) & 7)) << 4), lo);
      };
      float* rw = red + q * RS;                                    // [0, AP) dlog_std, [AP, 2 AP) head bias, [2 AP] loss
      if (net == 0) {
        // distrax MultivariateNormalDiag: z = (a - loc) * (1/scale); train.py:223, 234-239.  zz: action -> z in place
        float ohi[CW], olo[CW];
        tmem_ld_32xn(th + j0, ohi);
        tmem_ld_32xn(th + AP + j0, olo);
        tmem_ld_wait();
        float quad = 0.f;
#pragma unroll
        for (int jj = 0; jj < CW; ++jj) {
          const int j = j0 + jj;
          const float mean = (ohi[jj] + olo[jj]) + hb[j];                   // W2_hi and W2_lo contributions
          const float z = j < aout ? (zz[jj] - mean) * hb[2 * AP + j] : 0.f;
          zz[jj] = z;
          if (j < aout) quad += gauss_logp_term(z);
        }
        // qp aliases the hidden biases, last read in epilogue 2.  Every warp's reads precede its h2r arrivals, which precede
        // the head MMAs, headf and this point -- an mbarrier / tcgen05.commit chain that compute-sanitizer's racecheck does not
        // follow (it reported the pair); the named barrier makes the order explicit (~100 cycles, all 16 warps arrive together)
        worker_bar();
        qp[sub * 128 + erow] = quad;
        worker_bar();
        quad = ((qp[erow] + qp[128 + erow]) + qp[256 + erow]) + qp[384 + erow];   // fixed order: column groups 0..3
        float s_loss = 0.f, g_logp = 0.f;
        if (live) {
          const PpoActorRow ar = ppo_actor_row(quad - hb[3 * AP], in0, in1, adv_sum, adv_sq, L.inv_mb, L.clip_eps);
          s_loss = ar.loss; g_logp = ar.g_logp; st_a = ar.logr; st_b = ar.ratio;
        }
        // tile sums of dlog_std and of the head-bias gradient g through a 2 CW x 32 transpose-reduce
        float v[2 * CW];
#pragma unroll
        for (int jj = 0; jj < CW; ++jj) {
          const int j = j0 + jj;
          const float gj = g_logp * (zz[jj] * hb[2 * AP + j]);
          if (j < aout) put_g(j, gj);
          v[jj] = j < aout ? g_logp * (zz[jj] * zz[jj] - 1.f) : 0.f;
          v[CW + jj] = gj;
        }
        const float cs = warp_colsum_n<2 * CW>(v);
        if (lane < CW) rw[j0 + lane] = cs;
        else if (lane < 2 * CW) rw[AP + j0 + lane - CW] = cs;
        if (sub == 0) {
          s_loss = warp_sum(s_loss);
          if (lane == 0) rw[2 * AP] = s_loss;
        }
      } else if (sub == 0) {
        const float ohi = tmem_ld_32x1(th);
        const float olo = tmem_ld_32x1(th + AP);
        tmem_ld_wait();
        float s_loss = 0.f, g0 = 0.f;
        if (live) {
          const PpoValueRow vr = ppo_value_row((ohi + olo) + hb[0], in0, in1, L.inv_mb, L.clip_eps, L.vf_coef);
          s_loss = vr.loss; g0 = vr.g_v; st_a = vr.dv;
        }
        put_g(0, g0);
        const float gs = warp_sum(g0);
        s_loss = warp_sum(s_loss);
        for (int i = lane; i < 2 * AP; i += 32) rw[i] = i == AP ? gs : 0.f;       // head bias gradient = sum of g; no log_std
        if (lane == 0) rw[2 * AP] = s_loss;
      }
    }
    fence_proxy_async_smem();
    tc_fence_before();
    __syncwarp();
    if (lane == 0) mbar_arrive(gr);
    // statistics sums, off the path to the dA2 / dW2 MMAs that g^T starts: red[q][2 AP + 1, 2 AP + 3) (po_stat).  The four
    // warps of an actor lane quadrant hold the same rows: warp sub == 0 sums them.
    if (sub == 0) {
      float* rw = red + q * RS + 2 * AP + 1;
      if (net == 0) {
        const float kl = live ? approx_kl_term(st_a) : 0.f;
        const float clipped = live ? ratio_clipped(st_b, L.clip_eps) : 0.f;
        const float s_kl = warp_sum(kl), s_clip = warp_sum(clipped);
        if (lane == 0) { rw[0] = s_kl; rw[1] = s_clip; }
      } else {
        const float s_vclip = warp_sum(live ? value_clipped(st_a, L.clip_eps) : 0.f);
        if (lane == 0) rw[0] = s_vclip;
      }
    }
    worker_bar();
    if (wt == 0) FS_STAMP(7);
    float* part = p.part + static_cast<size_t>(tile) * p.part_stride;
    if (wt < 2 * AP + (net == 0 ? 3 : 2)) {
      float s = 0.f;
      for (int w = 0; w < 4; ++w) s += red[w * RS + wt];         // fixed order: the four loss warps
      if (wt > 2 * AP) part[G.po_stat + wt - 2 * AP - 1] = s;
      else if (wt == 2 * AP) part[G.po_loss] = s;
      else if (wt >= AP) { if (wt - AP < aout) part[G.po_b2 + wt - AP] = s; }
      else if (net == 0 && wt < aout) part[p.po_logstd + wt] = s;
    }

    // ---- dW2 (head kernel gradient) and dZ2 = dA2 * f'(H2) ----------------------------------------
    mbar_wait(bwdf, 0);
    tc_fence_after();
    if (wt == 0) FS_STAMP(8);
    if (sub < mtH) {                                             // warp (q, sub) reads the 128-column tile mh = sub
      // staged in shared memory as the [H][aout] fp32 block of the partial (the W2T image is dead once bwdf has fired) and
      // written by ONE bulk copy: as per-thread stores (a row of aout floats per lane: ~11 lines per store instruction) this
      // section held the dZ2 epilogue of these warps back by ~2k cycles
      const uint32_t td = acc_dw + 2 * AP * sub + (static_cast<uint32_t>(q * 32) << 16);
      const int c = sub * 128 + erow;
#pragma unroll
      for (int ch = 0; ch < AP / 16; ++ch) {
        float dhi[16], dlo[16];
        tmem_ld_32x16(td + 16 * ch, dhi);
        tmem_ld_32x16(td + AP + 16 * ch, dlo);
        tmem_ld_wait();
        if (c < H) {
#pragma unroll
          for (int jj = 0; jj < 16; ++jj)
            if (16 * ch + jj < aout) sts32(W2T + static_cast<uint32_t>(c * aout + 16 * ch + jj) * 4u, dhi[jj] + dlo[jj]);   // g_hi and g_lo contributions
        }
      }
      fence_proxy_async_smem();
      asm volatile("bar.sync 2, %0;" ::"r"(128 * mtH) : "memory");   // the warps with sub < mtH = threads [0, 128 mtH)
      if (wt == 0) {
        bulk_store_1d(part + G.po_w2, W2T, static_cast<uint32_t>(H * aout) * 4u);
        tma_store_commit();
      }
    }
    FS_STAMP_W(2, 0);
    epilogue_dact(acc0, R1, R1, act, erow, q, sub * 16, 64, nkH, dz2r);            // in place: H2 -> dZ2, block b published on dz2r[b]
    FS_STAMP_W(2, 1);
    if (wt == 0) FS_STAMP(9);
    // The dZ2 store is issued in one batch, and only once the TMA producer has issued its last weight load: the TMA unit works its
    // queue in order and a 16 KB store drains at the SM's ~32 B/clk egress rate, so stores issued block by block held the last
    // dH1 weight stages back by 1-2.7k cycles (measured: stage requested -> landed).  dZ2 stays in R1 until the end of the tile:
    // epilogue 3 writes dZ1 over H1 in R0, so nothing waits for this store.
    if (wt == FS_STORE_THREAD) {
      for (int b = 0; b < nkH; ++b) mbar_wait(&dz2r[b], 0);
      mbar_wait(ldi, 0);
      for (int b = 0; b < nkH; ++b) tma_store_2d(R1 + b * 16384, &G.tm_dz2, b * 64, tile * 128);
      tma_store_commit();
    }

    // ---- epilogue 3: dZ1 = acc1 * f'(H1) -> R0 (in place over H1) -> TMA store ---------------------------------------
    mbar_wait(dh1f, 0);                                            // dH1 accumulator complete
    mbar_wait(cs2f, 0);                                            // column sums of dZ2 complete
    tc_fence_after();
    if (wt == 0) FS_STAMP(10);
    if (wt == FS_STORE_THREAD) asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");   // the H1 store (all but the newest group, dZ2) has read R0
    float cs2 = 0.f;
    if (sub < mtH) cs2 = tmem_ld_32x1(acc_cs2 + 16 * sub + (static_cast<uint32_t>(q * 32) << 16));
    tmem_ld_wait();
    worker_bar();
    if (sub < mtH && sub * 128 + erow < H) part[G.po_db1 + sub * 128 + erow] = cs2;     // layer-1 bias gradient of this tile
    FS_STAMP_W(3, 0);
    epilogue_dact(acc1, R0, R0, act, erow, q, sub * 16, 64, nkH, dz1r);   // in place: H1 -> dZ1; 64-column blocks, each stored as soon as it is complete
    FS_STAMP_W(3, 1);
    if (wt == 0) FS_STAMP(11);
    if (wt == FS_STORE_THREAD) {
      for (int b = 0; b < nkH; ++b) {
        mbar_wait(&dz1r[b], 0);
        tma_store_2d(R0 + b * 16384, &G.tm_dz1, b * 64, tile * 128);
      }
      tma_store_commit();
    }
    mbar_wait(cs1f, 0);
    tc_fence_after();
    if (sub < mtH) {
      const float cs1 = tmem_ld_32x1(acc_cs1 + 16 * sub + (static_cast<uint32_t>(q * 32) << 16));
      tmem_ld_wait();
      if (sub * 128 + erow < H) part[G.po_db0 + sub * 128 + erow] = cs1;               // layer-0 bias gradient of this tile
    }
    // The bulk stores must have READ shared memory before the CTA exits; their global writes complete with the grid.
    if (wt == FS_STORE_THREAD || wt == 0) tma_store_wait_read0();   // thread 0: the dW2 bulk copy (and, critic CTA, the X stores)
    if (wt == 0) FS_STAMP(12);
  }

  // all TMEM reads of this unit are complete (tcgen05.wait::ld) before the caller reuses or frees the columns
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
}

// One launch = one minibatch step: CTA blockIdx.x handles unit blockIdx.x.
template <int AP>
__global__ void __launch_bounds__(FS_THREADS, 1) fused_step_kernel(const __grid_constant__ FusedParams p) {
  extern __shared__ uint8_t smem_raw[];
  __shared__ uint32_t tmem_slot;
  const uint32_t raw = smem_u32(smem_raw);
  const uint32_t base = (raw + 1023u) & ~1023u;
  uint8_t* sm = smem_raw + (base - raw);
  const int warp = threadIdx.x >> 5;
  const int unit = static_cast<int>(blockIdx.x);
  if ((unit >> 1) * 128 < min(p.loss.count[p.loss.step], p.loss.cap)) {   // live tile: needs the tensor memory
    if (warp == FS_MMA_WARP) {
      tmem_alloc(&tmem_slot, 512);
      tmem_relinquish();
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = tmem_slot;
    fused_tile<AP>(p, unit, p.loss.step, sm, base, tmem_base);
    if (warp == FS_MMA_WARP) tmem_dealloc(tmem_base, 512);
  } else {
    fused_tile<AP>(p, unit, p.loss.step, sm, base, 0u);                      // dead tile: zeroes its partials and returns
  }
}

}  // namespace minppo
