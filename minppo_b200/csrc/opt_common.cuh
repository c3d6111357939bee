// minppo_b200 -- device helpers of the optimizer (dwopt.cuh) and of the weight-image kernel (adam.cu).
#pragma once

#include "common.cuh"
#include "minppo_internal.h"

namespace minppo {

// Sense-free grid barrier on a monotonically increasing 64-bit counter.  All blocks of the
// grid are co-resident (grid <= #SMs, one block per SM).  Arrive = atom.add.release.gpu, wait =
// ld.acquire.gpu polling by one thread, bracketed by CTA barriers (cumulativity carries the other
// threads' writes).  A bounded spin turns a scheduling surprise into an error flag instead of a
// hung GPU.
MINPPO_DEVINL void grid_barrier(unsigned long long* counter, int* err_flag) {
  __syncthreads();
  if (threadIdx.x == 0) {
    unsigned long long old;
    asm volatile("atom.add.release.gpu.global.u64 %0, [%1], 1;" : "=l"(old) : "l"(counter) : "memory");
    const unsigned long long target = (old / gridDim.x + 1ULL) * gridDim.x;
    const long long t0 = clock64();
    for (;;) {
      unsigned long long cur;
      asm volatile("ld.acquire.gpu.global.u64 %0, [%1];" : "=l"(cur) : "l"(counter) : "memory");
      if (cur >= target) break;
      if (clock64() - t0 > 4000000000LL) { atomicExch(err_flag, MINPPO_ERR_BARRIER); break; }
    }
  }
  __syncthreads();
}

// One Adam step on one element (optax.scale_by_adam + scale(-lr), train.py:116-124), after the
// global-norm clip (optax.clip_by_global_norm: g unchanged if gnorm < max_norm, else g / gnorm * max_norm).
struct AdamScalars { float gnorm, lr, c1, c2; bool trigger; };
MINPPO_DEVINL void adam_element(const OptArgs& a, const AdamScalars& sc, float g, float& p, float& m, float& v) {
  if (!sc.trigger) g = (g / sc.gnorm) * a.max_norm;
  m = a.one_minus_b1 * g + a.b1 * m;
  v = a.one_minus_b2 * (g * g) + a.b2 * v;
  const float u = (m / sc.c1) / (sqrtf(v / sc.c2 + a.eps_root) + a.eps);
  p = p + (-sc.lr) * u;
}
// learning rate of this step (train.py:98-101 annealed, else opt.lr) and the Adam bias corrections
MINPPO_DEVINL void step_scalars(const OptArgs& a, int count, float& lr, float& c1, float& c2) {
  if (a.anneal) {
    const float frac = 1.0f - static_cast<float>(count / a.anneal_div) / static_cast<float>(a.num_updates);
    lr = a.lr * frac;
  } else {
    lr = a.lr;
  }
  const float cnt1 = static_cast<float>(count + 1);
  c1 = 1.0f - powf(a.b1, cnt1);
  c2 = 1.0f - powf(a.b2, cnt1);
}
// bf16 images of a kernel element (what the tcgen05 GEMMs read)
MINPPO_DEVINL void write_images(const OptLeaf& L, int i, float p) {
  if (L.img_n) L.img_n[i - L.offset] = __float2bfloat16_rn(p);      // same [in][out] layout as the arena leaf: coalesced
  if (L.img_w2) {                                          // head kernel [in=r][out=j] -> kernel^T hi / lo, SW128
    const int e = i - L.offset;
    const int r = e / L.cols, j = e % L.cols;
    uint32_t hi, lo;
    split_bf16(p, hi, lo);
    *reinterpret_cast<uint16_t*>(L.img_w2 + swp_off(L.ap, j, r)) = static_cast<uint16_t>(hi);
    *reinterpret_cast<uint16_t*>(L.img_w2 + swp_off(L.ap, L.ap + j, r)) = static_cast<uint16_t>(lo);
  }
}

// ---- leaf table in shared memory ---------------------------------------------------------------
// Kernel parameters live in the constant bank; indexing them with a run-time leaf index costs one
// dependent LDC per field (the first merged kernel spent most of its optimizer phases there).  Every
// CTA copies the table to shared memory once and the strided loops below walk it monotonically.
constexpr int OPT_TAB_LEAVES = 20;   // >= 4 (num_layers + 1) + 1 leaves for num_layers <= 3 (validate_config); static shared memory is scarce
struct LeafTab {
  OptLeaf leaf[OPT_TAB_LEAVES];
  int size[OPT_TAB_LEAVES];
  int nleaves;
  int n_early;                   // elements of the leaves with late == 0
};
MINPPO_DEVINL void leaf_tab_build(LeafTab& T, const OptArgs& a, int tid, int nthreads) {
  // every word by a different thread: the constant-bank misses of a cold launch overlap instead of queueing behind one
  // thread (a serial walk over the leaves by thread 0 cost ~3k cycles at the head of every launch)
  constexpr int WORDS = sizeof(OptLeaf) / 4;
  const uint32_t* src = reinterpret_cast<const uint32_t*>(a.leaf);
  uint32_t* dst = reinterpret_cast<uint32_t*>(T.leaf);
  for (int w = tid; w < a.nleaves * WORDS; w += nthreads) dst[w] = src[w];
  for (int l = tid; l < a.nleaves; l += nthreads) T.size[l] = a.leaf[l].size;
  if (tid == nthreads - 1) { T.nleaves = a.nleaves; T.n_early = a.n_early; }
}

// fixed-order sum of `nparts` partials, 16 loads in flight
MINPPO_DEVINL float sum_partials16(const float* __restrict__ src, int nparts, size_t stride) {
  float acc = 0.f;
  int p = 0;
#pragma unroll 1
  for (; p + 16 <= nparts; p += 16) {
    float v[16];
#pragma unroll
    for (int u = 0; u < 16; ++u) v[u] = __ldcg(src + static_cast<size_t>(p + u) * stride);
#pragma unroll
    for (int u = 0; u < 16; ++u) acc += v[u];
  }
#pragma unroll 1
  for (; p < nparts; ++p) acc += __ldcg(src + static_cast<size_t>(p) * stride);
  return acc;
}
// split-K partials: read once, written by another SM just before (L2-resident): no L1 allocation, 256-byte L2 sectors
// (a warp reads 512 contiguous bytes of every partial)
MINPPO_DEVINL float4 ld_partial_v4(const float* p) {
  float4 v;
  asm volatile("ld.global.L1::no_allocate.L2::256B.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p) : "memory");
  return v;
}
// same, four consecutive elements at once (16-byte loads; src 16-byte aligned, stride % 4 == 0).  Below 16 partials the loads
// go out in batches of REM (4, or 8 where the registers allow it: dwopt's S = 8 partials in one L2 round trip instead of two);
// the summation order is the same for every REM.
template <int REM = 4>
MINPPO_DEVINL float4 sum_partials16_v4(const float* __restrict__ src, int nparts, size_t stride) {
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
  int p = 0;
#pragma unroll 1
  for (; p + 16 <= nparts; p += 16) {
    float4 v[16];
#pragma unroll
    for (int u = 0; u < 16; ++u) v[u] = ld_partial_v4(src + static_cast<size_t>(p + u) * stride);
#pragma unroll
    for (int u = 0; u < 16; ++u) { acc.x += v[u].x; acc.y += v[u].y; acc.z += v[u].z; acc.w += v[u].w; }
  }
#pragma unroll 1
  for (; REM > 4 && p + REM <= nparts; p += REM) {
    float4 v[REM];
#pragma unroll
    for (int u = 0; u < REM; ++u) v[u] = ld_partial_v4(src + static_cast<size_t>(p + u) * stride);
#pragma unroll
    for (int u = 0; u < REM; ++u) { acc.x += v[u].x; acc.y += v[u].y; acc.z += v[u].z; acc.w += v[u].w; }
  }
#pragma unroll 1
  for (; p + 4 <= nparts; p += 4) {                      // remainders in batches of 4 loads in flight (same summation order)
    float4 v[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) v[u] = ld_partial_v4(src + static_cast<size_t>(p + u) * stride);
#pragma unroll
    for (int u = 0; u < 4; ++u) { acc.x += v[u].x; acc.y += v[u].y; acc.z += v[u].z; acc.w += v[u].w; }
  }
#pragma unroll 1
  for (; p < nparts; ++p) {
    const float4 v = ld_partial_v4(src + static_cast<size_t>(p) * stride);
    acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
  }
  return acc;
}

// Gradient reduction of one class of leaves -> gflat; returns this thread's sum of squares.
//   LATE == false: leaves whose partials the fused step kernel wrote (biases of the output heads, head
//                  kernels, log_std, ...): one element per job, then the LOSS_SUMS loss sums.
//   LATE == true : leaves whose partials the dW GEMM writes (hidden kernels): four
//                  elements per job (sizes and partial strides are multiples of 4, partial buffers 16-byte
//                  aligned; gflat itself is only 4-byte aligned at a leaf offset).
// Jobs are dealt round-robin (job = first + k * stride); the leaf walk is monotonic in k.
// `ready(leaf, element)` runs before the partials of a LATE job are read (dwopt.cuh: waits for the dW GEMM tile).
struct NoWait { MINPPO_DEVINL void operator()(const OptLeaf&, int) const {} };
template <bool LATE, typename ReadyFn = NoWait>
MINPPO_DEVINL float reduce_leaves(const OptArgs& a, const LeafTab& T, int first, int stride, int max_parts = 0x7fffffff,
                                  ReadyFn ready = ReadyFn()) {
  const int nl = T.nleaves;
  int l = -1, base = 0, n = 0;
  float ss = 0.f;
#pragma unroll 1
  for (int j = first;; j += stride) {
    while (l < nl && j >= base + n) {
      base += n;
      n = 0;
      do { ++l; } while (l < nl && (T.leaf[l].late != 0) != LATE);
      if (l < nl) n = LATE ? (T.size[l] >> 2) : T.size[l];
    }
    if (l >= nl) {
      if (!LATE && j - base < LOSS_SUMS)  // the loss sums ride behind the early leaves
        a.gflat[a.P + (j - base)] = sum_partials16(a.loss_src + a.loss_src_offset + (j - base), min(a.loss_nparts, max_parts), a.loss_part_stride);
      break;
    }
    const OptLeaf& L = T.leaf[l];
    const int x = j - base;
    if (LATE) {
      ready(L, 4 * x);
      const float4 g = sum_partials16_v4(L.grad_src + L.src_offset + 4 * x, L.nparts, L.part_stride);
      float* dst = a.gflat + L.offset + 4 * x;
      dst[0] = g.x; dst[1] = g.y; dst[2] = g.z; dst[3] = g.w;
      ss = fmaf(g.x, g.x, ss); ss = fmaf(g.y, g.y, ss); ss = fmaf(g.z, g.z, ss); ss = fmaf(g.w, g.w, ss);
    } else {
      const float g = sum_partials16(L.grad_src + L.src_offset + x, min(L.nparts, max_parts), L.part_stride) + L.grad_bias;
      a.gflat[L.offset + x] = g;
      ss = fmaf(g, g, ss);
    }
  }
  return ss;
}

// clip + Adam over the arena, four elements in flight per thread; gradient from gflat
MINPPO_DEVINL void apply_adam(const OptArgs& a, const LeafTab& T, const AdamScalars& sc, int first, int stride,
                              const float* gsrc = nullptr) {
  const int P = a.P;
  const float* gbuf = gsrc ? gsrc : a.gflat;
  int l = 0;
#pragma unroll 1
  for (int i0 = first; i0 < P; i0 += 4 * stride) {
    float g[4], pv[4], mv[4], nv[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int i = i0 + u * stride;
      if (i < P) { g[u] = __ldcg(gbuf + i); pv[u] = __ldcg(a.params + i); mv[u] = __ldcg(a.mu + i); nv[u] = __ldcg(a.nu + i); }
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int i = i0 + u * stride;
      if (i < P) {
        adam_element(a, sc, g[u], pv[u], mv[u], nv[u]);
        a.params[i] = pv[u];
        a.mu[i] = mv[u];
        a.nu[i] = nv[u];
        while (l + 1 < T.nleaves && i >= T.leaf[l + 1].offset) ++l;
        write_images(T.leaf[l], i, pv[u]);
      }
    }
  }
}

// clip + Adam restricted to the leaves of one class (same job numbering as reduce_leaves<LATE>, one element per
// job): used by the merged kernel for the small leaves when the hidden-kernel elements stay in registers.
template <bool LATE>
MINPPO_DEVINL void apply_adam_class(const OptArgs& a, const LeafTab& T, const AdamScalars& sc, int first, int stride) {
  if (!LATE && first >= T.n_early) return;
  const int nl = T.nleaves;
  int l = -1, base = 0, n = 0;
#pragma unroll 1
  for (int j = first;; j += stride) {
    while (l < nl && j >= base + n) {
      base += n;
      n = 0;
      do { ++l; } while (l < nl && (T.leaf[l].late != 0) != LATE);
      if (l < nl) n = T.size[l];
    }
    if (l >= nl) break;
    const OptLeaf& L = T.leaf[l];
    const int i = L.offset + (j - base);
    float g = __ldcg(a.gflat + i), pv = __ldcg(a.params + i), mv = __ldcg(a.mu + i), nv = __ldcg(a.nu + i);
    adam_element(a, sc, g, pv, mv, nv);
    a.params[i] = pv;
    a.mu[i] = mv;
    a.nu[i] = nv;
    write_images(L, i, pv);
  }
}

}  // namespace minppo
