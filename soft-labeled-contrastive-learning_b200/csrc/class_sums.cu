// class_sums.cu -- per-class (and per rMC partition) weighted feature sums over an
// NCHW map, their finalisers (EMA class centres, centroids) and the centroid
// backward.
//
// Replaces (reference, file:line):
//   update_class_center_iter   utils/utils_.py:568-594  (K masked full-map passes + K host syncs)
//   cal_centroid               utils/utils_.py:479-565  (hard / soft / arg-max weights, partitions, EMA)
//   autograd backward of cal_centroid (dfeat and d soft-label), SURVEY.md appendix A.3 / A.4
//
// Roofline: HBM.  Segmented warp reduction: a lane owns VEC (=4) consecutive
// pixels, a warp owns CPW channels; the lane's weight row w[pixel][column] is
// built once per tile in registers, each channel plane is read with one
// coalesced 128-bit load per lane, and the partial sums acc[channel][column]
// stay in registers across ALL tiles of the persistent block.  The cross-lane
// (shuffle) reduction happens once per block at the very end, so the steady
// state is load + FMA only: 4C + 8 bytes per pixel, one pass, no atomics.
// Per-block partials are summed in fp64 by a second tiny kernel in block
// order (deterministic; exact integer counts beyond 2^24).
#include "centroid_pair.cuh"
#include "common.cuh"
#include "peer.cuh"
#include "proto_math.cuh"

#include <cuda.h>
#include <limits.h>
#include <math.h>
#include <stdlib.h>

#include <algorithm>
#include <type_traits>

namespace slcl {
namespace {

constexpr int kThreads = 256;
constexpr int kWarps = kThreads / 32;
constexpr size_t kTicketBytes = 256;     // tail of the workspace: the reduce kernel's block counter

enum WeightMode { kHard = 0, kSoft = 1, kPlanar = 2 };

struct SumArgs {
  const float* feat;
  int64_t batch, channels, pixels, sb, sc, sp;
  int mode;
  const int64_t* labels;     // kHard: [N]
  const float* probs;        // kSoft: [B,K,HW]
  int weighted;              // kSoft: 1 = p_k weights, 0 = arg-max one-hot
  float threshold;           // certainty threshold, active when 0 < t < 1
  const int32_t* part_id;    // [N] or null
  int n_part, n_class;
  const float* planar;       // kPlanar: [cols][N]
  int n_cols;                // logical columns (n_part * n_class, or planar cols)
  int64_t tiles_per_image, n_tiles;
  int cg_per_block, pt_per_block;   // warps = cg_per_block * pt_per_block
  int n_cw;                         // v3: consumer warps in use (channels per block = n_cw * CPW)
  int n_stages;                     // v3: ring depth
  float* partial;            // [gridDim.x][KWT][C+1]
  unsigned int* ticket;      // block counter of the reduce kernel (zeroed by the sweep, self-resetting)
};

template <int VEC>
__device__ __forceinline__ void ld_vec(const float* p, float (&v)[VEC]) {
  if constexpr (VEC == 4) { float4 t = ld_stream4(p); v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w; }
  else { v[0] = ld_stream1(p); }
}
template <int VEC>
__device__ __forceinline__ void ld_vec_keep(const float* p, float (&v)[VEC]) {
  if constexpr (VEC == 4) { float4 t = *reinterpret_cast<const float4*>(p); v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w; }
  else { v[0] = *p; }
}
template <int VEC>
__device__ __forceinline__ void st_vec(float* p, const float (&v)[VEC]) {
  if constexpr (VEC == 4) st_stream4(p, make_float4(v[0], v[1], v[2], v[3]));
  else st_stream1(p, v[0]);
}

// Logits mode (SLCL_SOFT_LOGITS): the K values z[0..K) of one pixel become softmax(z) in place.  `arg` = first index of
// the largest logit (torch.argmax), `pmax` = 1/s = the largest probability.  Full-precision expf and an IEEE division,
// the arithmetic of torch.softmax, so certainty and arg-max decisions agree with softmax-then-probabilities except
// within the last bits of a tie.
__device__ __forceinline__ void softmax_inplace(float (&z)[SLCL_MAX_CLASSES], int K, float& pmax, int& arg) {
  float zmax = -INFINITY;
  arg = 0;
#pragma unroll
  for (int k = 0; k < SLCL_MAX_CLASSES; ++k)
    if (k < K && z[k] > zmax) { zmax = z[k]; arg = k; }
  float s = 0.f;
#pragma unroll
  for (int k = 0; k < SLCL_MAX_CLASSES; ++k)
    if (k < K) { z[k] = expf(z[k] - zmax); s += z[k]; }
#pragma unroll
  for (int k = 0; k < SLCL_MAX_CLASSES; ++k)
    if (k < K) z[k] = z[k] / s;
  pmax = 1.f / s;
}

// Weight row(s) of VEC pixels starting at image b, pixel p (flat index pix).
// Hard labels: utils_.py:581 / :535.  Soft: :517-519 (weighted) or :524-525
// (arg-max one-hot); certainty :511-514; partitions: SURVEY.md 8(c)-2.  LOGITS: `probs` holds logits, softmax first.
template <int KWT, int VEC, bool LOGITS = false>
__device__ __forceinline__ void build_weights(const SumArgs& a, int64_t b, int64_t p, int64_t pix, float (&w)[VEC][KWT]) {
#pragma unroll
  for (int v = 0; v < VEC; ++v)
#pragma unroll
    for (int j = 0; j < KWT; ++j) w[v][j] = 0.f;

  if (a.mode == kPlanar) {
    const int64_t n = a.batch * a.pixels;
#pragma unroll
    for (int j = 0; j < KWT; ++j) {
      if (j < a.n_cols) {
        float t[VEC];
        ld_vec_keep<VEC>(a.planar + (int64_t)j * n + pix, t);
#pragma unroll
        for (int v = 0; v < VEC; ++v) w[v][j] = t[v];
      }
    }
    return;
  }
  int part[VEC];
#pragma unroll
  for (int v = 0; v < VEC; ++v) part[v] = a.part_id ? a.part_id[pix + v] : 0;

  if (a.mode == kHard) {
#pragma unroll
    for (int v = 0; v < VEC; ++v) {
      long long lab = a.labels[pix + v];
      bool ok = lab >= 0 && lab < a.n_class && part[v] >= 0 && part[v] < a.n_part;
      int col = ok ? part[v] * a.n_class + (int)lab : -1;
#pragma unroll
      for (int j = 0; j < KWT; ++j) w[v][j] = (j == col) ? 1.0f : 0.0f;
    }
    return;
  }
  // soft probabilities, planar per image: probs[(b*K + k)*HW + p]
  float pr[SLCL_MAX_CLASSES][VEC];
#pragma unroll
  for (int k = 0; k < SLCL_MAX_CLASSES; ++k) {
    if (k < a.n_class) ld_vec_keep<VEC>(a.probs + (b * a.n_class + k) * a.pixels + p, pr[k]);
  }
#pragma unroll
  for (int v = 0; v < VEC; ++v) {
    float best = -INFINITY;
    int arg = 0;
    if constexpr (LOGITS) {
      float z[SLCL_MAX_CLASSES];
#pragma unroll
      for (int k = 0; k < SLCL_MAX_CLASSES; ++k) z[k] = (k < a.n_class) ? pr[k][v] : 0.f;
      softmax_inplace(z, a.n_class, best, arg);
#pragma unroll
      for (int k = 0; k < SLCL_MAX_CLASSES; ++k) pr[k][v] = z[k];
    } else {
#pragma unroll
      for (int k = 0; k < SLCL_MAX_CLASSES; ++k) {
        if (k < a.n_class && pr[k][v] > best) { best = pr[k][v]; arg = k; }
      }
    }
    float cert = (a.threshold > 0.f && a.threshold < 1.f) ? ((best >= a.threshold) ? 1.f : 0.f) : 1.f;
    bool ok = part[v] >= 0 && part[v] < a.n_part;
#pragma unroll
    for (int k = 0; k < SLCL_MAX_CLASSES; ++k) {
      if (k < a.n_class) {
        float wk = a.weighted ? pr[k][v] * cert : ((k == arg) ? cert : 0.f);
        int col = part[v] * a.n_class + k;
#pragma unroll
        for (int j = 0; j < KWT; ++j) if (ok && j == col) w[v][j] = wk;
      }
    }
  }
}

// Block tile = kChunks x (32*VEC) pixels.  Phase A: each thread builds the weight rows of VEC pixels
// ONCE and parks them in shared memory as sW[column][pixel]; phase B: a warp owns CPW channels of the
// tile's chunks, streams them with 128-bit loads and reads the weights back with conflict-free
// 128-bit shared loads.  The weights therefore cost registers only transiently, whatever P*K is.
constexpr int kChunks = 8;

template <int KWT, int CPW, int VEC, bool LOGITS>
__global__ void __launch_bounds__(kThreads, 2) class_sums_kernel(const SumArgs a) {
  constexpr bool kPipe = KWT <= 8;       // wide weight rows: keep one x buffer, the accumulators need the registers
  extern __shared__ __align__(16) float sW[];            // [KWT][TP]
  __shared__ float s_acc[kWarps][CPW * KWT];
  __shared__ float s_w[kWarps][KWT];
  constexpr int TP = kChunks * 32 * VEC;                 // pixels per block tile (1024 or 256)
  constexpr int CPS = (8 / CPW) < 1 ? 1 : (8 / CPW);     // chunks loaded together (8 vector loads in flight per lane)
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int cg = warp % a.cg_per_block, pt = warp / a.cg_per_block;
  const int C = (int)a.channels;
  const int c0 = (blockIdx.y * a.cg_per_block + cg) * CPW;
  const bool count_weights = blockIdx.y == 0;
  if (blockIdx.x == 0 && blockIdx.y == 0 && threadIdx.x == 0) *a.ticket = 0u;

  float acc[CPW][KWT];
  float wacc[KWT];
#pragma unroll
  for (int j = 0; j < CPW; ++j)
#pragma unroll
    for (int q = 0; q < KWT; ++q) acc[j][q] = 0.f;
#pragma unroll
  for (int q = 0; q < KWT; ++q) wacc[q] = 0.f;

  for (int64_t tile = blockIdx.x; tile < a.n_tiles; tile += gridDim.x) {
    const int64_t b = tile / a.tiles_per_image;
    const int64_t p_tile = (tile - b * a.tiles_per_image) * TP;
    {   // ---- phase A: weights of this tile -> shared memory
      // one pixel at a time keeps the register footprint of this phase at KWT (+ K probabilities);
      // consecutive threads take consecutive pixels, so loads and the smem stores are conflict-free
#pragma unroll 1
      for (int v = 0; v < VEC; ++v) {
        const int pl = v * kThreads + threadIdx.x;
        const int64_t p = p_tile + pl;
        float w1[1][KWT];
        if (p < a.pixels) build_weights<KWT, 1, LOGITS>(a, b, p, b * a.pixels + p, w1);
        else {
#pragma unroll
          for (int q = 0; q < KWT; ++q) w1[0][q] = 0.f;
        }
#pragma unroll
        for (int q = 0; q < KWT; ++q) {
          sW[q * TP + pl] = w1[0][q];
          if (count_weights) wacc[q] += w1[0][q];
        }
      }
    }
    __syncthreads();
    // ---- phase B: stream the channels of this warp's chunks, software-pipelined: the loads of step
    // i+1 are in flight while step i is being accumulated (two register buffers)
    const float* img = a.feat + b * a.sb;
    const int step_stride = a.pt_per_block * CPS;
    // interior tiles (all pixels and all CPW channels exist) take a predicate-free load path
    const bool full = (p_tile + TP <= a.pixels) && (c0 + CPW <= C) && (kChunks % step_stride == 0 || true);
    const float* lane_base = img + (int64_t)c0 * a.sc + (p_tile + (int64_t)lane * VEC) * a.sp;
    const int64_t chunk_stride = (int64_t)(32 * VEC) * a.sp;
    auto load_step = [&](int ch0, float (&x)[CPS][CPW][VEC]) {
      if (full) {
#pragma unroll
        for (int u = 0; u < CPS; ++u) {
          const int ch = ch0 + u * a.pt_per_block;
          if (ch < kChunks) {
            const float* pch = lane_base + ch * chunk_stride;
#pragma unroll
            for (int j = 0; j < CPW; ++j) ld_vec<VEC>(pch + (int64_t)j * a.sc, x[u][j]);
          }
        }
        return;
      }
#pragma unroll
      for (int u = 0; u < CPS; ++u) {
        const int ch = ch0 + u * a.pt_per_block;
        const int64_t p = p_tile + (int64_t)ch * (32 * VEC) + lane * VEC;
        const bool ok = ch < kChunks && p < a.pixels;
#pragma unroll
        for (int j = 0; j < CPW; ++j) {
          if (ok && c0 + j < C) ld_vec<VEC>(img + (int64_t)(c0 + j) * a.sc + p * a.sp, x[u][j]);
          else {
#pragma unroll
            for (int v = 0; v < VEC; ++v) x[u][j][v] = 0.f;
          }
        }
      }
    };
    auto accumulate = [&](int ch0, const float (&x)[CPS][CPW][VEC]) {
#pragma unroll
      for (int u = 0; u < CPS; ++u) {
        const int ch = ch0 + u * a.pt_per_block;
        if (ch < kChunks) {
          const int pl = ch * (32 * VEC) + lane * VEC;
#pragma unroll
          for (int q = 0; q < KWT; ++q) {
            float wq[VEC];
            if constexpr (VEC == 4) {
              const float4 t = *reinterpret_cast<const float4*>(sW + q * TP + pl);
              wq[0] = t.x; wq[1] = t.y; wq[2] = t.z; wq[3] = t.w;
            } else {
              wq[0] = sW[q * TP + pl];
            }
#pragma unroll
            for (int j = 0; j < CPW; ++j)
#pragma unroll
              for (int v = 0; v < VEC; ++v) acc[j][q] = fmaf(wq[v], x[u][j][v], acc[j][q]);
          }
        }
      }
    };
    if constexpr (!kPipe) {
      float xa[CPS][CPW][VEC];
      for (int ch0 = pt; ch0 < kChunks; ch0 += step_stride) { load_step(ch0, xa); accumulate(ch0, xa); }
    } else {
      float xa[CPS][CPW][VEC], xb[CPS][CPW][VEC];
      int ch0 = pt;
      if (ch0 < kChunks) load_step(ch0, xa);
      while (ch0 < kChunks) {
        const int ch1 = ch0 + step_stride;
        if (ch1 < kChunks) load_step(ch1, xb);
        accumulate(ch0, xa);
        if (ch1 >= kChunks) break;
        const int ch2 = ch1 + step_stride;
        if (ch2 < kChunks) load_step(ch2, xa);
        accumulate(ch1, xb);
        ch0 = ch2;
      }
    }
    __syncthreads();
  }
  // one cross-lane reduction per block
#pragma unroll
  for (int j = 0; j < CPW; ++j)
#pragma unroll
    for (int q = 0; q < KWT; ++q) {
      float r = warp_sum(acc[j][q]);
      if (lane == 0) s_acc[warp][j * KWT + q] = r;
    }
#pragma unroll
  for (int q = 0; q < KWT; ++q) {
    float r = warp_sum(wacc[q]);
    if (lane == 0) s_w[warp][q] = r;
  }
  __syncthreads();
  // combine the pixel-tile warps that share a channel group, in fixed order
  float* out = a.partial + (int64_t)blockIdx.x * KWT * (C + 1);
  for (int idx = threadIdx.x; idx < a.cg_per_block * CPW * KWT; idx += kThreads) {
    int g = idx / (CPW * KWT), r = idx % (CPW * KWT);
    int j = r / KWT, q = r % KWT;
    int c = (blockIdx.y * a.cg_per_block + g) * CPW + j;
    if (c < C) {
      float t = 0.f;
      for (int pp = 0; pp < a.pt_per_block; ++pp) t += s_acc[pp * a.cg_per_block + g][r];
      out[(int64_t)q * (C + 1) + c] = t;
    }
  }
  if (blockIdx.y == 0 && threadIdx.x < KWT) {
    float t = 0.f;
    for (int w = 0; w < kWarps; ++w) t += s_w[w][threadIdx.x];
    out[(int64_t)threadIdx.x * (C + 1) + C] = t;
  }
}

// ---------------------------------------------------------------------------
// v3: TMA-fed, warp-specialised class sums (the default for contiguous-pixel maps with HW % 4 == 0).
//
// The v2 kernel above issues its loads from the warps that also do the arithmetic, 16 warps per SM at
// 128 registers: with wide weight rows (soft labels x partitions) it is latency-bound at ~45 % of the HBM
// roofline.  Here the jobs are separate roles of one persistent CTA per SM, and EVERY global read is issued by the
// TMA unit into a shared-memory ring (up to 12 stages, ~200 KB in flight per SM, completion on mbarriers):
//   warp 0       producer: per stage one cp.async.bulk.tensor.3d box [128 pixels x CB channels] of the feature map
//                (x_full), plus the stage's RAW weight inputs (r_full): the [K x 128] box of soft probabilities (or the
//                planar weight rows) as a second tensor map, the 128 int64 labels and the 128 int32 partition ids as
//                1-D bulk copies
//   NBW warps    weight builders (round 2: they no longer touch global memory, so no load latency to hide and half
//                as many warps): raw inputs of the stage -> sW[stage][column][pixel]; two warps per stage, teams
//                round-robin over the stages
//   last warp    counter (channel block 0 only): sums the weights themselves -> the class-count column (folding this
//                into consumer 0 was measured in round 2: that warp becomes the straggler of every stage, 0.83 -> 0.75)
//   consumers    (as many as the channel count needs, <= NCW): warp w owns CPW channels; lane l owns pixels 4l..4l+3
//                of the stage; x and the weights come back from shared memory with conflict-free LDS.128;
//                acc[CPW][KWT] in registers for the whole sweep; every channel has exactly one owner, so the block
//                result needs no combine.  CPW = 8 for 6..10 weight columns: each consumer re-reads the stage's
//                KWT weight rows, so fat consumers halve the shared-memory traffic (LDS.128 per FMA: 16/256 vs 12/128).
// Partials and the fp64 second stage are those of v2.
// ---------------------------------------------------------------------------
constexpr int kV3ConsumerWarps = 16;
constexpr int kV3Px = 128;
constexpr int kV3MaxStages = 12;      // ring depth is chosen per shape: as many stages as fit in ~200 KB, at most this

__device__ __forceinline__ uint32_t v3_smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void v3_mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(v3_smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void v3_mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(v3_smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void v3_mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(v3_smem_u32(bar)) : "memory");
}
#ifdef SLCL_V3_DEBUG
// bring-up aid: bounded waits that say who is stuck (build with SLCL_EXTRA_NVCC_FLAGS=-DSLCL_V3_DEBUG)
__device__ __forceinline__ void v3_mbar_wait_dbg(uint64_t* bar, uint32_t parity, int role, int slot, long long it) {
  for (unsigned int spin = 0;; ++spin) {
    uint32_t ok;
    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}\n"
                 : "=r"(ok) : "r"(v3_smem_u32(bar)), "r"(parity) : "memory");
    if (ok) return;
    if (spin > (1u << 22)) {
      if ((threadIdx.x & 31) == 0)
        printf("v3 stuck: role %d warp %d block (%d,%d) slot %d it %lld parity %u\n", role, threadIdx.x >> 5, blockIdx.x, blockIdx.y,
               slot, it, parity);
      __trap();
    }
  }
}
#define V3_WAIT(bar, parity, role, slot, it) v3_mbar_wait_dbg(bar, parity, role, slot, it)
#else
#define V3_WAIT(bar, parity, role, slot, it) v3_mbar_wait(bar, parity)
#endif
__device__ __forceinline__ void v3_mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "V3_WAIT_LOOP:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra V3_WAIT_DONE;\n\t"
      "bra V3_WAIT_LOOP;\n\t"
      "V3_WAIT_DONE:\n\t"
      "}\n" ::"r"(v3_smem_u32(bar)), "r"(parity)
      : "memory");
}
__device__ __forceinline__ void v3_tma_load_3d(uint32_t smem_dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];" ::"r"(
          smem_dst),
      "l"(reinterpret_cast<uint64_t>(map)), "r"(v3_smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
// 1-D bulk copy global -> shared (16-byte aligned source, destination and size)
__device__ __forceinline__ void v3_bulk_load(uint32_t smem_dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_dst),
               "l"(reinterpret_cast<uint64_t>(src)), "r"(bytes), "r"(v3_smem_u32(bar))
               : "memory");
}

// Explicit shared-memory accesses by 32-bit shared address.  The ring is carved out of one dynamic buffer through
// pointer arithmetic the compiler cannot prove to stay in the shared window: plain C++ dereferences compile to GENERIC
// LD.E / ST.E (address translation, long-scoreboard latency) instead of LDS / STS -- the first thing ncu's source view
// showed for this kernel in round 2 (soft x 2 partitions at C = 32: 0.665 -> 0.758 of the HBM roofline from this alone).
__device__ __forceinline__ float4 v3_lds128(uint32_t addr) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
  return v;
}
// 4 consecutive floats as two packed pairs, and the packed FMA of Blackwell's FP32 pipe: {a.lo, a.hi} * {b.lo, b.hi} +
// {c.lo, c.hi} in ONE issue slot (same FMA rate, half the instructions: the sweep is issue-limited, not FMA-limited).
__device__ __forceinline__ void v3_lds2x64(uint32_t addr, unsigned long long& lo, unsigned long long& hi) {
  asm volatile("ld.shared.v2.b64 {%0, %1}, [%2];" : "=l"(lo), "=l"(hi) : "r"(addr));
}
__device__ __forceinline__ void v3_ffma2(unsigned long long& acc, unsigned long long a, unsigned long long b) {
  asm("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(acc) : "l"(a), "l"(b));
}
__device__ __forceinline__ float v3_pair_sum(unsigned long long v) {
  float lo, hi;
  asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
  return lo + hi;
}
__device__ __forceinline__ float2 v3_lds64f(uint32_t addr) {
  float2 v;
  asm volatile("ld.shared.v2.f32 {%0, %1}, [%2];" : "=f"(v.x), "=f"(v.y) : "r"(addr));
  return v;
}
__device__ __forceinline__ float v3_lds32(uint32_t addr) {
  float v;
  asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(addr));
  return v;
}
__device__ __forceinline__ int v3_lds32i(uint32_t addr) {
  int v;
  asm volatile("ld.shared.s32 %0, [%1];" : "=r"(v) : "r"(addr));
  return v;
}
__device__ __forceinline__ long long v3_lds64i(uint32_t addr) {
  long long v;
  asm volatile("ld.shared.s64 %0, [%1];" : "=l"(v) : "r"(addr));
  return v;
}
__device__ __forceinline__ void v3_sts32(uint32_t addr, float v) {
  asm volatile("st.shared.f32 [%0], %1;" ::"r"(addr), "f"(v) : "memory");
}

// ring position of iteration `it`: slot = it % n, phase = (it / n) & 1, advanced without divisions
struct V3Pos {
  int slot, phase, n;
  __device__ __forceinline__ V3Pos(int start, int n_) : slot(start), phase(0), n(n_) { norm(); }
  __device__ __forceinline__ void norm() { while (slot >= n) { slot -= n; phase ^= 1; } }
  __device__ __forceinline__ void advance(int step) { slot += step; norm(); }
};

struct __align__(8) V3Bars { uint64_t x_full[kV3MaxStages], r_full[kV3MaxStages], w_full[kV3MaxStages], empty[kV3MaxStages]; };

// per-stage shared memory: x [CB][128] fp32 | w [KWT][128] fp32 | raw [KWT][128] fp32 (soft: K probability rows; planar:
// the weight rows; hard: the first 1 KB holds 128 int64 labels) | part [128] int32
__host__ __device__ constexpr int v3_raw_rows(int kwt) { return kwt < 2 ? 2 : kwt; }

// NCW = upper bound of the consumer warps (8 or 16), NBW = builder warps: together they set the register budget.
template <int KWT, int CPW, int NCW, int NBW, bool LOGITS>
__global__ void __launch_bounds__(32 * (3 + NBW + NCW), 1)
class_sums_v3_kernel(const __grid_constant__ CUtensorMap map_feat, const __grid_constant__ CUtensorMap map_raw,
                     const SumArgs a) {
  const int kV3Stages = a.n_stages;
  const int CB = a.n_cw * CPW;                                 // channels per block
  const int kStageBytes = CB * kV3Px * 4;
  constexpr int kRawRows = v3_raw_rows(KWT);
  extern __shared__ __align__(128) uint8_t v3_smem[];
  uint8_t* base = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(v3_smem) + 127) & ~(uintptr_t)127);
  const uint32_t sX_u32 = v3_smem_u32(base);                                                // [stages][CB][128]
  const uint32_t sWt_u32 = sX_u32 + (uint32_t)(kV3Stages * kStageBytes);                    // [stages][KWT][128]
  const uint32_t sRaw_u32 = sWt_u32 + (uint32_t)(kV3Stages * KWT * kV3Px * 4);              // [stages][kRawRows][128]
  const uint32_t sPart_u32 = sRaw_u32 + (uint32_t)(kV3Stages * kRawRows * kV3Px * 4);       // [stages][128]
  V3Bars* bars = reinterpret_cast<V3Bars*>(base + (size_t)kV3Stages * ((size_t)kStageBytes + (size_t)(KWT + kRawRows + 1) * kV3Px * 4));

  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int C = (int)a.channels;
  const int c_base = blockIdx.y * CB;
  const int64_t tiles_per_image = (a.pixels + kV3Px - 1) / kV3Px;
  const int64_t n_tiles = a.batch * tiles_per_image;
  const int64_t n_iter = n_tiles > blockIdx.x ? (n_tiles - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;
  const bool ragged = (a.pixels % kV3Px) != 0;                 // the last tile of an image is short

  if (threadIdx.x == 0) {
    if (blockIdx.x == 0 && blockIdx.y == 0) *a.ticket = 0u;
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&map_feat)) : "memory");
    if (a.mode != kHard) asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&map_raw)) : "memory");
    for (int s = 0; s < kV3Stages; ++s) {
      v3_mbar_init(&bars->x_full[s], 1);
      v3_mbar_init(&bars->r_full[s], 1);
      v3_mbar_init(&bars->w_full[s], 2);
      v3_mbar_init(&bars->empty[s], a.n_cw + (blockIdx.y == 0 ? 1 : 0));      // + the counter warp of channel block 0
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();

  // tile -> (image, first pixel) without a 64-bit division per stage: the tile index advances by gridDim.x
  struct TilePos {
    int64_t b; int64_t t, step, per;
    __device__ TilePos(int64_t tile0, int64_t step_, int64_t per_) : step(step_), per(per_) { b = tile0 / per_; t = tile0 - b * per_; }
    __device__ __forceinline__ void next() { t += step; if (t >= per) { const int64_t q = t / per; b += q; t -= q * per; } }
    __device__ __forceinline__ int p0() const { return (int)(t * kV3Px); }
  };
  if (warp == 0) {
    // ===================== TMA producer 1: the feature tile =====================
    if (lane == 0) {
      V3Pos pos(0, kV3Stages);
      TilePos tp(blockIdx.x, gridDim.x, tiles_per_image);
      for (int64_t it = 0; it < n_iter; ++it, pos.advance(1), tp.next()) {
        const int s = pos.slot;
        V3_WAIT(&bars->empty[s], (uint32_t)(pos.phase ^ 1), 0, s, (long long)it);
        v3_mbar_expect_tx(&bars->x_full[s], kStageBytes);
        v3_tma_load_3d(sX_u32 + (uint32_t)(s * kStageBytes), &map_feat, &bars->x_full[s], tp.p0(), c_base, (int)tp.b);
      }
    }
  } else if (warp == 1) {
    // ===================== TMA producer 2: the raw weight inputs of the tile =====================
    if (lane == 0) {
      V3Pos pos(0, kV3Stages);
      TilePos tp(blockIdx.x, gridDim.x, tiles_per_image);
      for (int64_t it = 0; it < n_iter; ++it, pos.advance(1), tp.next()) {
        const int s = pos.slot;
        const int p0 = tp.p0();
        const int64_t b = tp.b;
        V3_WAIT(&bars->empty[s], (uint32_t)(pos.phase ^ 1), 5, s, (long long)it);
        const int valid = min(kV3Px, (int)(a.pixels - p0));                  // pixels of this tile inside the image
        uint32_t raw_bytes = 0;
        if (a.mode == kSoft) raw_bytes = (uint32_t)(a.n_class * kV3Px * 4);   // full box (out-of-image pixels zero-filled)
        else if (a.mode == kPlanar) raw_bytes = (uint32_t)(KWT * kV3Px * 4);
        else raw_bytes = (uint32_t)valid * 8u;
        if (a.part_id) raw_bytes += (uint32_t)valid * 4u;
        v3_mbar_expect_tx(&bars->r_full[s], raw_bytes);
        const uint32_t raw_dst = sRaw_u32 + (uint32_t)(s * kRawRows * kV3Px * 4);
        if (a.mode == kSoft) v3_tma_load_3d(raw_dst, &map_raw, &bars->r_full[s], p0, 0, (int)b);
        else if (a.mode == kPlanar) v3_tma_load_3d(raw_dst, &map_raw, &bars->r_full[s], p0, (int)b, 0);
        else v3_bulk_load(raw_dst, a.labels + b * a.pixels + p0, (uint32_t)valid * 8u, &bars->r_full[s]);
        if (a.part_id)
          v3_bulk_load(sPart_u32 + (uint32_t)(s * kV3Px * 4), a.part_id + b * a.pixels + p0, (uint32_t)valid * 4u,
                       &bars->r_full[s]);
      }
    }
  } else if (warp <= 1 + NBW) {
    // ===================== weight builders (shared memory -> shared memory) =====================
    // Two warps per stage (64 pixels each, 2 per lane); kTeams = NBW / 2 teams take the stages round-robin, so a team
    // has kTeams stage periods for one build.  The ring depth is a MULTIPLE of kTeams (host side): a team then meets the
    // same slots every round and sees every phase of their barriers.  (Round 1 let the depth be odd: a team met a slot
    // only every second round, its parity wait could not tell "previous round" from "two rounds ago", and it could run
    // ahead of the consumers.)
    const int wv = warp - 2;
    const int team = wv >> 1, hf = wv & 1;
    constexpr int kTeams = NBW / 2;
    constexpr int kPl = 2;                              // pixels per lane
    const bool use_thr = a.threshold > 0.f && a.threshold < 1.f;
    V3Pos bpos(team, kV3Stages);
    TilePos tp(blockIdx.x + (int64_t)team * gridDim.x, (int64_t)kTeams * gridDim.x, tiles_per_image);
    for (int64_t it = team; it < n_iter; it += kTeams, bpos.advance(kTeams), tp.next()) {
      const int s = bpos.slot;
      const int valid = ragged ? min(kV3Px, (int)(a.pixels - tp.p0())) : kV3Px;
      V3_WAIT(&bars->r_full[s], (uint32_t)bpos.phase, 1, s, (long long)it);     // raw inputs landed (and the slot's previous round is done)
      const uint32_t raw = sRaw_u32 + (uint32_t)(s * kRawRows * kV3Px * 4);
      const uint32_t prt = sPart_u32 + (uint32_t)(s * kV3Px * 4);
      const uint32_t dst = sWt_u32 + (uint32_t)((s * KWT * kV3Px + hf * 64 + lane) * 4);
#pragma unroll
      for (int i = 0; i < kPl; ++i) {
        const int px = hf * 64 + lane + 32 * i;
        const uint32_t d = dst + 32 * 4 * i;
        if (a.mode == kPlanar) {
#pragma unroll
          for (int q = 0; q < KWT; ++q) v3_sts32(d + q * kV3Px * 4, v3_lds32(raw + (uint32_t)((q * kV3Px + px) * 4)));
          continue;
        }
        // every column zero, then the (at most K) columns of the pixel's partition: no select chains, the column index
        // only ever appears in a shared-memory address
#pragma unroll
        for (int q = 0; q < KWT; ++q) v3_sts32(d + q * kV3Px * 4, 0.f);
        const bool inside = px < valid;
        const int part = (a.part_id && inside) ? v3_lds32i(prt + px * 4) : 0;
        const bool part_ok = inside && part >= 0 && part < a.n_part;
        if (a.mode == kHard) {
          // utils_.py:581 / :535
          const long long lab = inside ? v3_lds64i(raw + px * 8) : -1;
          if (part_ok && lab >= 0 && lab < a.n_class) v3_sts32(d + (uint32_t)((part * a.n_class + (int)lab) * kV3Px * 4), 1.0f);
        } else if (part_ok) {
          // soft probabilities: :517-519 (weighted) or :524-525 (arg-max one-hot); certainty :511-514
          float pr[SLCL_MAX_CLASSES];
#pragma unroll
          for (int k = 0; k < SLCL_MAX_CLASSES; ++k) pr[k] = (k < a.n_class) ? v3_lds32(raw + (uint32_t)((k * kV3Px + px) * 4)) : 0.f;
          float cert = 1.f;
          int arg = 0;
          if constexpr (LOGITS) {          // logits -> probabilities (SLCL_SOFT_LOGITS); the largest one is 1/s
            float pmax;
            softmax_inplace(pr, a.n_class, pmax, arg);
            if (use_thr) cert = pmax >= a.threshold ? 1.f : 0.f;
          } else if (use_thr || !a.weighted) {
            float best = -INFINITY;
#pragma unroll
            for (int k = 0; k < SLCL_MAX_CLASSES; ++k)
              if (k < a.n_class && pr[k] > best) { best = pr[k]; arg = k; }
            if (use_thr) cert = best >= a.threshold ? 1.f : 0.f;
          }
          const uint32_t dp = d + (uint32_t)(part * a.n_class * kV3Px * 4);
#pragma unroll
          for (int k = 0; k < SLCL_MAX_CLASSES; ++k)
            if (k < a.n_class) v3_sts32(dp + k * kV3Px * 4, a.weighted ? pr[k] * cert : ((k == arg) ? cert : 0.f));
        }
      }
      __syncwarp();
      if (lane == 0) v3_mbar_arrive(&bars->w_full[s]);
    }
  } else {
    // ===================== consumers =====================
    const int cw = warp - 2 - NBW;
    if (cw < a.n_cw) {
    // kPack: acc[j][q] = {sum over the lane's pixels 0,2 ; sum over its pixels 1,3} as one packed pair, accumulated with
    // FFMA2 (half the issue slots).  Costs 2 registers per accumulator: only where the register budget allows it.
    constexpr bool kPack = (NCW <= 8) && (CPW * KWT <= 40);
    using AccT = typename std::conditional<kPack, unsigned long long, float>::type;
    AccT acc[CPW][KWT];
#pragma unroll
    for (int q = 0; q < KWT; ++q)
#pragma unroll
      for (int j = 0; j < CPW; ++j) acc[j][q] = AccT(0);
    V3Pos cpos(0, kV3Stages);
    for (int64_t it = 0; it < n_iter; ++it, cpos.advance(1)) {
      const int s = cpos.slot;
      const uint32_t par = (uint32_t)cpos.phase;
      V3_WAIT(&bars->x_full[s], par, 2, s, (long long)it);
      const uint32_t xs = sX_u32 + (uint32_t)(s * kStageBytes + ((cw * CPW) * kV3Px + lane * 4) * 4);
      const uint32_t ws = sWt_u32 + (uint32_t)((s * KWT * kV3Px + lane * 4) * 4);
      if constexpr (kPack) {
        unsigned long long x01[CPW], x23[CPW];
#pragma unroll
        for (int j = 0; j < CPW; ++j) v3_lds2x64(xs + j * kV3Px * 4, x01[j], x23[j]);
        V3_WAIT(&bars->w_full[s], par, 3, s, (long long)it);
#pragma unroll
        for (int q = 0; q < KWT; ++q) {
          unsigned long long w01, w23;
          v3_lds2x64(ws + q * kV3Px * 4, w01, w23);
#pragma unroll
          for (int j = 0; j < CPW; ++j) {
            v3_ffma2(acc[j][q], w01, x01[j]);
            v3_ffma2(acc[j][q], w23, x23[j]);
          }
        }
      } else {
        float4 x[CPW];
#pragma unroll
        for (int j = 0; j < CPW; ++j) x[j] = v3_lds128(xs + j * kV3Px * 4);
        V3_WAIT(&bars->w_full[s], par, 3, s, (long long)it);
#pragma unroll
        for (int q = 0; q < KWT; ++q) {
          const float4 w = v3_lds128(ws + q * kV3Px * 4);
#pragma unroll
          for (int j = 0; j < CPW; ++j) {
            acc[j][q] = fmaf(w.x, x[j].x, acc[j][q]);
            acc[j][q] = fmaf(w.y, x[j].y, acc[j][q]);
            acc[j][q] = fmaf(w.z, x[j].z, acc[j][q]);
            acc[j][q] = fmaf(w.w, x[j].w, acc[j][q]);
          }
        }
      }
      __syncwarp();
      if (lane == 0) v3_mbar_arrive(&bars->empty[s]);
    }
    float* out = a.partial + (int64_t)blockIdx.x * KWT * (C + 1);
#pragma unroll
    for (int j = 0; j < CPW; ++j) {
      const int c = c_base + cw * CPW + j;
#pragma unroll
      for (int q = 0; q < KWT; ++q) {
        float t;
        if constexpr (kPack) t = v3_pair_sum(acc[j][q]); else t = acc[j][q];
        const float r = warp_sum(t);
        if (lane == 0 && c < C) out[(int64_t)q * (C + 1) + c] = r;
      }
    }
    } else if (cw == a.n_cw && blockIdx.y == 0) {
      // ===================== counter: the weight-sum ("class count") column =====================
      // sums of the weights themselves, read back like a consumer does (exact integers for hard labels)
      float cacc[KWT];
#pragma unroll
      for (int q = 0; q < KWT; ++q) cacc[q] = 0.f;
      V3Pos cpos(0, kV3Stages);
      for (int64_t it = 0; it < n_iter; ++it, cpos.advance(1)) {
        const int s = cpos.slot;
        V3_WAIT(&bars->w_full[s], (uint32_t)cpos.phase, 4, s, (long long)it);
        const uint32_t ws = sWt_u32 + (uint32_t)((s * KWT * kV3Px + lane * 4) * 4);
#pragma unroll
        for (int q = 0; q < KWT; ++q) {
          const float4 w = v3_lds128(ws + q * kV3Px * 4);
          cacc[q] += (w.x + w.y) + (w.z + w.w);
        }
        __syncwarp();
        if (lane == 0) v3_mbar_arrive(&bars->empty[s]);
      }
      float* out = a.partial + (int64_t)blockIdx.x * KWT * (C + 1);
#pragma unroll
      for (int q = 0; q < KWT; ++q) {
        const float r = warp_sum(cacc[q]);
        if (lane == 0) out[(int64_t)q * (C + 1) + C] = r;
      }
    }
  }
}

// ---------------------------------------------------------------------------
// Fused target step (SURVEY.md 8(f)-1): generate_pseudo_label (utils/utils_.py:597-624) + the target-side
// mpcl_loss_calc forward (trainer/Trainer_MPSCL.py:135,144) + the per-class sums of the SAME target map under the pseudo
// labels just generated (the hard target centroids of cal_centroid, utils/utils_.py:524-529 with the map's own arg-max
// labels) -- in ONE pass over F_t.  The class-sum ring above already has every pixel's full channel vector in shared
// memory, so the weight builders become "pixel warps": one pixel per lane, they walk the stage's C channel rows,
// form the cosines against the unit centres, derive label / selection mask / loss row / backward stash exactly as
// proto_fwd_kernel's fused-target path does (same fmaf order over the channels, so labels, masks and the stash are
// bit-identical), write the one-hot weight row, and the consumers accumulate the class sums from the same stage.
//   warp 0: TMA producer   warps 1..8: pixel warps (teams of two, round robin over the stages)   then n_cw consumers, 1 counter
// Needs all C channels in one stage: C <= 16 * CPW (CPW = 4 or 8).
// ---------------------------------------------------------------------------
struct TileArgs {
  const float* feat;
  int64_t batch, channels, pixels, n_total;
  const float* cstate;        // unit centres [K*C] (prep_centres_kernel)
  MarginConst mc;
  float sel_threshold;
  int weight_by_sel;          // class-sum weights: one-hot(label) * sel instead of one-hot(label)
  int64_t* out_label;
  float* out_sel;
  float* stash;               // [(K+1) * N]
  double2* loss_partial;      // [gridDim.x] {sum sel*row, sum sel}
  float* partial;             // class sums per block [gridDim.x][K][C+1]
  unsigned int* ticket;
  int n_cw, n_stages, n_teams, wide;
};
// Stages are 64 pixels x C channels (half the class-sum kernel's tile): the pixel work is latency-bound per warp -- a
// serial walk over the channels, then ~300 dependent instructions of margin arithmetic -- so what sets the speed is how
// many pixel warps are in flight on DIFFERENT stages, and that takes a deep ring of small stages (with 128-pixel stages
// C = 128 leaves room for three, and one team of pixel warps: 318 us at cfg2, every role waiting on another; an
// explicit suspend-time hint on the mbarrier waits changed nothing, and four pixels per lane -- fewer shared loads per
// FMA but a third of the warps -- was slower, 368 us).
// Pixel warps come in teams of two (32 pixels per warp, one per lane); a.n_teams (2..4) teams take the stages round
// robin, and the ring depth is a multiple of n_teams so a team always meets the same slots and sees every phase of
// their barriers.  Consumers own CPW channels and two pixels per lane.
constexpr int kTPx = 64;                 // pixels per stage of the fused target kernel
// Up to 6 teams (12 pixel warps) next to <= 8 consumer warps (C <= 64 at CPW = 8, C <= 32 at CPW = 4), 4 teams next to 16.
__host__ __device__ constexpr int tile_teams_max(int ncw_max) { return ncw_max <= 8 ? 6 : 4; }
template <int K, int CPW, int NCWMAX>
__global__ void __launch_bounds__(32 * (2 + 2 * tile_teams_max(NCWMAX) + NCWMAX), 1)
target_tile_kernel(const __grid_constant__ CUtensorMap map_feat, const TileArgs a) {
  constexpr int kTilePixelWarps = 2 * tile_teams_max(NCWMAX);
  const int kTeams = a.n_teams;
  constexpr int KP = K <= 4 ? 4 : 8;
  const int C = (int)a.channels;
  const int kStages = a.n_stages;
  const int kStageBytes = C * kTPx * 4;
  extern __shared__ __align__(128) uint8_t v3_smem[];
  const uint32_t pad = (128u - (v3_smem_u32(v3_smem) & 127u)) & 127u;                       // align the carve-up to 128 bytes
  uint8_t* base = v3_smem + pad;
  const uint32_t sX_u32 = v3_smem_u32(base);                                               // [stages][C][64]
  const uint32_t sWt_u32 = sX_u32 + (uint32_t)(kStages * kStageBytes);                     // [stages][K][64]
  const uint32_t sC_u32 = sWt_u32 + (uint32_t)(kStages * K * kTPx * 4);                    // [C][KP] unit centres
  const size_t sC_off = (size_t)kStages * ((size_t)kStageBytes + (size_t)K * kTPx * 4);
  V3Bars* bars = reinterpret_cast<V3Bars*>(base + (size_t)kStages * ((size_t)kStageBytes + (size_t)K * kTPx * 4) +
                                           (size_t)C * KP * 4);
  __shared__ double s_red[2][kTilePixelWarps];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int64_t tiles_per_image = (a.pixels + kTPx - 1) / kTPx;
  const int64_t n_tiles = a.batch * tiles_per_image;
  const int64_t n_iter = n_tiles > blockIdx.x ? (n_tiles - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;

  pdl_trigger();
  pdl_wait();                                   // cstate comes from prep_centres_kernel in front of us
  for (int idx = threadIdx.x; idx < C * KP; idx += blockDim.x) {
    const int c = idx / KP, k = idx % KP;
    v3_sts32(sC_u32 + idx * 4, (k < K) ? a.cstate[(int64_t)k * C + c] : 0.f);
  }
  if (threadIdx.x == 0) {
    if (blockIdx.x == 0) *a.ticket = 0u;
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&map_feat)) : "memory");
    for (int s = 0; s < kStages; ++s) {
      v3_mbar_init(&bars->x_full[s], 1);
      v3_mbar_init(&bars->w_full[s], 2);
      v3_mbar_init(&bars->empty[s], a.n_cw + 1);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  struct TilePos {
    int64_t b; int64_t t, step, per;
    __device__ TilePos(int64_t tile0, int64_t step_, int64_t per_) : step(step_), per(per_) { b = tile0 / per_; t = tile0 - b * per_; }
    __device__ __forceinline__ void next() { t += step; if (t >= per) { const int64_t q = t / per; b += q; t -= q * per; } }
    __device__ __forceinline__ int p0() const { return (int)(t * kTPx); }
  };

  if (warp == 0) {
    if (lane == 0) {
      V3Pos pos(0, kStages);
      TilePos tp(blockIdx.x, gridDim.x, tiles_per_image);
      for (int64_t it = 0; it < n_iter; ++it, pos.advance(1), tp.next()) {
        const int s = pos.slot;
        v3_mbar_wait(&bars->empty[s], (uint32_t)(pos.phase ^ 1));
        v3_mbar_expect_tx(&bars->x_full[s], kStageBytes);
        v3_tma_load_3d(sX_u32 + (uint32_t)(s * kStageBytes), &map_feat, &bars->x_full[s], tp.p0(), 0, (int)tp.b);
      }
    }
  } else if (warp <= kTilePixelWarps) {
    // ===================== pixel warps: cosines, pseudo label, loss row, stash, one-hot weights =====================
    const int team = (warp - 1) >> 1;
    const int px = ((warp - 1) & 1) * 32 + lane;
    double loss_acc = 0.0, sel_acc = 0.0;
    if (team < kTeams) {
      V3Pos bpos(team, kStages);
      TilePos tp(blockIdx.x + (int64_t)team * gridDim.x, (int64_t)kTeams * gridDim.x, tiles_per_image);
      for (int64_t it = team; it < n_iter; it += kTeams, bpos.advance(kTeams), tp.next()) {
        const int s = bpos.slot;
        const int p0 = tp.p0();
        const bool inside = (int64_t)p0 + px < a.pixels;
        v3_mbar_wait(&bars->x_full[s], (uint32_t)bpos.phase);
        // plain C++ loads through pointers that stay in the shared window (offsets from the extern array itself), so the
        // compiler emits LDS AND may software-pipeline them across the unrolled channel loop
        const float* xs = reinterpret_cast<const float*>(v3_smem + pad + (size_t)s * kStageBytes) + px;
        const float4* cs = reinterpret_cast<const float4*>(v3_smem + pad + sC_off);
        float nrm = 0.f, dot[K];
#pragma unroll
        for (int k = 0; k < K; ++k) dot[k] = 0.f;
#pragma unroll 8
        for (int c = 0; c < C; ++c) {
          const float x = xs[c * kTPx];
          float ck[8];
          { const float4 t = cs[c * (KP / 4)]; ck[0] = t.x; ck[1] = t.y; ck[2] = t.z; ck[3] = t.w; }
          if constexpr (K > 4) { const float4 t = cs[c * (KP / 4) + 1]; ck[4] = t.x; ck[5] = t.y; ck[6] = t.z; ck[7] = t.w; }
          nrm = fmaf(x, x, nrm);
#pragma unroll
          for (int k = 0; k < K; ++k) dot[k] = fmaf(x, ck[k], dot[k]);
        }
        // generate_pseudo_label on the cosines (same arithmetic as pseudo_label_kernel / proto_fwd_kernel's fused path)
        const float n = fmaxf(sqrtf(nrm), 1e-12f);
        float t1 = -INFINITY, t2 = -INFINITY;
        int best = 0;
#pragma unroll
        for (int k = 0; k < K; ++k) {
          const float cs_ = dot[k] / n;
          if (cs_ > t1) { t2 = t1; t1 = cs_; best = k; }
          else if (cs_ > t2) { t2 = cs_; }
        }
        const float selv = (t1 - t2 > a.sel_threshold) ? 1.0f : 0.0f;
        const float inv_n = 1.0f / n;
        float cosv[K], M[K], coef[K + 1];
#pragma unroll
        for (int k = 0; k < K; ++k) { cosv[k] = dot[k] * inv_n; M[k] = (best == k) ? 1.0f : 0.0f; }
        const float row = margin_row<K>(cosv, M, selv, inv_n, a.mc, coef);
        const uint32_t wd = sWt_u32 + (uint32_t)((s * K * kTPx + px) * 4);
        const float wsel = a.weight_by_sel ? selv : 1.0f;
#pragma unroll
        for (int k = 0; k < K; ++k) v3_sts32(wd + (uint32_t)(k * kTPx * 4), (inside && best == k) ? wsel : 0.f);
        if (inside) {
          const int64_t pix = tp.b * a.pixels + p0 + px;
          a.out_label[pix] = best;
          a.out_sel[pix] = selv;
#pragma unroll
          for (int k = 0; k <= K; ++k) a.stash[(int64_t)k * a.n_total + pix] = coef[k];
          loss_acc += (double)(selv * row);
          sel_acc += (double)selv;
        }
        __syncwarp();
        if (lane == 0) v3_mbar_arrive(&bars->w_full[s]);
      }
    }
    loss_acc = warp_sum(loss_acc);
    sel_acc = warp_sum(sel_acc);
    if (lane == 0) { s_red[0][warp - 1] = loss_acc; s_red[1][warp - 1] = sel_acc; }
    asm volatile("bar.sync 1, %0;" ::"n"(32 * kTilePixelWarps) : "memory");         // the pixel warps only
    if (warp == 1 && lane == 0) {
      double l = 0.0, sv = 0.0;
#pragma unroll
      for (int w = 0; w < kTilePixelWarps; ++w) { l += s_red[0][w]; sv += s_red[1][w]; }
      a.loss_partial[blockIdx.x] = make_double2(l, sv);
    }
  } else {
    const int cw = warp - 1 - kTilePixelWarps;
    if (cw < a.n_cw) {
      // ===================== consumers =====================
      // a.wide == 0: CPW channels per warp, two pixels per lane.  a.wide == 1 (C > 64): 2 x CPW channels per warp -- each
      // half warp owns CPW of them and four pixels per lane -- so 8 consumer warps cover 128 channels and leave room
      // for six teams of pixel warps; the consumers have the slack (they wait most of the time), the pixel warps do not.
      float acc[CPW][K];
#pragma unroll
      for (int q = 0; q < K; ++q)
#pragma unroll
        for (int j = 0; j < CPW; ++j) acc[j][q] = 0.f;
      const int half = lane >> 4, l16 = lane & 15;
      const int c_first = a.wide ? cw * 2 * CPW + half * CPW : cw * CPW;
      const uint32_t px_off = (uint32_t)((a.wide ? l16 * 4 : lane * 2) * 4);
      V3Pos cpos(0, kStages);
      for (int64_t it = 0; it < n_iter; ++it, cpos.advance(1)) {
        const int s = cpos.slot;
        const uint32_t par = (uint32_t)cpos.phase;
        v3_mbar_wait(&bars->x_full[s], par);
        v3_mbar_wait(&bars->w_full[s], par);
        const uint32_t xs = sX_u32 + (uint32_t)(s * kStageBytes + c_first * kTPx * 4) + px_off;
        const uint32_t ws = sWt_u32 + (uint32_t)(s * K * kTPx * 4) + px_off;
        if (a.wide) {
          float4 w[K];
#pragma unroll
          for (int q = 0; q < K; ++q) w[q] = v3_lds128(ws + q * kTPx * 4);
#pragma unroll
          for (int j = 0; j < CPW; ++j) {
            const float4 x = v3_lds128(xs + j * kTPx * 4);
#pragma unroll
            for (int q = 0; q < K; ++q) {
              acc[j][q] = fmaf(w[q].x, x.x, acc[j][q]);
              acc[j][q] = fmaf(w[q].y, x.y, acc[j][q]);
              acc[j][q] = fmaf(w[q].z, x.z, acc[j][q]);
              acc[j][q] = fmaf(w[q].w, x.w, acc[j][q]);
            }
          }
        } else {
          float2 w[K];
#pragma unroll
          for (int q = 0; q < K; ++q) w[q] = v3_lds64f(ws + q * kTPx * 4);
#pragma unroll
          for (int j = 0; j < CPW; ++j) {
            const float2 x = v3_lds64f(xs + j * kTPx * 4);
#pragma unroll
            for (int q = 0; q < K; ++q) {
              acc[j][q] = fmaf(w[q].x, x.x, acc[j][q]);
              acc[j][q] = fmaf(w[q].y, x.y, acc[j][q]);
            }
          }
        }
        __syncwarp();
        if (lane == 0) v3_mbar_arrive(&bars->empty[s]);
      }
      float* out = a.partial + (int64_t)blockIdx.x * K * (C + 1);
#pragma unroll
      for (int j = 0; j < CPW; ++j) {
        const int c = c_first + j;
#pragma unroll
        for (int q = 0; q < K; ++q) {
          float r = acc[j][q];
          if (a.wide) {          // the two halves hold different channels: reduce within 16 lanes
#pragma unroll
            for (int o = 8; o > 0; o >>= 1) r += __shfl_xor_sync(0xffffffffu, r, o);
            if (l16 == 0 && c < C) out[(int64_t)q * (C + 1) + c] = r;
          } else {
            r = warp_sum(r);
            if (lane == 0 && c < C) out[(int64_t)q * (C + 1) + c] = r;
          }
        }
      }
    } else if (cw == a.n_cw) {
      // ===================== counter =====================
      float cacc[K];
#pragma unroll
      for (int q = 0; q < K; ++q) cacc[q] = 0.f;
      V3Pos cpos(0, kStages);
      for (int64_t it = 0; it < n_iter; ++it, cpos.advance(1)) {
        const int s = cpos.slot;
        v3_mbar_wait(&bars->w_full[s], (uint32_t)cpos.phase);
        const uint32_t ws = sWt_u32 + (uint32_t)((s * K * kTPx + lane * 2) * 4);
#pragma unroll
        for (int q = 0; q < K; ++q) {
          const float2 w = v3_lds64f(ws + q * kTPx * 4);
          cacc[q] += w.x + w.y;
        }
        __syncwarp();
        if (lane == 0) v3_mbar_arrive(&bars->empty[s]);
      }
      float* out = a.partial + (int64_t)blockIdx.x * K * (C + 1);
#pragma unroll
      for (int q = 0; q < K; ++q) {
        const float r = warp_sum(cacc[q]);
        if (lane == 0) out[(int64_t)q * (C + 1) + C] = r;
      }
    }
  }
}

// Finaliser folded into the reduce kernel (its last block runs it): 0 none, 1 EMA class centres
// (utils_.py:585-592), 2 centroids (utils_.py:520-523 / :538, EMA :552-563).
enum FinMode { kFinNone = 0, kFinEma = 1, kFinCentroid = 2 };
struct FinArgs {
  int mode;
  const float* prev;     // kFinEma: old centres [K,C]; kFinCentroid: previous centroid [K,C] or null
  float m;               // EMA momentum
  int K;                 // classes (rows of prev)
  float* out;            // [rows, C]
  float* inv_w;          // kFinCentroid: [rows]
};

__device__ __forceinline__ void finalize_rows(const double* sums, const FinArgs& fin, int rows, int C, int first, int step) {
  for (int idx = first; idx < rows * C; idx += step) {
    const int r = idx / C, c = idx % C;
    const double cnt = __ldcg(sums + (int64_t)r * (C + 1) + C);
    const double sv = __ldcg(sums + (int64_t)r * (C + 1) + c);
    if (fin.mode == kFinEma) {
      const float old = fin.prev[idx];
      float batch;
      if (cnt == 0.0) batch = old;                                              // :585-586
      else batch = (float)sv / (float)cnt;                                      // :588
      fin.out[idx] = fin.m * old + (1.0f - fin.m) * batch;                      // :592
    } else {
      const float wsum = (float)cnt + 1e-7f;
      float mu = (float)sv / wsum;
      if (fin.prev != nullptr) mu = fin.m * fin.prev[(r % fin.K) * C + c] + (1.0f - fin.m) * mu;
      fin.out[idx] = mu;
      if (c == 0) fin.inv_w[r] = 1.0f / wsum;
    }
  }
}

// sums[col][c] = sum over blocks in fp64.  One warp per output element: lane l adds blocks l, l+32, ...
// then a fixed-shape shuffle tree, so the result is deterministic and the serial chain is n_blocks/32 long.
// PEER: the element is then all-reduced over the ranks through the NVLink mailboxes (peer.cuh) by the same warp --
// the only cross-GPU exchange of the class-centre / centroid path, with no collective launch.  The block that
// finishes last runs the finaliser over the complete `sums`.
template <bool PEER>
__global__ void __launch_bounds__(kThreads) class_sums_reduce_kernel(const float* partial, int n_blocks, int kwt,
                                                                     int n_cols, int C, double* sums, const PeerCtx pc,
                                                                     const FinArgs fin, unsigned int* ticket) {
  __shared__ int s_last;
  const int lane = threadIdx.x & 31;
  const int idx = blockIdx.x * kWarps + (threadIdx.x >> 5);
  const int row = C + 1;
  unsigned int e = 0u;
  if constexpr (PEER) e = peer_epoch_begin(pc);
  if (idx < n_cols * row) {
    const int col = idx / row, c = idx % row;
    double t = 0.0;
    for (int b = lane; b < n_blocks; b += 32) t += (double)partial[((int64_t)b * kwt + col) * row + c];
    t = warp_sum(t);
    if constexpr (PEER) t = peer_warp_allreduce(pc, e, idx, t);
    if (lane == 0) sums[idx] = t;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    bool last;
    if constexpr (PEER) last = peer_epoch_end(pc, e, gridDim.x);
    else {
      __threadfence();
      last = atomicAdd(ticket, 1u) == gridDim.x - 1;
      if (last) *ticket = 0u;
    }
    s_last = last ? 1 : 0;
  }
  __syncthreads();
  if (!s_last || fin.mode == kFinNone) return;
  __threadfence();
  finalize_rows(sums, fin, n_cols, C, threadIdx.x, kThreads);
}

// utils_.py:585-592
__global__ void __launch_bounds__(kThreads) ema_finalize_kernel(const double* sums, const float* old_c, float m, int K,
                                                                int C, float* out) {
  FinArgs fin{kFinEma, old_c, m, K, out, nullptr};
  finalize_rows(sums, fin, K, C, blockIdx.x * kThreads + threadIdx.x, gridDim.x * kThreads);
}

// utils_.py:520-523 / :538 and EMA :552-563
__global__ void __launch_bounds__(kThreads) centroid_finalize_kernel(const double* sums, const float* prev, float mom,
                                                                     int rows, int K, int C, float* cen, float* inv_w) {
  FinArgs fin{kFinCentroid, prev, mom, K, cen, inv_w};
  finalize_rows(sums, fin, rows, C, blockIdx.x * kThreads + threadIdx.x, gridDim.x * kThreads);
}

// ---------------------------------------------------------------------------
// centroid backward (A.4):  dfeat = sum_j w_ij gc_j ;  dprobs_ik = cert*[part]*(x_i.gc_j - mu_j.gc_j)
// ---------------------------------------------------------------------------
struct CenBwdArgs {
  SumArgs s;
  const float* gc;          // [cols][C]
  const float* mu_dot_gc;   // [cols]
  float* dfeat;
  float* dprobs;            // [B,K,HW] or null
};

// gc_j = dL/dcentroid_j * ema_scale / (W_j + 1e-7);  mu_dot_gc_j = mu_j . gc_j  with mu_j = S_j / (W_j + 1e-7)
// One block per row j; grad(i) is dL/dcentroid at flat index i = j * C + c.
template <class Grad>
__device__ __forceinline__ void centroid_bwd_prep_row(Grad grad, const double* sums, float ema_scale, int C, int j, float* gc,
                                                      float* mu_dot_gc) {
  __shared__ float red[kWarps];
  const float wsum = (float)sums[(int64_t)j * (C + 1) + C] + 1e-7f;
  float acc = 0.f;
  for (int c = threadIdx.x; c < C; c += kThreads) {
    const float g = grad((int64_t)j * C + c) * ema_scale / wsum;
    const float mu = (float)sums[(int64_t)j * (C + 1) + c] / wsum;
    gc[(int64_t)j * C + c] = g;
    acc = fmaf(mu, g, acc);
  }
  acc = warp_sum(acc);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    float t = 0.f;
    for (int w = 0; w < kWarps; ++w) t += red[w];
    mu_dot_gc[j] = t;
  }
}

__global__ void __launch_bounds__(kThreads) centroid_bwd_prep_kernel(const float* grad_cen, const double* sums,
                                                                     float ema_scale, int C, float* gc, float* mu_dot_gc) {
  centroid_bwd_prep_row([=](int64_t i) { return grad_cen[i]; }, sums, ema_scale, C, blockIdx.x, gc, mu_dot_gc);
}

template <int KWT> constexpr int kwpad() { return (KWT + 3) / 4 * 4; }
constexpr int kCenRing = 8;         // channels in flight per thread in the centroid backward (cp.async ring; a power of two)

template <int KWT, int VEC, bool HAS_DP, bool LOGITS>
__global__ void __launch_bounds__(kThreads) centroid_bwd_kernel(const CenBwdArgs a) {
  constexpr int KP = kwpad<KWT>();
  extern __shared__ __align__(16) float sG[];        // [C][KP]
  const int C = (int)a.s.channels;
  for (int idx = threadIdx.x; idx < C * KP; idx += kThreads) {
    int c = idx / KP, j = idx % KP;
    sG[idx] = (j < a.s.n_cols) ? a.gc[(int64_t)j * C + c] : 0.f;
  }
  __syncthreads();
  const int64_t g = (int64_t)blockIdx.x * kThreads + threadIdx.x;
  const int64_t groups = a.s.pixels / VEC;
  if (g >= a.s.batch * groups) return;
  const int64_t b = g / groups;
  const int64_t p = (g - b * groups) * VEC;
  const int64_t pix = b * a.s.pixels + p;
  float w[VEC][KWT];
  build_weights<KWT, VEC, LOGITS>(a.s, b, p, pix, w);
  const float* src = a.s.feat + b * a.s.sb + p * a.s.sp;
  float* dst = a.dfeat + b * a.s.sb + p * a.s.sp;
  float dot[HAS_DP ? KWT : 1][VEC];
#pragma unroll
  for (int j = 0; j < (HAS_DP ? KWT : 1); ++j)
#pragma unroll
    for (int v = 0; v < VEC; ++v) dot[j][v] = 0.f;

  constexpr int U = 4;
  // With soft labels the kernel also reads x (for d probs).  Those loads go through a per-thread cp.async ring in
  // shared memory, kCenRing channels deep (each thread copies and later reads only its own 16 bytes, so no barrier is
  // involved): ~48 KB per block in flight without spending registers on it.
  constexpr bool kRing = HAS_DP && VEC == 4;
  float4* ring = reinterpret_cast<float4*>(sG + (size_t)((C * KP + 3) / 4 * 4));
  auto ring_fetch = [&](int c) {
    if (c < C) {
      const uint32_t dst_s = (uint32_t)__cvta_generic_to_shared(ring + (size_t)(c % kCenRing) * kThreads + threadIdx.x);
      asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst_s), "l"(src + (int64_t)c * a.s.sc) : "memory");
    }
    asm volatile("cp.async.commit_group;" ::: "memory");          // one group per channel, empty past the end
  };
  if constexpr (kRing) {
    for (int c = 0; c < kCenRing; ++c) ring_fetch(c);
  }
  for (int c = 0; c < C; c += U) {
    float x[U][VEC];
    if constexpr (HAS_DP && !kRing) {
#pragma unroll
      for (int u = 0; u < U; ++u) {
        if (c + u < C) ld_vec<VEC>(src + (int64_t)(c + u) * a.s.sc, x[u]);
      }
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      if (c + u < C) {
        if constexpr (kRing) {
          asm volatile("cp.async.wait_group %0;" ::"n"(kCenRing - 1) : "memory");
          const float4 t = ring[(size_t)((c + u) % kCenRing) * kThreads + threadIdx.x];
          x[u][0] = t.x; x[u][1] = t.y; x[u][2] = t.z; x[u][3] = t.w;
          ring_fetch(c + u + kCenRing);
        }
        float gj[KP];
        const float4* row = reinterpret_cast<const float4*>(sG + (size_t)(c + u) * KP);
#pragma unroll
        for (int q = 0; q < KP / 4; ++q) { float4 t = row[q]; gj[4 * q] = t.x; gj[4 * q + 1] = t.y; gj[4 * q + 2] = t.z; gj[4 * q + 3] = t.w; }
        float o[VEC];
#pragma unroll
        for (int v = 0; v < VEC; ++v) {
          float t = 0.f;
#pragma unroll
          for (int j = 0; j < KWT; ++j) t = fmaf(w[v][j], gj[j], t);
          o[v] = t;
          if constexpr (HAS_DP) {
#pragma unroll
            for (int j = 0; j < KWT; ++j) dot[j][v] = fmaf(x[u][v], gj[j], dot[j][v]);
          }
        }
        st_vec<VEC>(dst + (int64_t)(c + u) * a.s.sc, o);
      }
    }
  }
  if constexpr (HAS_DP && LOGITS) {
    // d z_ik = p_ik * (g_ik - sum_m p_im g_im),  g_ik = cert_i * (x_i.gc_j - mu_j.gc_j),  j = part_i*K + k.  The weight row
    // holds p_ik * cert_i in the pixel's K columns and zeros elsewhere, so with S_i = sum_j w_ij (x_i.gc_j - mu_j.gc_j) over
    // every column, column j of the pixel's partition gives w_ij (x_i.gc_j - mu_j.gc_j - S_i) = d z_ik, certainty included.
    const int K = a.s.n_class;
    int part[VEC];
    float S[VEC];
#pragma unroll
    for (int v = 0; v < VEC; ++v) {
      part[v] = a.s.part_id ? a.s.part_id[pix + v] : 0;
      S[v] = 0.f;
#pragma unroll
      for (int j = 0; j < KWT; ++j) {
        dot[j][v] -= (j < a.s.n_cols) ? a.mu_dot_gc[j] : 0.f;
        S[v] = fmaf(w[v][j], dot[j][v], S[v]);
      }
    }
#pragma unroll
    for (int k = 0; k < SLCL_MAX_CLASSES; ++k) {
      if (k < K) {
        float o[VEC];
#pragma unroll
        for (int v = 0; v < VEC; ++v) {
          const int col = part[v] * K + k;
          float val = 0.f;
#pragma unroll
          for (int j = 0; j < KWT; ++j) val = (j == col) ? w[v][j] * (dot[j][v] - S[v]) : val;
          o[v] = val;
        }
        st_vec<VEC>(a.dprobs + (b * K + k) * a.s.pixels + p, o);
      }
    }
  } else if constexpr (HAS_DP) {
    // d w_ij / d p_ik = cert_i * [part_i == j / K]  (weighted soft labels only)
    const int K = a.s.n_class;
    const bool use_thr = a.s.threshold > 0.f && a.s.threshold < 1.f;
    float cert[VEC];
    int part[VEC];
#pragma unroll
    for (int v = 0; v < VEC; ++v) { cert[v] = 1.f; part[v] = a.s.part_id ? a.s.part_id[pix + v] : 0; }
    if (use_thr) {
      float pr_max[VEC];
#pragma unroll
      for (int v = 0; v < VEC; ++v) pr_max[v] = -INFINITY;
      for (int k = 0; k < K; ++k) {
        float t[VEC];
        ld_vec_keep<VEC>(a.s.probs + (b * K + k) * a.s.pixels + p, t);
#pragma unroll
        for (int v = 0; v < VEC; ++v) pr_max[v] = fmaxf(pr_max[v], t[v]);
      }
#pragma unroll
      for (int v = 0; v < VEC; ++v) cert[v] = (pr_max[v] >= a.s.threshold) ? 1.f : 0.f;
    }
#pragma unroll
    for (int v = 0; v < VEC; ++v)
      if (part[v] < 0 || part[v] >= a.s.n_part) cert[v] = 0.f;
    // statically indexed selection of column part*K + k (keeps dot[][] in registers)
#pragma unroll
    for (int k = 0; k < SLCL_MAX_CLASSES; ++k) {
      if (k < K) {
        float o[VEC];
#pragma unroll
        for (int v = 0; v < VEC; ++v) {
          const int col = part[v] * K + k;
          float val = 0.f;
#pragma unroll
          for (int j = 0; j < KWT; ++j) val = (j == col) ? dot[j][v] - a.mu_dot_gc[j] : val;
          o[v] = cert[v] * val;
        }
        st_vec<VEC>(a.dprobs + (b * K + k) * a.s.pixels + p, o);
      }
    }
  }
}

// ---------------------------------------------------------------------------
// centroid backward, round-2 form for 128-bit maps (HW % 4 == 0): same arithmetic as centroid_bwd_kernel with
//   * the weight rows and the d-probs gather placed through a THREAD-PRIVATE shared scratch [KWT][threads] float4
//     (a dynamic column index becomes a shared-memory address; the round-1 kernel resolved it with KWT x K predicated
//     moves per pixel in the prologue and again in the epilogue -- 19 % + 6 % of its stall samples in ncu's source view),
//   * packed FFMA2 arithmetic over pixel pairs: per channel 32 packed FMAs instead of 64 scalar ones; gc sits in shared
//     memory pre-duplicated as {g, g} pairs so the broadcast load already has the packed form.
// ---------------------------------------------------------------------------
__device__ __forceinline__ uint32_t cb_smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void cb_sts128(uint32_t addr, float4 v) {
  asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}
__device__ __forceinline__ void cb_sts32(uint32_t addr, float v) { asm volatile("st.shared.f32 [%0], %1;" ::"r"(addr), "f"(v) : "memory"); }
__device__ __forceinline__ float cb_lds32(uint32_t addr) { float v; asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(addr)); return v; }
__device__ __forceinline__ void cb_lds2x64(uint32_t addr, unsigned long long& lo, unsigned long long& hi) {
  asm volatile("ld.shared.v2.b64 {%0, %1}, [%2];" : "=l"(lo), "=l"(hi) : "r"(addr));
}
__device__ __forceinline__ void cb_ffma2(unsigned long long& acc, unsigned long long a, unsigned long long b) {
  asm("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(acc) : "l"(a), "l"(b));
}
__device__ __forceinline__ unsigned long long cb_fmul2(unsigned long long a, unsigned long long b) {
  unsigned long long d;
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
  return d;
}
__device__ __forceinline__ float2 cb_unpack(unsigned long long v) {
  float2 r;
  asm("mov.b64 {%0, %1}, %2;" : "=f"(r.x), "=f"(r.y) : "l"(v));
  return r;
}

template <int KWT, bool HAS_DP, bool LOGITS>
__global__ void __launch_bounds__(kThreads, 2) centroid_bwd4_kernel(const CenBwdArgs a) {
  constexpr int KP = (KWT + 1) / 2 * 2;               // gc pairs are fetched two columns (one LDS.128) at a time
  extern __shared__ __align__(16) float cb_smem[];    // sG2 [C][KP] {g, g} pairs | scratch [KWT][threads] float4 | x ring
  const int C = (int)a.s.channels;
  const uint32_t sG2 = cb_smem_u32(cb_smem);
  const uint32_t scratch = sG2 + (uint32_t)(C * KP * 8) + threadIdx.x * 16;                   // + j * kThreads * 16
  const uint32_t ring = sG2 + (uint32_t)(C * KP * 8) + (uint32_t)(KWT * kThreads * 16) + threadIdx.x * 16;   // + slot * kThreads * 16
  for (int idx = threadIdx.x; idx < C * KP; idx += kThreads) {
    const int c = idx / KP, j = idx % KP;
    const float g = (j < a.s.n_cols) ? a.gc[(int64_t)j * C + c] : 0.f;
    reinterpret_cast<float2*>(cb_smem)[idx] = make_float2(g, g);
  }
  __syncthreads();
  const int64_t gidx = (int64_t)blockIdx.x * kThreads + threadIdx.x;
  const int64_t groups = a.s.pixels / 4;
  if (gidx >= a.s.batch * groups) return;
  const int64_t b = gidx / groups;
  const int64_t p = (gidx - b * groups) * 4;
  const int64_t pix = b * a.s.pixels + p;
  const float* src = a.s.feat + b * a.s.sb + p * a.s.sp;
  float* dst = a.dfeat + b * a.s.sb + p * a.s.sp;
  const int K = a.s.n_class;

  // x loads (needed for d probs only) go through a per-thread cp.async ring, kCenRing channels deep
  auto ring_fetch = [&](int c) {
    if (c < C) asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(ring + (uint32_t)((c % kCenRing) * kThreads * 16)),
                            "l"(src + (int64_t)c * a.s.sc) : "memory");
    asm volatile("cp.async.commit_group;" ::: "memory");          // one group per channel, empty past the end
  };
  if constexpr (HAS_DP) {
    for (int c = 0; c < kCenRing; ++c) ring_fetch(c);
  }

  // ---- weight rows of the 4 pixels -> scratch[column][pixel] (zero, then the <= K columns of each pixel's partition)
  int base[4];                                        // first column of the pixel's partition, or -1
  float cert[4];
  {
    int part[4] = {0, 0, 0, 0};
    if (a.s.part_id) { const int4 t = *reinterpret_cast<const int4*>(a.s.part_id + pix); part[0] = t.x; part[1] = t.y; part[2] = t.z; part[3] = t.w; }
#pragma unroll
    for (int j = 0; j < KWT; ++j) cb_sts128(scratch + (uint32_t)(j * kThreads * 16), make_float4(0.f, 0.f, 0.f, 0.f));
#pragma unroll
    for (int v = 0; v < 4; ++v) { base[v] = (part[v] >= 0 && part[v] < a.s.n_part) ? part[v] * K : -1; cert[v] = base[v] >= 0 ? 1.f : 0.f; }
    if (a.s.mode == kHard) {
      const longlong2* lp = reinterpret_cast<const longlong2*>(a.s.labels + pix);
      const longlong2 l0 = lp[0], l1 = lp[1];
      const long long lab[4] = {l0.x, l0.y, l1.x, l1.y};
#pragma unroll
      for (int v = 0; v < 4; ++v)
        if (base[v] >= 0 && lab[v] >= 0 && lab[v] < K) cb_sts32(scratch + (uint32_t)((base[v] + (int)lab[v]) * kThreads * 16 + v * 4), 1.0f);
    } else {
      const bool use_thr = a.s.threshold > 0.f && a.s.threshold < 1.f;
      float pr[SLCL_MAX_CLASSES][4];
#pragma unroll
      for (int k = 0; k < SLCL_MAX_CLASSES; ++k)
        if (k < K) { const float4 t = *reinterpret_cast<const float4*>(a.s.probs + (b * K + k) * a.s.pixels + p); pr[k][0] = t.x; pr[k][1] = t.y; pr[k][2] = t.z; pr[k][3] = t.w; }
#pragma unroll
      for (int v = 0; v < 4; ++v) {
        int arg = 0;
        if constexpr (LOGITS) {        // logits -> probabilities (SLCL_SOFT_LOGITS); the largest one is 1/s
          float z[SLCL_MAX_CLASSES], pmax;
#pragma unroll
          for (int k = 0; k < SLCL_MAX_CLASSES; ++k) z[k] = (k < K) ? pr[k][v] : 0.f;
          softmax_inplace(z, K, pmax, arg);
#pragma unroll
          for (int k = 0; k < SLCL_MAX_CLASSES; ++k) pr[k][v] = z[k];
          if (use_thr && !(pmax >= a.s.threshold)) cert[v] = 0.f;
        } else if (use_thr || !a.s.weighted) {
          float best = -INFINITY;
#pragma unroll
          for (int k = 0; k < SLCL_MAX_CLASSES; ++k)
            if (k < K && pr[k][v] > best) { best = pr[k][v]; arg = k; }
          if (use_thr && !(best >= a.s.threshold)) cert[v] = 0.f;
        }
        if (base[v] >= 0) {
#pragma unroll
          for (int k = 0; k < SLCL_MAX_CLASSES; ++k)
            if (k < K) cb_sts32(scratch + (uint32_t)((base[v] + k) * kThreads * 16 + v * 4),
                                a.s.weighted ? pr[k][v] * cert[v] : ((k == arg) ? cert[v] : 0.f));
        }
      }
    }
  }
  unsigned long long w01[KWT], w23[KWT];
#pragma unroll
  for (int j = 0; j < KWT; ++j) cb_lds2x64(scratch + (uint32_t)(j * kThreads * 16), w01[j], w23[j]);

  unsigned long long d01[HAS_DP ? KWT : 1], d23[HAS_DP ? KWT : 1];
#pragma unroll
  for (int j = 0; j < (HAS_DP ? KWT : 1); ++j) { d01[j] = 0ull; d23[j] = 0ull; }

  for (int c = 0; c < C; ++c) {
    unsigned long long x01 = 0ull, x23 = 0ull;
    if constexpr (HAS_DP) {
      asm volatile("cp.async.wait_group %0;" ::"n"(kCenRing - 1) : "memory");
      cb_lds2x64(ring + (uint32_t)((c % kCenRing) * kThreads * 16), x01, x23);
      ring_fetch(c + kCenRing);
    }
    unsigned long long o01 = 0ull, o23 = 0ull;
    const uint32_t grow = sG2 + (uint32_t)(c * KP * 8);
#pragma unroll
    for (int j = 0; j < KWT; j += 2) {
      unsigned long long g0, g1;                                  // {g_j, g_j}, {g_j+1, g_j+1}: warp-wide broadcast
      cb_lds2x64(grow + j * 8, g0, g1);
      cb_ffma2(o01, w01[j], g0);
      cb_ffma2(o23, w23[j], g0);
      if constexpr (HAS_DP) { cb_ffma2(d01[j], x01, g0); cb_ffma2(d23[j], x23, g0); }
      if (j + 1 < KWT) {
        cb_ffma2(o01, w01[j + 1], g1);
        cb_ffma2(o23, w23[j + 1], g1);
        if constexpr (HAS_DP) { cb_ffma2(d01[j + 1], x01, g1); cb_ffma2(d23[j + 1], x23, g1); }
      }
    }
    const float2 oa = cb_unpack(o01), ob = cb_unpack(o23);
    st_stream4(dst + (int64_t)c * a.s.sc, make_float4(oa.x, oa.y, ob.x, ob.y));
  }
  if constexpr (HAS_DP && LOGITS) {
    // d z[b,k,p] = p_k * (g_k - sum_m p_m g_m), g_k = cert * (x . gc_j - mu_j . gc_j), j = part*K + k.  The weight row
    // (still in the scratch) holds p_k * cert in the pixel's K columns and zeros elsewhere: with S = sum_j w_j (x . gc_j -
    // mu_j . gc_j) over every column, replace w_j by w_j (x . gc_j - mu_j . gc_j - S) and gather columns part*K + k by
    // address as below.  The weights come back from shared memory, so w01 / w23 need not live past the channel loop.
    float S[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int j = 0; j < KWT; ++j) {
      const float m = (j < a.s.n_cols) ? a.mu_dot_gc[j] : 0.f;
      const float2 da = cb_unpack(d01[j]), db = cb_unpack(d23[j]);
      unsigned long long wlo, whi;
      cb_lds2x64(scratch + (uint32_t)(j * kThreads * 16), wlo, whi);
      const float2 wa = cb_unpack(wlo), wb = cb_unpack(whi);
      S[0] = fmaf(wa.x, da.x - m, S[0]); S[1] = fmaf(wa.y, da.y - m, S[1]);
      S[2] = fmaf(wb.x, db.x - m, S[2]); S[3] = fmaf(wb.y, db.y - m, S[3]);
    }
#pragma unroll
    for (int j = 0; j < KWT; ++j) {
      const float m = (j < a.s.n_cols) ? a.mu_dot_gc[j] : 0.f;
      const float2 da = cb_unpack(d01[j]), db = cb_unpack(d23[j]);
      unsigned long long wlo, whi;
      cb_lds2x64(scratch + (uint32_t)(j * kThreads * 16), wlo, whi);
      const float2 wa = cb_unpack(wlo), wb = cb_unpack(whi);
      cb_sts128(scratch + (uint32_t)(j * kThreads * 16), make_float4(wa.x * (da.x - m - S[0]), wa.y * (da.y - m - S[1]),
                                                                     wb.x * (db.x - m - S[2]), wb.y * (db.y - m - S[3])));
    }
#pragma unroll
    for (int k = 0; k < SLCL_MAX_CLASSES; ++k) {
      if (k < K) {
        float o[4];
#pragma unroll
        for (int v = 0; v < 4; ++v) o[v] = base[v] >= 0 ? cb_lds32(scratch + (uint32_t)((base[v] + k) * kThreads * 16 + v * 4)) : 0.f;
        st_stream4(a.dprobs + (b * K + k) * a.s.pixels + p, make_float4(o[0], o[1], o[2], o[3]));
      }
    }
  } else if constexpr (HAS_DP) {
    // d probs[b,k,p] = cert * (x . gc_j - mu_j . gc_j), j = part*K + k: park the KWT dot rows in the scratch, gather by address
#pragma unroll
    for (int j = 0; j < KWT; ++j) {
      const float m = (j < a.s.n_cols) ? a.mu_dot_gc[j] : 0.f;
      const float2 da = cb_unpack(d01[j]), db = cb_unpack(d23[j]);
      cb_sts128(scratch + (uint32_t)(j * kThreads * 16), make_float4(da.x - m, da.y - m, db.x - m, db.y - m));
    }
#pragma unroll
    for (int k = 0; k < SLCL_MAX_CLASSES; ++k) {
      if (k < K) {
        float o[4];
#pragma unroll
        for (int v = 0; v < 4; ++v)
          o[v] = base[v] >= 0 ? cert[v] * cb_lds32(scratch + (uint32_t)((base[v] + k) * kThreads * 16 + v * 4)) : 0.f;
        st_stream4(a.dprobs + (b * K + k) * a.s.pixels + p, make_float4(o[0], o[1], o[2], o[3]));
      }
    }
  }
}

// ------------------------------ host side ----------------------------------
int pick_kwt(int n_cols) {
  static const int opts[] = {2, 3, 4, 5, 6, 8, 10, 12, 16};
  for (int o : opts) if (n_cols <= o) return o;
  return -1;
}

struct SumPlan { int kwt, cpw, vec, cg_per_block, pt_per_block; dim3 grid; int64_t tiles_per_image, n_tiles; };

SumPlan plan_sums(int64_t B, int64_t C, int64_t HW, int n_cols, bool vec4) {
  SumPlan p;
  p.kwt = pick_kwt(n_cols);
  p.cpw = p.kwt <= 3 ? 8 : 4;
  p.vec = vec4 ? 4 : 1;
  int n_groups = (int)ceil_div<int64_t>(C, p.cpw);
  int cg = 1;
  while (cg < n_groups && cg < kWarps) cg *= 2;
  p.cg_per_block = cg;
  p.pt_per_block = kWarps / cg;
  p.tiles_per_image = ceil_div<int64_t>(HW, kChunks * 32 * p.vec);
  p.n_tiles = B * p.tiles_per_image;
  int gy = (int)ceil_div<int64_t>(n_groups, cg);
  int64_t gx = (int64_t)sm_count() * 2 / gy;
  if (gx < 1) gx = 1;
  // keep at least 2 block tiles per block so the end-of-block reduction is amortised
  if (gx > ceil_div<int64_t>(p.n_tiles, 2)) gx = ceil_div<int64_t>(p.n_tiles, 2);
  if (gx < 1) gx = 1;
  p.grid = dim3((unsigned)gx, (unsigned)gy, 1);
  return p;
}

size_t partial_bytes(const SumPlan& p, int64_t C) {
  return align_up((size_t)p.grid.x * p.kwt * (C + 1) * sizeof(float), 256);
}

template <int KWT, int CPW, bool LOGITS>
void launch_sums(const SumArgs& a, const SumPlan& p, cudaStream_t stream) {
  const size_t smem = (size_t)KWT * kChunks * 32 * p.vec * sizeof(float);
  if (p.vec == 4) {
    if (smem > 32 * 1024)
      cudaFuncSetAttribute(class_sums_kernel<KWT, CPW, 4, LOGITS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    class_sums_kernel<KWT, CPW, 4, LOGITS><<<p.grid, kThreads, smem, stream>>>(a);
  } else {
    class_sums_kernel<KWT, CPW, 1, LOGITS><<<p.grid, kThreads, smem, stream>>>(a);
  }
}

// ---- v3 host side ----
typedef CUresult (*V3EncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                               const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                               CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
V3EncodeFn v3_encode_fn() {
  static V3EncodeFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<V3EncodeFn>(p);
  }
  return fn;
}

struct V3Plan { bool ok; int kwt, cpw, n_cw, nbw, ncw_max; dim3 grid; };

// Register-tile shape per weight-column count (acc[CPW][KWT] lives in registers for the whole sweep):
//   KWT <= 10 : CPW 4, up to 16 consumer warps (64 channels per block)
//   KWT 12,16 : CPW 4, up to 8 consumer warps (acc[4][16] = 64 registers)
// (CPW 8 with half as many consumer warps was measured in round 2: fewer re-reads of the weight rows but one warp per
// scheduler cannot hide its own LDS latency -- 0.90 -> 0.80 at C = 128, KWT = 10 -- so it is not used.)
constexpr int v3_cpw(int kwt) { return 4; }
constexpr int v3_ncw(int kwt) { return kwt <= 10 ? 16 : 8; }
// builder warps: 4 teams (8 warps) when the stages are short and the accumulators few; 2 teams otherwise (long stages,
// or wide weight rows whose packed accumulators need the registers)
constexpr int v3_nbw(int ncw, int kwt) { return (ncw > 8 || kwt >= 6) ? 4 : 8; }

V3Plan plan_v3(const SumArgs& a, bool vec4) {
  V3Plan p{};
  p.ok = false;
  { const char* e = getenv("SLCL_CLASS_SUMS_V2"); if (e && atoi(e) != 0) return p; }
  if (!vec4 || a.sp != 1 || a.sc % 4 != 0 || a.sb % 4 != 0 || a.pixels > INT_MAX || a.batch > INT_MAX) return p;
  p.kwt = pick_kwt(a.n_cols);
  if (p.kwt < 0) return p;
  const int C = (int)a.channels;
  p.cpw = v3_cpw(p.kwt);
  p.ncw_max = v3_ncw(p.kwt);
  p.n_cw = ceil_div(C, p.cpw);
  if (p.n_cw > p.ncw_max) p.n_cw = p.ncw_max;
  if (p.n_cw <= 8) p.ncw_max = 8;
  p.nbw = v3_nbw(p.ncw_max, p.kwt);
  const int cb = p.n_cw * p.cpw;
  const int gy = ceil_div(C, cb);
  const int64_t n_tiles = a.batch * ceil_div<int64_t>(a.pixels, kV3Px);
  int64_t gx = sm_count() / gy;
  if (gx < 1) gx = 1;
  if (gx > n_tiles) gx = n_tiles;
  if (gx > (int64_t)sm_count() * 2) gx = (int64_t)sm_count() * 2;      // partial buffer is sized for 2 blocks per SM
  p.grid = dim3((unsigned)gx, (unsigned)gy, 1);
  p.ok = true;
  return p;
}

size_t v3_stage_bytes(int kwt, int cpw, int n_cw) { return (size_t)(n_cw * cpw + kwt + v3_raw_rows(kwt) + 1) * kV3Px * 4; }
// as deep as ~200 KB allow (small-C stages are short, the ring must be long), rounded down to a multiple of the
// builder teams so that every team sees every phase of the slots it works on
int v3_stages(int kwt, int cpw, int n_cw, int teams) {
  int n = (int)((200 * 1024) / v3_stage_bytes(kwt, cpw, n_cw));
  if (n > kV3MaxStages) n = kV3MaxStages;
  n = n / teams * teams;
  return n < teams ? teams : n;
}
size_t v3_smem_bytes(int kwt, int cpw, int n_cw, int teams) {
  return 128 + (size_t)v3_stages(kwt, cpw, n_cw, teams) * v3_stage_bytes(kwt, cpw, n_cw) + sizeof(V3Bars) + 64;
}

int v3_encode(CUtensorMap* map, const void* base, const cuuint64_t (&dims)[3], const cuuint64_t (&strides)[2],
              const cuuint32_t (&box)[3]) {
  V3EncodeFn fn = v3_encode_fn();
  if (!fn) return SLCL_ERR_CUDA;
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<void*>(base), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) { set_cuda_error(cudaErrorInvalidValue, "cuTensorMapEncodeTiled(class sums)"); return SLCL_ERR_CUDA; }
  return SLCL_OK;
}

template <int KWT, int CPW, int NCW, int NBW, bool LOGITS>
int launch_v3(const SumArgs& a, const V3Plan& p, cudaStream_t stream) {
  ensure_context_on_this_thread();
  CUtensorMap map, map_raw;
  {
    const cuuint64_t dims[3] = {(cuuint64_t)a.pixels, (cuuint64_t)a.channels, (cuuint64_t)a.batch};
    const cuuint64_t strides[2] = {(cuuint64_t)a.sc * 4, (cuuint64_t)a.sb * 4};
    const cuuint32_t box[3] = {(cuuint32_t)kV3Px, (cuuint32_t)(p.n_cw * CPW), 1};
    int st = v3_encode(&map, a.feat, dims, strides, box);
    if (st != SLCL_OK) return st;
  }
  map_raw = map;
  if (a.mode == kSoft) {              // probs (or logits) [B, K, HW]: box = all K rows of 128 pixels of one image
    const cuuint64_t dims[3] = {(cuuint64_t)a.pixels, (cuuint64_t)a.n_class, (cuuint64_t)a.batch};
    const cuuint64_t strides[2] = {(cuuint64_t)a.pixels * 4, (cuuint64_t)a.pixels * a.n_class * 4};
    const cuuint32_t box[3] = {(cuuint32_t)kV3Px, (cuuint32_t)a.n_class, 1};
    int st = v3_encode(&map_raw, a.probs, dims, strides, box);
    if (st != SLCL_OK) return st;
  } else if (a.mode == kPlanar) {     // planar weights [cols][B*HW] seen as {HW, B, cols}: rows beyond n_cols read as zero
    const cuuint64_t dims[3] = {(cuuint64_t)a.pixels, (cuuint64_t)a.batch, (cuuint64_t)a.n_cols};
    const cuuint64_t strides[2] = {(cuuint64_t)a.pixels * 4, (cuuint64_t)a.pixels * a.batch * 4};
    const cuuint32_t box[3] = {(cuuint32_t)kV3Px, 1, (cuuint32_t)KWT};
    int st = v3_encode(&map_raw, a.planar, dims, strides, box);
    if (st != SLCL_OK) return st;
  }
  const size_t smem = v3_smem_bytes(KWT, CPW, p.n_cw, NBW / 2);
  static bool attr_set_dev[64] = {};          // function attributes are per device
  bool& attr_set = attr_set_dev[current_device_slot()];
  if (!attr_set) {
    cudaError_t e = cudaFuncSetAttribute(class_sums_v3_kernel<KWT, CPW, NCW, NBW, LOGITS>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         220 * 1024);
    if (e != cudaSuccess) { set_cuda_error(e, "cudaFuncSetAttribute(class_sums_v3_kernel)"); return SLCL_ERR_CUDA; }
    attr_set = true;
  }
  SumArgs av = a;
  av.n_cw = p.n_cw;
  av.n_stages = v3_stages(KWT, CPW, p.n_cw, NBW / 2);
  if (smem > 220 * 1024) return SLCL_ERR_UNSUPPORTED;
  class_sums_v3_kernel<KWT, CPW, NCW, NBW, LOGITS><<<p.grid, 32 * (3 + NBW + p.n_cw), smem, stream>>>(map, map_raw, av);
  return SLCL_OK;
}

template <int KWT, bool LOGITS>
int launch_v3_cpw(const SumArgs& a, const V3Plan& p, cudaStream_t stream) {
  constexpr int CPW = v3_cpw(KWT);
  if constexpr (v3_ncw(KWT) > 8) {
    if (p.n_cw > 8) return launch_v3<KWT, CPW, 16, v3_nbw(16, KWT), LOGITS>(a, p, stream);
  }
  return launch_v3<KWT, CPW, 8, v3_nbw(8, KWT), LOGITS>(a, p, stream);
}

void launch_reduce(const SumArgs& a, int n_blocks, int kwt, double* sums, const slcl_peer_t* peer, const FinArgs& fin,
                   cudaStream_t stream) {
  const int total = a.n_cols * ((int)a.channels + 1);
  const dim3 grid(ceil_div(total, kWarps));
  if (peer != nullptr && peer->world > 1)
    class_sums_reduce_kernel<true><<<grid, kThreads, 0, stream>>>(a.partial, n_blocks, kwt, a.n_cols, (int)a.channels, sums,
                                                                   peer_ctx(peer), fin, a.ticket);
  else
    class_sums_reduce_kernel<false><<<grid, kThreads, 0, stream>>>(a.partial, n_blocks, kwt, a.n_cols, (int)a.channels, sums,
                                                                    PeerCtx{}, fin, a.ticket);
}

// The sweep alone: per-block partials of `a` at `workspace` (`usable` bytes); the caller has set a.ticket.  On return
// a.partial, n_blocks and kwt describe the partials for the reduce (launch_reduce or the MCCL step's tail).
int launch_sweep(SumArgs& a, bool vec4, void* workspace, size_t usable, cudaStream_t stream, bool logits, int& n_blocks,
                 int& kwt) {
  SumPlan p = plan_sums(a.batch, a.channels, a.pixels, a.n_cols, vec4);
  if (p.kwt < 0) return SLCL_ERR_INVALID_ARGUMENT;
  const V3Plan v3 = plan_v3(a, vec4);
  if (v3.ok && (size_t)v3.grid.x * v3.kwt * (a.channels + 1) * sizeof(float) <= usable) {
    a.partial = reinterpret_cast<float*>(workspace);
    int st;
    switch (v3.kwt) {
      case 2: st = logits ? launch_v3_cpw<2, true>(a, v3, stream) : launch_v3_cpw<2, false>(a, v3, stream); break;
      case 3: st = logits ? launch_v3_cpw<3, true>(a, v3, stream) : launch_v3_cpw<3, false>(a, v3, stream); break;
      case 4: st = logits ? launch_v3_cpw<4, true>(a, v3, stream) : launch_v3_cpw<4, false>(a, v3, stream); break;
      case 5: st = logits ? launch_v3_cpw<5, true>(a, v3, stream) : launch_v3_cpw<5, false>(a, v3, stream); break;
      case 6: st = logits ? launch_v3_cpw<6, true>(a, v3, stream) : launch_v3_cpw<6, false>(a, v3, stream); break;
      case 8: st = logits ? launch_v3_cpw<8, true>(a, v3, stream) : launch_v3_cpw<8, false>(a, v3, stream); break;
      case 10: st = logits ? launch_v3_cpw<10, true>(a, v3, stream) : launch_v3_cpw<10, false>(a, v3, stream); break;
      case 12: st = logits ? launch_v3_cpw<12, true>(a, v3, stream) : launch_v3_cpw<12, false>(a, v3, stream); break;
      case 16: st = logits ? launch_v3_cpw<16, true>(a, v3, stream) : launch_v3_cpw<16, false>(a, v3, stream); break;
      default: return SLCL_ERR_INVALID_ARGUMENT;
    }
    n_blocks = (int)v3.grid.x;
    kwt = v3.kwt;
    return st;
  }
  if (partial_bytes(p, a.channels) > usable) return SLCL_ERR_WORKSPACE;
  a.tiles_per_image = p.tiles_per_image; a.n_tiles = p.n_tiles;
  a.cg_per_block = p.cg_per_block; a.pt_per_block = p.pt_per_block;
  a.partial = reinterpret_cast<float*>(workspace);
  switch (p.kwt) {
    case 2: logits ? launch_sums<2, 8, true>(a, p, stream) : launch_sums<2, 8, false>(a, p, stream); break;
    case 3: logits ? launch_sums<3, 8, true>(a, p, stream) : launch_sums<3, 8, false>(a, p, stream); break;
    case 4: logits ? launch_sums<4, 4, true>(a, p, stream) : launch_sums<4, 4, false>(a, p, stream); break;
    case 5: logits ? launch_sums<5, 4, true>(a, p, stream) : launch_sums<5, 4, false>(a, p, stream); break;
    case 6: logits ? launch_sums<6, 4, true>(a, p, stream) : launch_sums<6, 4, false>(a, p, stream); break;
    case 8: logits ? launch_sums<8, 4, true>(a, p, stream) : launch_sums<8, 4, false>(a, p, stream); break;
    case 10: logits ? launch_sums<10, 4, true>(a, p, stream) : launch_sums<10, 4, false>(a, p, stream); break;
    case 12: logits ? launch_sums<12, 4, true>(a, p, stream) : launch_sums<12, 4, false>(a, p, stream); break;
    case 16: logits ? launch_sums<16, 4, true>(a, p, stream) : launch_sums<16, 4, false>(a, p, stream); break;
    default: return SLCL_ERR_INVALID_ARGUMENT;
  }
  n_blocks = (int)p.grid.x;
  kwt = p.kwt;
  return SLCL_OK;
}

// sweep + reduce (+ cross-rank exchange through `peer`, + finaliser `fin` in the reduce kernel's last block).
// logits: soft mode with logits in a.probs (the sweep applies the softmax).
int run_class_sums(SumArgs a, bool vec4, double* sums, void* workspace, size_t workspace_bytes, cudaStream_t stream,
                   const slcl_peer_t* peer = nullptr, FinArgs fin = FinArgs{}, bool logits = false) {
  if (a.n_cols < 1 || a.n_cols > SLCL_MAX_WEIGHT_COLS) return SLCL_ERR_INVALID_ARGUMENT;
  if (peer != nullptr) {
    if (!peer_valid(peer)) return SLCL_ERR_INVALID_ARGUMENT;
    if (2 * (int64_t)a.n_cols * (a.channels + 1) > peer->capacity_words) return SLCL_ERR_INVALID_ARGUMENT;
  }
  SumPlan p = plan_sums(a.batch, a.channels, a.pixels, a.n_cols, vec4);
  if (p.kwt < 0) return SLCL_ERR_INVALID_ARGUMENT;
  if (workspace_bytes < partial_bytes(p, a.channels) + kTicketBytes || !aligned16(workspace)) return SLCL_ERR_WORKSPACE;
  // the ticket lives in the last 256 bytes of the workspace the caller sized with class_sums_ws_bytes()
  a.ticket = reinterpret_cast<unsigned int*>(reinterpret_cast<char*>(workspace) + (workspace_bytes - kTicketBytes) / 16 * 16);
  int n_blocks = 0, kwt = 0;
  const int st = launch_sweep(a, vec4, workspace, workspace_bytes - kTicketBytes, stream, logits, n_blocks, kwt);
  if (st != SLCL_OK) return st;
  launch_reduce(a, n_blocks, kwt, sums, peer, fin, stream);
  return check_launch("slcl_class_sums");
}

bool nchw_vec4(const float* feat, int64_t C, int64_t HW, std::initializer_list<const void*> ptrs) {
  bool ok = (HW % 4 == 0);
  for (const void* q : ptrs) ok = ok && (q == nullptr || aligned16(q));
  (void)feat; (void)C;
  return ok;
}

// `weighted` of the soft-label entry points is a flags word: SLCL_SOFT_WEIGHTED | SLCL_SOFT_LOGITS, the latter for soft
// labels only.
bool soft_flags_ok(int flags, const int64_t* labels) {
  if (flags & ~(SLCL_SOFT_WEIGHTED | SLCL_SOFT_LOGITS)) return false;
  return !((flags & SLCL_SOFT_LOGITS) && labels != nullptr);
}

}  // namespace

size_t class_sums_ws_bytes(int64_t batch, int64_t channels, int64_t pixels, int n_cols) {
  if (batch <= 0 || channels <= 0 || pixels <= 0 || n_cols < 1 || n_cols > SLCL_MAX_WEIGHT_COLS) return 0;
  // the grid never exceeds 2 blocks per SM; size for the worst case of either vector width
  int kwt = pick_kwt(n_cols);
  size_t blocks = (size_t)sm_count() * 2;
  return align_up(blocks * kwt * (channels + 1) * sizeof(float), 256) + kTicketBytes;
}

// used by slcl_proto_bwd_centres: weights are the planar stash rows [cols][N]
int class_sums_planar_weights(const float* feat, const slcl_map_t* map, const float* weights, int n_cols, double* sums,
                              void* workspace, size_t workspace_bytes, cudaStream_t stream) {
  SumArgs a{};
  a.feat = feat;
  a.batch = map->batch; a.channels = map->channels; a.pixels = map->pixels;
  a.sb = map->stride_b; a.sc = map->stride_c; a.sp = map->stride_p;
  a.mode = kPlanar; a.planar = weights; a.n_cols = n_cols; a.n_part = 1; a.n_class = n_cols;
  bool vec4 = (map->stride_p == 1) && (map->pixels % 4 == 0) && (map->stride_c % 4 == 0) && (map->stride_b % 4 == 0) &&
              aligned16(feat) && aligned16(weights);
  return run_class_sums(a, vec4, sums, workspace, workspace_bytes, stream);
}

}  // namespace slcl

using namespace slcl;

extern "C" size_t slcl_class_sums_workspace_bytes(int64_t batch, int64_t channels, int64_t pixels, int n_cols) {
  return class_sums_ws_bytes(batch, channels, pixels, n_cols);
}

extern "C" int slcl_class_sums(const float* feat, int64_t batch, int64_t channels, int64_t pixels,
                               const int64_t* labels, const float* probs, int weighted, float threshold,
                               const int32_t* part_id, int n_partitions, int n_class, double* sums, void* workspace,
                               size_t workspace_bytes, slcl_stream_t stream_) {
  if (!feat || batch <= 0 || channels <= 0 || pixels <= 0 || !sums || !workspace) return SLCL_ERR_INVALID_ARGUMENT;
  if ((labels == nullptr) == (probs == nullptr) || !soft_flags_ok(weighted, labels)) return SLCL_ERR_INVALID_ARGUMENT;
  if (n_class < 1 || n_class > kMaxK || n_partitions < 1 || n_partitions * n_class > SLCL_MAX_WEIGHT_COLS)
    return SLCL_ERR_INVALID_ARGUMENT;
  if (n_partitions > 1 && part_id == nullptr) return SLCL_ERR_INVALID_ARGUMENT;
  SumArgs a{};
  a.feat = feat;
  a.batch = batch; a.channels = channels; a.pixels = pixels;
  a.sb = channels * pixels; a.sc = pixels; a.sp = 1;
  a.mode = labels ? kHard : kSoft;
  a.labels = labels; a.probs = probs; a.weighted = weighted & SLCL_SOFT_WEIGHTED; a.threshold = threshold;
  a.part_id = part_id; a.n_part = n_partitions; a.n_class = n_class;
  a.n_cols = n_partitions * n_class;
  bool vec4 = nchw_vec4(feat, channels, pixels, {feat, labels, probs, part_id});
  return run_class_sums(a, vec4, sums, workspace, workspace_bytes, (cudaStream_t)stream_, nullptr, FinArgs{},
                        (weighted & SLCL_SOFT_LOGITS) != 0);
}

extern "C" int slcl_class_centres_update(const float* feat, int64_t batch, int64_t channels, int64_t pixels,
                                         const int64_t* labels, int n_class, const float* old_centres, float m,
                                         float* new_centres, double* sums, const slcl_peer_t* peer, void* workspace,
                                         size_t workspace_bytes, slcl_stream_t stream_) {
  if (!feat || batch <= 0 || channels <= 0 || pixels <= 0 || !labels || !old_centres || !new_centres || !sums || !workspace)
    return SLCL_ERR_INVALID_ARGUMENT;
  if (n_class < 1 || n_class > kMaxK) return SLCL_ERR_INVALID_ARGUMENT;
  SumArgs a{};
  a.feat = feat;
  a.batch = batch; a.channels = channels; a.pixels = pixels;
  a.sb = channels * pixels; a.sc = pixels; a.sp = 1;
  a.mode = kHard; a.labels = labels; a.n_part = 1; a.n_class = n_class; a.n_cols = n_class;
  const bool vec4 = nchw_vec4(feat, channels, pixels, {feat, labels});
  FinArgs fin{kFinEma, old_centres, m, n_class, new_centres, nullptr};
  return run_class_sums(a, vec4, sums, workspace, workspace_bytes, (cudaStream_t)stream_, peer, fin);
}

extern "C" int slcl_centroids_fwd(const float* feat, int64_t batch, int64_t channels, int64_t pixels,
                                  const int64_t* labels, const float* probs, int weighted, float threshold,
                                  const int32_t* part_id, int n_partitions, int n_class, const float* previous,
                                  float momentum, float* centroids, float* inv_weight, double* sums,
                                  const slcl_peer_t* peer, void* workspace, size_t workspace_bytes,
                                  slcl_stream_t stream_) {
  if (!feat || batch <= 0 || channels <= 0 || pixels <= 0 || !centroids || !inv_weight || !sums || !workspace)
    return SLCL_ERR_INVALID_ARGUMENT;
  if ((labels == nullptr) == (probs == nullptr) || !soft_flags_ok(weighted, labels)) return SLCL_ERR_INVALID_ARGUMENT;
  if (n_class < 1 || n_class > kMaxK || n_partitions < 1 || n_partitions * n_class > SLCL_MAX_WEIGHT_COLS)
    return SLCL_ERR_INVALID_ARGUMENT;
  if (n_partitions > 1 && part_id == nullptr) return SLCL_ERR_INVALID_ARGUMENT;
  SumArgs a{};
  a.feat = feat;
  a.batch = batch; a.channels = channels; a.pixels = pixels;
  a.sb = channels * pixels; a.sc = pixels; a.sp = 1;
  a.mode = labels ? kHard : kSoft;
  a.labels = labels; a.probs = probs; a.weighted = weighted & SLCL_SOFT_WEIGHTED; a.threshold = threshold;
  a.part_id = part_id; a.n_part = n_partitions; a.n_class = n_class;
  a.n_cols = n_partitions * n_class;
  const bool vec4 = nchw_vec4(feat, channels, pixels, {feat, labels, probs, part_id});
  FinArgs fin{kFinCentroid, previous, momentum, n_class, centroids, inv_weight};
  return run_class_sums(a, vec4, sums, workspace, workspace_bytes, (cudaStream_t)stream_, peer, fin,
                        (weighted & SLCL_SOFT_LOGITS) != 0);
}

namespace slcl {
void launch_prep_centres(const float* centres, int C, int K, int normalize, float* cstate, cudaStream_t stream);
void launch_proto_finalize(const void* partial, int n_blocks, int64_t n_total, int has_sel, float* scal,
                           const slcl_peer_t* peer, cudaStream_t stream);
namespace {
struct TilePlan { bool ok; int cpw, n_cw, npw, stages, wide; unsigned grid; size_t smem; };
TilePlan plan_tile(int64_t batch, int64_t C, int64_t pixels, int K) {
  TilePlan p{};
  p.ok = false;
  if (C < 1 || C > 128 || K < 2 || K > kMaxK || pixels % 4 != 0 || pixels > INT_MAX || batch > INT_MAX) return p;
  // register tile per shape (acc[CPW][K] <= 40 registers)
  if (C <= 32) p.cpw = 4;
  else if (C <= 64 && K <= 5) p.cpw = 8;
  else if (C <= 64) p.cpw = 4;
  else if (K <= 5) p.cpw = 8;
  else return p;
  p.wide = (C > 64 && p.cpw == 8 && !getenv("SLCL_TILE_NARROW")) ? 1 : 0;          // consumer warps of 2 x CPW channels
  p.n_cw = (int)ceil_div<int64_t>(C, p.cpw * (p.wide ? 2 : 1));
  const int kp = K <= 4 ? 4 : 8;
  const size_t stage = (size_t)(C + K) * kTPx * 4;
  const size_t fixed = 128 + (size_t)C * kp * 4 + sizeof(V3Bars) + 64;
  int n = (int)((216 * 1024 - fixed) / stage);          // C = 128, K = 5: six 33 KB stages
  if (n > kV3MaxStages) n = kV3MaxStages;
  if (n < 4) return p;
  // teams of pixel warps: four (measured at cfg2, C = 128, six stages fit: 4 teams x 1 slot 290 us, 3 x 2 305 us,
  // 2 x 3 344 us -- pixel warps in flight count for more than spare slots)
  p.npw = 4;
  if (p.n_cw <= 8 && n >= 6) p.npw = 6;          // room for 12 pixel warps next to 8 consumers (and 6 divides the 12-deep ring)
  { const char* e = getenv("SLCL_TILE_TEAMS"); if (e && atoi(e) >= 1 && atoi(e) <= tile_teams_max(p.n_cw <= 8 ? 8 : 16) && atoi(e) <= n) p.npw = atoi(e); }
  n = n / p.npw * p.npw;
  p.stages = n;
  p.smem = fixed + (size_t)n * stage;
  const int64_t n_tiles = batch * ceil_div<int64_t>(pixels, kTPx);
  p.grid = (unsigned)std::min<int64_t>(sm_count(), n_tiles);
  p.ok = true;
  return p;
}
template <int K, int CPW, int NCWMAX>
int launch_tile(const CUtensorMap& map, const TileArgs& a, const TilePlan& p, cudaStream_t stream) {
  static bool attr_set_dev[64] = {};
  bool& attr_set = attr_set_dev[current_device_slot()];
  if (!attr_set) {
    cudaError_t e = cudaFuncSetAttribute(target_tile_kernel<K, CPW, NCWMAX>, cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024);
    if (e != cudaSuccess) { set_cuda_error(e, "cudaFuncSetAttribute(target_tile_kernel)"); return SLCL_ERR_CUDA; }
    attr_set = true;
  }
  launch_pdl(target_tile_kernel<K, CPW, NCWMAX>, dim3(p.grid), dim3(32 * (2 + 2 * tile_teams_max(NCWMAX) + p.n_cw)), p.smem, stream, map, a);
  return SLCL_OK;
}
template <int K>
int launch_tile_k(const CUtensorMap& map, const TileArgs& a, const TilePlan& p, cudaStream_t stream) {
  if (p.cpw == 4 && p.n_cw <= 8) return launch_tile<K, 4, 8>(map, a, p, stream);
  if (p.cpw == 4) return launch_tile<K, 4, 16>(map, a, p, stream);
  if constexpr (K <= 5) {
    if (p.n_cw <= 8) return launch_tile<K, 8, 8>(map, a, p, stream);
    return launch_tile<K, 8, 16>(map, a, p, stream);
  }
  return SLCL_ERR_UNSUPPORTED;
}
}  // namespace
}  // namespace slcl

extern "C" size_t slcl_target_step_workspace_bytes(int64_t channels, int n_class) {
  if (channels <= 0 || n_class < 1) return 0;
  const size_t blocks = (size_t)sm_count();
  return align_up(blocks * sizeof(double2), 256) + align_up(blocks * n_class * (channels + 1) * sizeof(float), 256) + kTicketBytes;
}

extern "C" int slcl_target_step(const float* feat, int64_t batch, int64_t channels, int64_t pixels, const float* centres,
                                const slcl_proto_params_t* params, float sel_threshold, int weight_by_sel,
                                int64_t* label, float* sel, float* stash, float* cstate, float* scal, double* sums,
                                const float* previous, float momentum, float* centroids, float* inv_weight,
                                const slcl_peer_t* peer, void* workspace, size_t workspace_bytes, slcl_stream_t stream_) {
  if (!feat || batch <= 0 || channels <= 0 || pixels <= 0 || !centres || !params || !label || !sel || !stash || !cstate ||
      !scal || !sums || !centroids || !inv_weight || !workspace)
    return SLCL_ERR_INVALID_ARGUMENT;
  const int K = params->n_class;
  if (K < 2 || K > kMaxK || !(params->temperature > 0.f) || !(params->base_temperature > 0.f) || !params->normalize)
    return SLCL_ERR_INVALID_ARGUMENT;
  if (peer != nullptr && (!peer_valid(peer) || 2 * (int64_t)K * (channels + 1) > peer->capacity_words)) return SLCL_ERR_INVALID_ARGUMENT;
  if (workspace_bytes < slcl_target_step_workspace_bytes(channels, K) || !aligned16(workspace)) return SLCL_ERR_WORKSPACE;
  const TilePlan p = plan_tile(batch, channels, pixels, K);
  if (!p.ok || !aligned16(feat) || !aligned16(label) || !aligned16(sel) || !aligned16(stash)) return SLCL_ERR_UNSUPPORTED;
  cudaStream_t stream = (cudaStream_t)stream_;
  ensure_context_on_this_thread();
  CUtensorMap map;
  {
    const cuuint64_t dims[3] = {(cuuint64_t)pixels, (cuuint64_t)channels, (cuuint64_t)batch};
    const cuuint64_t strides[2] = {(cuuint64_t)pixels * 4, (cuuint64_t)pixels * channels * 4};
    const cuuint32_t box[3] = {(cuuint32_t)kTPx, (cuuint32_t)channels, 1};
    int st = v3_encode(&map, feat, dims, strides, box);
    if (st != SLCL_OK) return st;
  }
  const size_t blocks = (size_t)sm_count();
  char* ws = reinterpret_cast<char*>(workspace);
  TileArgs a{};
  a.feat = feat; a.batch = batch; a.channels = channels; a.pixels = pixels; a.n_total = batch * pixels;
  a.cstate = cstate; a.mc = make_margin_const(params); a.sel_threshold = sel_threshold; a.weight_by_sel = weight_by_sel;
  a.out_label = label; a.out_sel = sel; a.stash = stash;
  a.loss_partial = reinterpret_cast<double2*>(ws);
  a.partial = reinterpret_cast<float*>(ws + align_up(blocks * sizeof(double2), 256));
  a.ticket = reinterpret_cast<unsigned int*>(ws + (workspace_bytes - kTicketBytes) / 16 * 16);
  a.n_cw = p.n_cw; a.n_stages = p.stages; a.n_teams = p.npw; a.wide = p.wide;
  launch_prep_centres(centres, (int)channels, K, 1, cstate, stream);
  int st = SLCL_ERR_UNSUPPORTED;
  switch (K) {
    case 2: st = launch_tile_k<2>(map, a, p, stream); break;
    case 3: st = launch_tile_k<3>(map, a, p, stream); break;
    case 4: st = launch_tile_k<4>(map, a, p, stream); break;
    case 5: st = launch_tile_k<5>(map, a, p, stream); break;
    case 6: st = launch_tile_k<6>(map, a, p, stream); break;
    case 7: st = launch_tile_k<7>(map, a, p, stream); break;
    case 8: st = launch_tile_k<8>(map, a, p, stream); break;
    default: return SLCL_ERR_INVALID_ARGUMENT;
  }
  if (st != SLCL_OK) return st;
  launch_proto_finalize(a.loss_partial, (int)p.grid, a.n_total, 1, scal, peer, stream);      // loss pair exchanged here too
  SumArgs sa{};
  sa.channels = channels; sa.n_cols = K; sa.partial = a.partial; sa.ticket = a.ticket;
  FinArgs fin{kFinCentroid, previous, momentum, K, centroids, inv_weight};
  launch_reduce(sa, (int)p.grid, K, sums, peer, fin, stream);
  return check_launch("slcl_target_step");
}

extern "C" int slcl_ema_finalize(const double* sums, const float* old_centres, float m, int n_class, int64_t channels,
                                 float* new_centres, slcl_stream_t stream_) {
  if (!sums || !old_centres || !new_centres || n_class < 1 || channels <= 0) return SLCL_ERR_INVALID_ARGUMENT;
  const int total = n_class * (int)channels;
  ema_finalize_kernel<<<ceil_div(total, kThreads), kThreads, 0, (cudaStream_t)stream_>>>(sums, old_centres, m, n_class,
                                                                                        (int)channels, new_centres);
  return check_launch("slcl_ema_finalize");
}

extern "C" int slcl_centroid_finalize(const double* sums, const float* previous, float momentum, int n_sets,
                                      int n_class, int64_t channels, float* centroids, float* inv_weight,
                                      slcl_stream_t stream_) {
  if (!sums || !centroids || !inv_weight || n_sets < 1 || n_class < 1 || channels <= 0)
    return SLCL_ERR_INVALID_ARGUMENT;
  const int rows = n_sets * n_class;
  const int total = rows * (int)channels;
  centroid_finalize_kernel<<<ceil_div(total, kThreads), kThreads, 0, (cudaStream_t)stream_>>>(
      sums, previous, momentum, rows, n_class, (int)channels, centroids, inv_weight);
  return check_launch("slcl_centroid_finalize");
}

namespace slcl {
namespace {
// The centroid backward sweep of `a` (a.gc / a.mu_dot_gc prepared): centroid_bwd4_kernel on 128-bit maps, else
// centroid_bwd_kernel; a.dprobs may be null.
int launch_centroid_bwd(const CenBwdArgs& a, bool vec4, bool logits, cudaStream_t stream) {
  const int64_t channels = a.s.channels;
  const float* dprobs = a.dprobs;
  const int kwt = pick_kwt(a.s.n_cols);
  const int vec = vec4 ? 4 : 1;
  size_t smem = (size_t)channels * ((kwt + 3) / 4 * 4) * sizeof(float);
  if (vec4) {      // centroid_bwd4_kernel: {g, g} pairs [C][KP] + per-thread scratch [KWT][threads] float4 (+ the cp.async ring)
    smem = (size_t)channels * ((kwt + 1) / 2 * 2) * 8 + (size_t)kwt * kThreads * 16;
    if (dprobs) smem += (size_t)kCenRing * kThreads * 16;
  }
  if (smem > 200 * 1024) return SLCL_ERR_UNSUPPORTED;
  const int blocks = (int)ceil_div<int64_t>(a.s.batch * a.s.pixels / vec, kThreads);
#define SLCL_CB(KW_)                                                                                          \
  case KW_: {                                                                                                 \
    auto launch = [&](auto kern) -> int {                                                                     \
      if (smem > 48 * 1024) {                                                                                 \
        cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);   \
        if (e != cudaSuccess) { set_cuda_error(e, "cudaFuncSetAttribute"); return SLCL_ERR_CUDA; }            \
      }                                                                                                       \
      kern<<<blocks, kThreads, smem, stream>>>(a);                                                            \
      return SLCL_OK;                                                                                         \
    };                                                                                                        \
    int st;                                                                                                   \
    if (logits) {                                                                                             \
      if (dprobs) st = vec4 ? launch(centroid_bwd4_kernel<KW_, true, true>) : launch(centroid_bwd_kernel<KW_, 1, true, true>); \
      else st = vec4 ? launch(centroid_bwd4_kernel<KW_, false, true>) : launch(centroid_bwd_kernel<KW_, 1, false, true>); \
    } else if (dprobs) {                                                                                      \
      st = vec4 ? launch(centroid_bwd4_kernel<KW_, true, false>) : launch(centroid_bwd_kernel<KW_, 1, true, false>); \
    } else {                                                                                                  \
      st = vec4 ? launch(centroid_bwd4_kernel<KW_, false, false>) : launch(centroid_bwd_kernel<KW_, 1, false, false>); \
    }                                                                                                         \
    if (st != SLCL_OK) return st;                                                                             \
  } break;
  switch (kwt) {
    SLCL_CB(2) SLCL_CB(3) SLCL_CB(4) SLCL_CB(5) SLCL_CB(6) SLCL_CB(8) SLCL_CB(10) SLCL_CB(12) SLCL_CB(16)
    default: return SLCL_ERR_INVALID_ARGUMENT;
  }
#undef SLCL_CB
  return SLCL_OK;
}
}  // namespace
}  // namespace slcl

extern "C" size_t slcl_centroid_bwd_workspace_bytes(int64_t channels, int n_cols) {
  if (channels <= 0 || n_cols < 1) return 0;
  return align_up((size_t)n_cols * (channels + 1) * sizeof(float), 256);
}

extern "C" int slcl_centroid_bwd(const float* feat, int64_t batch, int64_t channels, int64_t pixels,
                                 const int64_t* labels, const float* probs, int weighted, float threshold,
                                 const int32_t* part_id, int n_partitions, int n_class, const float* grad_centroids,
                                 const double* sums, float ema_scale, float* dfeat, float* dprobs, void* workspace,
                                 size_t workspace_bytes, slcl_stream_t stream_) {
  if (!feat || batch <= 0 || channels <= 0 || pixels <= 0 || !grad_centroids || !sums || !dfeat || !workspace)
    return SLCL_ERR_INVALID_ARGUMENT;
  if ((labels == nullptr) == (probs == nullptr) || !soft_flags_ok(weighted, labels)) return SLCL_ERR_INVALID_ARGUMENT;
  if (n_class < 1 || n_class > kMaxK || n_partitions < 1 || n_partitions * n_class > SLCL_MAX_WEIGHT_COLS)
    return SLCL_ERR_INVALID_ARGUMENT;
  if (n_partitions > 1 && part_id == nullptr) return SLCL_ERR_INVALID_ARGUMENT;
  if (dprobs != nullptr && (probs == nullptr || !(weighted & SLCL_SOFT_WEIGHTED))) return SLCL_ERR_INVALID_ARGUMENT;
  const bool logits = (weighted & SLCL_SOFT_LOGITS) != 0;
  const int n_cols = n_partitions * n_class;
  if (workspace_bytes < slcl_centroid_bwd_workspace_bytes(channels, n_cols) || !aligned16(workspace))
    return SLCL_ERR_WORKSPACE;
  float* gc = reinterpret_cast<float*>(workspace);
  float* mu_dot_gc = gc + (size_t)n_cols * channels;
  centroid_bwd_prep_kernel<<<n_cols, kThreads, 0, (cudaStream_t)stream_>>>(grad_centroids, sums, ema_scale, (int)channels,
                                                                           gc, mu_dot_gc);
  CenBwdArgs a{};
  a.s.feat = feat;
  a.s.batch = batch; a.s.channels = channels; a.s.pixels = pixels;
  a.s.sb = channels * pixels; a.s.sc = pixels; a.s.sp = 1;
  a.s.mode = labels ? kHard : kSoft;
  a.s.labels = labels; a.s.probs = probs; a.s.weighted = weighted & SLCL_SOFT_WEIGHTED; a.s.threshold = threshold;
  a.s.part_id = part_id; a.s.n_part = n_partitions; a.s.n_class = n_class;
  a.s.n_cols = n_partitions * n_class;
  a.gc = gc; a.mu_dot_gc = mu_dot_gc; a.dfeat = dfeat; a.dprobs = dprobs;
  const bool vec4 = nchw_vec4(feat, channels, pixels, {feat, labels, probs, part_id, dfeat, dprobs});
  const int st = launch_centroid_bwd(a, vec4, logits, (cudaStream_t)stream_);
  if (st != SLCL_OK) return st;
  return check_launch("slcl_centroid_bwd");
}

// ===========================================================================
// The MCCL loss section as one call (trainer/Trainer_MCCL.py:275-326):
//   cs = cal_centroid(ft_s, labels_s, previous_centroid_s)              hard labels, EMA'd; detached (:277)
//   ct = cal_centroid(ft_t, pred_t, pseudo_label, partition = P)        soft labels (probabilities or logits)
//   ca = cal_centroid(ft_t_aug, pred_t_aug, pseudo_label)               P = 1, optional
//   total, terms = mccl_centroid_losses(cs, ct, ca, ...)
// Forward: the existing class-sum sweep once per set, each into its own region of one workspace, then ONE tail kernel
// that reduces every set's partials in block order into one sums matrix
//   rows [0, K) source | [K, (P+1)K) target partitions | [(P+1)K, (P+2)K) augmented target
// (bit-identical to the separate calls' reduce), exchanges the whole matrix in one mailbox epoch, and in its last block
// finalises the centroids and evaluates every centroid <-> centroid term and its gradient dL/dC (centroid_pair.cuh).
// Backward: one coefficient kernel (grad_out * dL/dC scaled as centroid_bwd_prep_kernel does), then the existing
// centroid backward sweep for the target set and for the augmented set.
// ===========================================================================
namespace slcl {
namespace {

constexpr int kStepMaxSets = 3;

struct StepTail {
  const float* partial[kStepMaxSets];
  int n_blocks[kStepMaxSets], kwt[kStepMaxSets];
  int row_end[kStepMaxSets];        // set s holds sums rows [row_end[s-1], row_end[s])
  int rows, K, C;
  double* sums;                     // [rows, C+1]
  unsigned int* ticket;
  const float* prev_s;              // previous source centroids [K, C] or null
  float momentum;
  float* cen;                       // [rows, C]
  float* inv_w;                     // [rows] (scratch)
  cpair::McclArgs loss;             // S, T, A = rows of cen; dS, dT, dA = rows of dL/dC
};

// One block: centroids from the complete sums, then every pair term and the weighted combination.
__device__ __forceinline__ void mccl_step_finish_block(const StepTail& t) {
  const FinArgs fs{kFinCentroid, t.prev_s, t.momentum, t.K, t.cen, t.inv_w};
  finalize_rows(t.sums, fs, t.K, t.C, threadIdx.x, kThreads);
  const FinArgs ft{kFinCentroid, nullptr, t.momentum, t.K, t.cen + (size_t)t.K * t.C, t.inv_w + t.K};
  finalize_rows(t.sums + (size_t)t.K * (t.C + 1), ft, t.rows - t.K, t.C, threadIdx.x, kThreads);
  __syncthreads();
  for (int i = 0; i < 3 * t.loss.P; ++i) {
    cpair::mccl_pair(t.loss, i);
    __syncthreads();
  }
  cpair::mccl_combine<true>(t.loss);
}

// One warp per sums element, as class_sums_reduce_kernel; PEER: the element is all-reduced over the ranks in the same
// epoch for every set.  `finish` = 0 leaves the (local) sums only: the NCCL route sums them and runs the finish kernel.
template <bool PEER>
__global__ void __launch_bounds__(kThreads) mccl_step_tail_kernel(const StepTail t, const PeerCtx pc, int finish) {
  __shared__ int s_last;
  const int lane = threadIdx.x & 31;
  const int idx = blockIdx.x * kWarps + (threadIdx.x >> 5);
  const int row = t.C + 1;
  unsigned int e = 0u;
  if constexpr (PEER) e = peer_epoch_begin(pc);
  if (idx < t.rows * row) {
    const int r = idx / row, c = idx % row;
    int s = 0, r0 = 0;
    while (r >= t.row_end[s]) { r0 = t.row_end[s]; ++s; }
    const float* partial = t.partial[s];
    const int kwt = t.kwt[s], n_blocks = t.n_blocks[s], col = r - r0;
    double v = 0.0;                                   // the block order of class_sums_reduce_kernel: identical bits
    for (int b = lane; b < n_blocks; b += 32) v += (double)partial[((int64_t)b * kwt + col) * row + c];
    v = warp_sum(v);
    if constexpr (PEER) v = peer_warp_allreduce(pc, e, idx, v);
    if (lane == 0) t.sums[idx] = v;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    bool last;
    if constexpr (PEER) last = peer_epoch_end(pc, e, gridDim.x);
    else {
      __threadfence();
      last = atomicAdd(t.ticket, 1u) == gridDim.x - 1;
      if (last) *t.ticket = 0u;
    }
    s_last = last ? 1 : 0;
  }
  __syncthreads();
  if (!s_last || !finish) return;
  __threadfence();
  mccl_step_finish_block(t);
}

__global__ void __launch_bounds__(kThreads) mccl_step_finish_kernel(const StepTail t) { mccl_step_finish_block(t); }

// gc_j = (grad_out * dL/dC_j) / (W_j + 1e-7), mu_j . gc_j for the target and augmented rows (one block per row): the
// arithmetic of the separate calls' backward, where autograd hands cal_centroid grad_out * dL/dC.
__global__ void __launch_bounds__(kThreads) mccl_step_bwd_prep_kernel(const float* grad_out, const float* d_cen,
                                                                      const double* sums, int C, float* gc,
                                                                      float* mu_dot_gc) {
  const float g = *grad_out;
  centroid_bwd_prep_row([=](int64_t i) { return g * d_cen[i]; }, sums, 1.0f, C, blockIdx.x, gc, mu_dot_gc);
}

struct StepIn {
  const float* feat_s; const int64_t* labels_s; int64_t batch_s;
  const float* feat_t; const float* pred_t; const int32_t* part_id; int64_t batch_t;
  const float* feat_a; const float* pred_a; int64_t batch_a;
  int64_t channels, pixels;
  int P, K, flags;
  float threshold;
};

bool step_shape_ok(int64_t batch_s, int64_t batch_t, int64_t batch_a, int64_t channels, int64_t pixels, int P, int K) {
  return batch_s > 0 && batch_t > 0 && batch_a >= 0 && channels > 0 && pixels > 0 && K >= 2 && K <= kMaxK && P >= 1 &&
         P * K <= SLCL_MAX_WEIGHT_COLS && (int64_t)(P + 2) * K * (channels + 1) <= INT_MAX;
}

bool step_in_ok(const StepIn& in) {
  if (!step_shape_ok(in.batch_s, in.batch_t, in.batch_a, in.channels, in.pixels, in.P, in.K)) return false;
  if (!in.feat_s || !in.labels_s || !in.feat_t || !in.pred_t) return false;
  if ((in.feat_a == nullptr) != (in.pred_a == nullptr) || (in.feat_a == nullptr) != (in.batch_a == 0)) return false;
  if (in.P > 1 && in.part_id == nullptr) return false;
  return (in.flags & ~(SLCL_SOFT_WEIGHTED | SLCL_SOFT_LOGITS)) == 0;
}

int step_rows(int P, int K, bool aug) { return (P + 1 + (aug ? 1 : 0)) * K; }

size_t step_scratch_bytes(int rows, int P, int K, int64_t C) {
  return align_up((size_t)rows * sizeof(float), 256) + slcl_mccl_losses_workspace_bytes(P, K, C);
}

size_t step_ws_bytes(int64_t batch_s, int64_t batch_t, int64_t batch_a, int64_t C, int64_t HW, int P, int K) {
  size_t b = step_scratch_bytes(step_rows(P, K, batch_a > 0), P, K, C) + kTicketBytes;
  b += class_sums_ws_bytes(batch_s, C, HW, K) - kTicketBytes;
  b += class_sums_ws_bytes(batch_t, C, HW, P * K) - kTicketBytes;
  if (batch_a > 0) b += class_sums_ws_bytes(batch_a, C, HW, K) - kTicketBytes;
  return b;
}

// The loss half of the tail's arguments: centroids, dL/dC and the pair scratch.
void step_loss_args(StepTail& t, int P, bool aug, int split, int bg, int norm, float inter_w, float intra_w, float cnr_w,
                    float* losses, float* d_cen, void* scratch) {
  const size_t kc = (size_t)t.K * t.C;
  t.inv_w = reinterpret_cast<float*>(scratch);
  cpair::McclArgs& a = t.loss;
  a.S = t.cen; a.T = t.cen + kc; a.A = aug ? t.cen + (size_t)(P + 1) * kc : nullptr;
  a.P = P; a.K = t.K; a.C = t.C; a.split = split; a.first = bg ? 0 : 1; a.norm = norm;
  a.inter_w = inter_w; a.intra_w = intra_w; a.cnr_w = cnr_w;
  a.scratch = reinterpret_cast<float*>(reinterpret_cast<char*>(scratch) + align_up((size_t)t.rows * sizeof(float), 256));
  a.loss = losses; a.dS = d_cen; a.dT = d_cen + kc; a.dA = aug ? d_cen + (size_t)(P + 1) * kc : nullptr;
}

// One class-sum sweep per set, each into its own region of `workspace`; fills the reduce half of `t`.
int step_sweeps(const StepIn& in, double* sums, void* workspace, size_t workspace_bytes, cudaStream_t stream, StepTail& t) {
  const bool aug = in.feat_a != nullptr;
  if (workspace_bytes < step_ws_bytes(in.batch_s, in.batch_t, in.batch_a, in.channels, in.pixels, in.P, in.K) ||
      !aligned16(workspace))
    return SLCL_ERR_WORKSPACE;
  t.K = in.K; t.C = (int)in.channels; t.rows = step_rows(in.P, in.K, aug); t.sums = sums;
  char* base = reinterpret_cast<char*>(workspace);
  size_t off = step_scratch_bytes(t.rows, in.P, in.K, in.channels);
  t.ticket = reinterpret_cast<unsigned int*>(base + off);
  off += kTicketBytes;
  const bool logits = (in.flags & SLCL_SOFT_LOGITS) != 0;
  int row = 0;
  for (int s = 0; s < (aug ? 3 : 2); ++s) {
    SumArgs a{};
    a.batch = s == 0 ? in.batch_s : s == 1 ? in.batch_t : in.batch_a;
    a.feat = s == 0 ? in.feat_s : s == 1 ? in.feat_t : in.feat_a;
    a.channels = in.channels; a.pixels = in.pixels;
    a.sb = in.channels * in.pixels; a.sc = in.pixels; a.sp = 1;
    a.n_class = in.K; a.n_part = s == 1 ? in.P : 1; a.n_cols = a.n_part * in.K;
    if (s == 0) {
      a.mode = kHard; a.labels = in.labels_s;
    } else {
      a.mode = kSoft; a.probs = s == 1 ? in.pred_t : in.pred_a;
      a.weighted = in.flags & SLCL_SOFT_WEIGHTED; a.threshold = in.threshold;
      a.part_id = (s == 1 && in.P > 1) ? in.part_id : nullptr;
    }
    a.ticket = t.ticket;
    const bool vec4 = nchw_vec4(a.feat, a.channels, a.pixels, {a.feat, a.labels, a.probs, a.part_id});
    const size_t region = class_sums_ws_bytes(a.batch, in.channels, in.pixels, a.n_cols) - kTicketBytes;
    const int st = launch_sweep(a, vec4, base + off, region, stream, s > 0 && logits, t.n_blocks[s], t.kwt[s]);
    if (st != SLCL_OK) return st;
    t.partial[s] = a.partial;
    row += a.n_cols;
    t.row_end[s] = row;
    off += region;
  }
  for (int s = aug ? 3 : 2; s < kStepMaxSets; ++s) t.row_end[s] = INT_MAX;
  return SLCL_OK;
}

void launch_step_tail(const StepTail& t, const slcl_peer_t* peer, int finish, cudaStream_t stream) {
  const dim3 grid(ceil_div(t.rows * (t.C + 1), kWarps));
  if (peer != nullptr && peer->world > 1)
    mccl_step_tail_kernel<true><<<grid, kThreads, 0, stream>>>(t, peer_ctx(peer), finish);
  else
    mccl_step_tail_kernel<false><<<grid, kThreads, 0, stream>>>(t, PeerCtx{}, finish);
}

}  // namespace
}  // namespace slcl

extern "C" size_t slcl_mccl_step_workspace_bytes(int64_t batch_s, int64_t batch_t, int64_t batch_a, int64_t channels,
                                                 int64_t pixels, int n_partitions, int n_class) {
  if (!step_shape_ok(batch_s, batch_t, batch_a, channels, pixels, n_partitions, n_class)) return 0;
  return step_ws_bytes(batch_s, batch_t, batch_a, channels, pixels, n_partitions, n_class);
}

extern "C" size_t slcl_mccl_step_finish_workspace_bytes(int has_aug, int64_t channels, int n_partitions, int n_class) {
  if (!step_shape_ok(1, 1, has_aug ? 1 : 0, channels, 1, n_partitions, n_class)) return 0;
  return step_scratch_bytes(step_rows(n_partitions, n_class, has_aug != 0), n_partitions, n_class, channels);
}

extern "C" int slcl_mccl_step_fwd(const float* feat_s, const int64_t* labels_s, int64_t batch_s, const float* feat_t,
                                  const float* pred_t, const int32_t* part_id, int64_t batch_t, const float* feat_a,
                                  const float* pred_a, int64_t batch_a, int64_t channels, int64_t pixels, int n_partitions,
                                  int n_class, int flags, float threshold, const float* previous_s, float momentum,
                                  int split, int bg, int norm, float inter_w, float intra_w, float cnr_w, double* sums,
                                  float* centroids, float* losses, float* d_centroids, const slcl_peer_t* peer,
                                  void* workspace, size_t workspace_bytes, slcl_stream_t stream_) {
  const StepIn in{feat_s, labels_s, batch_s, feat_t, pred_t, part_id, batch_t, feat_a, pred_a, batch_a, channels, pixels,
                  n_partitions, n_class, flags, threshold};
  if (!step_in_ok(in) || !sums || !centroids || !losses || !d_centroids || !workspace) return SLCL_ERR_INVALID_ARGUMENT;
  const int rows = step_rows(n_partitions, n_class, feat_a != nullptr);
  if (peer != nullptr) {
    if (!peer_valid(peer)) return SLCL_ERR_INVALID_ARGUMENT;
    if (2 * (int64_t)rows * (channels + 1) > peer->capacity_words) return SLCL_ERR_INVALID_ARGUMENT;
  }
  cudaStream_t stream = (cudaStream_t)stream_;
  StepTail t{};
  int st = step_sweeps(in, sums, workspace, workspace_bytes, stream, t);
  if (st != SLCL_OK) return st;
  t.prev_s = previous_s; t.momentum = momentum; t.cen = centroids;
  step_loss_args(t, n_partitions, feat_a != nullptr, split, bg, norm, inter_w, intra_w, cnr_w, losses, d_centroids, workspace);
  launch_step_tail(t, peer, 1, stream);
  return check_launch("slcl_mccl_step_fwd");
}

extern "C" int slcl_mccl_step_fwd_local(const float* feat_s, const int64_t* labels_s, int64_t batch_s, const float* feat_t,
                                        const float* pred_t, const int32_t* part_id, int64_t batch_t, const float* feat_a,
                                        const float* pred_a, int64_t batch_a, int64_t channels, int64_t pixels,
                                        int n_partitions, int n_class, int flags, float threshold, double* sums,
                                        void* workspace, size_t workspace_bytes, slcl_stream_t stream_) {
  const StepIn in{feat_s, labels_s, batch_s, feat_t, pred_t, part_id, batch_t, feat_a, pred_a, batch_a, channels, pixels,
                  n_partitions, n_class, flags, threshold};
  if (!step_in_ok(in) || !sums || !workspace) return SLCL_ERR_INVALID_ARGUMENT;
  cudaStream_t stream = (cudaStream_t)stream_;
  StepTail t{};
  int st = step_sweeps(in, sums, workspace, workspace_bytes, stream, t);
  if (st != SLCL_OK) return st;
  launch_step_tail(t, nullptr, 0, stream);
  return check_launch("slcl_mccl_step_fwd_local");
}

extern "C" int slcl_mccl_step_finish(const double* sums, int has_aug, int64_t channels, int n_partitions, int n_class,
                                     const float* previous_s, float momentum, int split, int bg, int norm, float inter_w,
                                     float intra_w, float cnr_w, float* centroids, float* losses, float* d_centroids,
                                     void* workspace, size_t workspace_bytes, slcl_stream_t stream_) {
  if (!step_shape_ok(1, 1, has_aug ? 1 : 0, channels, 1, n_partitions, n_class)) return SLCL_ERR_INVALID_ARGUMENT;
  if (!sums || !centroids || !losses || !d_centroids || !workspace) return SLCL_ERR_INVALID_ARGUMENT;
  if (workspace_bytes < slcl_mccl_step_finish_workspace_bytes(has_aug, channels, n_partitions, n_class) ||
      !aligned16(workspace))
    return SLCL_ERR_WORKSPACE;
  StepTail t{};
  t.K = n_class; t.C = (int)channels; t.rows = step_rows(n_partitions, n_class, has_aug != 0);
  t.sums = const_cast<double*>(sums);
  t.prev_s = previous_s; t.momentum = momentum; t.cen = centroids;
  step_loss_args(t, n_partitions, has_aug != 0, split, bg, norm, inter_w, intra_w, cnr_w, losses, d_centroids, workspace);
  mccl_step_finish_kernel<<<1, kThreads, 0, (cudaStream_t)stream_>>>(t);
  return check_launch("slcl_mccl_step_finish");
}

extern "C" int slcl_mccl_step_bwd(const float* feat_t, const float* pred_t, const int32_t* part_id, int64_t batch_t,
                                  const float* feat_a, const float* pred_a, int64_t batch_a, int64_t channels,
                                  int64_t pixels, int n_partitions, int n_class, int flags, float threshold,
                                  const double* sums, const float* d_centroids, const float* grad_out, float* dfeat_t,
                                  float* dpred_t, float* dfeat_a, float* dpred_a, void* workspace, size_t workspace_bytes,
                                  slcl_stream_t stream_) {
  if (!step_shape_ok(1, batch_t, batch_a, channels, pixels, n_partitions, n_class) || !feat_t || !pred_t)
    return SLCL_ERR_INVALID_ARGUMENT;
  if ((feat_a == nullptr) != (pred_a == nullptr) || (feat_a == nullptr) != (batch_a == 0)) return SLCL_ERR_INVALID_ARGUMENT;
  if ((flags & ~(SLCL_SOFT_WEIGHTED | SLCL_SOFT_LOGITS)) != 0 || (n_partitions > 1 && part_id == nullptr))
    return SLCL_ERR_INVALID_ARGUMENT;
  if (!sums || !d_centroids || !grad_out || !dfeat_t || (feat_a != nullptr && !dfeat_a)) return SLCL_ERR_INVALID_ARGUMENT;
  if ((dpred_t != nullptr || dpred_a != nullptr) && !(flags & SLCL_SOFT_WEIGHTED)) return SLCL_ERR_INVALID_ARGUMENT;
  const bool aug = feat_a != nullptr;
  const int K = n_class, C = (int)channels;
  const int g_rows = step_rows(n_partitions, K, aug) - K;            // target partitions + augmented target
  if (workspace_bytes < slcl_centroid_bwd_workspace_bytes(channels, g_rows) || !aligned16(workspace))
    return SLCL_ERR_WORKSPACE;
  cudaStream_t stream = (cudaStream_t)stream_;
  float* gc = reinterpret_cast<float*>(workspace);
  float* mu_dot_gc = gc + (size_t)g_rows * C;
  mccl_step_bwd_prep_kernel<<<g_rows, kThreads, 0, stream>>>(grad_out, d_centroids + (size_t)K * C, sums + (size_t)K * (C + 1),
                                                             C, gc, mu_dot_gc);
  const bool logits = (flags & SLCL_SOFT_LOGITS) != 0;
  for (int s = 1; s <= (aug ? 2 : 1); ++s) {
    CenBwdArgs a{};
    a.s.feat = s == 1 ? feat_t : feat_a;
    a.s.batch = s == 1 ? batch_t : batch_a; a.s.channels = channels; a.s.pixels = pixels;
    a.s.sb = channels * pixels; a.s.sc = pixels; a.s.sp = 1;
    a.s.mode = kSoft; a.s.probs = s == 1 ? pred_t : pred_a;
    a.s.weighted = flags & SLCL_SOFT_WEIGHTED; a.s.threshold = threshold;
    a.s.part_id = (s == 1 && n_partitions > 1) ? part_id : nullptr;
    a.s.n_part = s == 1 ? n_partitions : 1; a.s.n_class = K; a.s.n_cols = a.s.n_part * K;
    const size_t row0 = s == 1 ? 0 : (size_t)n_partitions * K;
    a.gc = gc + row0 * C; a.mu_dot_gc = mu_dot_gc + row0;
    a.dfeat = s == 1 ? dfeat_t : dfeat_a; a.dprobs = s == 1 ? dpred_t : dpred_a;
    const bool vec4 = nchw_vec4(a.s.feat, channels, pixels, {a.s.feat, a.s.probs, a.s.part_id, a.dfeat, a.dprobs});
    const int st = launch_centroid_bwd(a, vec4, logits, stream);
    if (st != SLCL_OK) return st;
  }
  return check_launch("slcl_mccl_step_bwd");
}
