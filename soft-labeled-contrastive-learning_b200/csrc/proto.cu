// proto.cu -- prototype path: pixel -> class-centre margin InfoNCE (fwd + bwd)
// and pseudo-label generation, straight from the NCHW feature map.
//
// Replaces (reference, file:line):
//   MPCL.forward              utils/loss.py:484-573
//   mpcl_loss_calc            utils/loss.py:576-605   (normalise + NCHW->NHWC copy fused away)
//   generate_pseudo_label     utils/utils_.py:597-624
// Closed forms: SURVEY.md appendix A.1 / A.2.
//
// Roofline: HBM.  One thread owns VEC (=4) consecutive pixels and walks the C
// channel planes with 128-bit streaming loads (coalesced along HW), keeping the
// squared norm and the K dot products in registers; the K unit centres sit in
// shared memory and are read as warp-wide broadcasts.  Forward reads F once
// (4C B/px) and stashes K+1 backward coefficients per pixel; backward reads F
// and the stash and writes dF (8C B/px).  Nothing of size [N,C] or [N,K] is
// materialised besides dF itself.
#include "common.cuh"
#include "peer.cuh"
#include "proto_math.cuh"

#include <math.h>
#include <stdlib.h>

namespace slcl {
namespace {

#ifndef SLCL_PROTO_THREADS
#define SLCL_PROTO_THREADS 256
#endif
constexpr int kThreads = SLCL_PROTO_THREADS;
#ifndef SLCL_FWD_UNROLL
#define SLCL_FWD_UNROLL 8
#endif
#ifndef SLCL_BWD_UNROLL
#define SLCL_BWD_UNROLL 8
#endif
#ifndef SLCL_FWD_MINBLK
#define SLCL_FWD_MINBLK 3
#endif
#ifndef SLCL_BWD_MINBLK
#define SLCL_BWD_MINBLK 3
#endif
#ifndef SLCL_MPSCL_L2_BOTH
#define SLCL_MPSCL_L2_BOTH 0      // 1: the MPSCL step keeps both maps in L2 when only each one alone fits (slower, DESIGN §3)
#endif
constexpr int kUnroll = SLCL_FWD_UNROLL;      // channel planes in flight per thread (8 x 16 B)
constexpr int kUnrollBwd = SLCL_BWD_UNROLL;

struct ProtoArgs {
  const float* feat;
  int64_t batch, channels, pixels, sb, sc, sp;
  int64_t n_total;            // batch * pixels
  const int64_t* labels;
  const float* soft_mask;
  const float* sel;
  const float* cstate;        // [K*C] unit centres, [K] norms
  float* stash;               // [(K+1) * N]
  double2* partial;           // per block {sum sel*row, sum sel}
  int64_t* out_label;         // pseudo-label mode
  float* out_sel;
  float sel_threshold;
  int fused_target;           // forward derives label/sel itself (generate_pseudo_label fused in) and writes them out
  int keep_l2;                // the map fits in L2: load it with evict_last so the backward's read of F hits L2
  int reverse;                // walk the pixel blocks back to front (forward kernels of L2-sized maps: zig-zag with the
                              // class-sum sweep in front and the backward behind, each starts where its predecessor ended)
  MarginConst mc;
};

template <int VEC> struct Vec;
template <> struct Vec<4> {
  static __device__ __forceinline__ void load(const float* p, float (&v)[4]) {
    float4 t = ld_stream4(p); v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
  }
  static __device__ __forceinline__ void load_keep(const float* p, float (&v)[4]) {
    float4 t = *reinterpret_cast<const float4*>(p); v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
  }
  static __device__ __forceinline__ void load_pol(const float* p, float (&v)[4], uint64_t pol) {
    float4 t = ld_policy4(p, pol); v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
  }
  static __device__ __forceinline__ void store(float* p, const float (&v)[4]) {
    st_stream4(p, make_float4(v[0], v[1], v[2], v[3]));
  }
  static __device__ __forceinline__ void store_keep(float* p, const float (&v)[4]) {
    *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2], v[3]);
  }
};
template <> struct Vec<1> {
  static __device__ __forceinline__ void load(const float* p, float (&v)[1]) { v[0] = ld_stream1(p); }
  static __device__ __forceinline__ void load_keep(const float* p, float (&v)[1]) { v[0] = *p; }
  static __device__ __forceinline__ void load_pol(const float* p, float (&v)[1], uint64_t pol) { v[0] = ld_policy1(p, pol); }
  static __device__ __forceinline__ void store(float* p, const float (&v)[1]) { st_stream1(p, v[0]); }
  static __device__ __forceinline__ void store_keep(float* p, const float (&v)[1]) { *p = v[0]; }
};

template <int K> constexpr int kpad() { return K <= 4 ? 4 : 8; }

// Unit centres -> shared memory as sC[c][KP] so one or two 128-bit broadcast
// loads fetch all K values of a channel.
template <int K>
__device__ __forceinline__ void load_centres_smem(float* sC, const float* cstate, int C) {
  constexpr int KP = kpad<K>();
  for (int idx = threadIdx.x; idx < C * KP; idx += blockDim.x) {
    int c = idx / KP, k = idx % KP;
    sC[idx] = (k < K) ? cstate[(int64_t)k * C + c] : 0.f;
  }
}

template <int K>
__device__ __forceinline__ void centre_row(const float* sC, int c, float (&ck)[K]) {
  constexpr int KP = kpad<K>();
  const float4* row = reinterpret_cast<const float4*>(sC + (size_t)c * KP);
  float4 a = row[0];
  float tmp[8];
  tmp[0] = a.x; tmp[1] = a.y; tmp[2] = a.z; tmp[3] = a.w;
  if (K > 4) { float4 b = row[1]; tmp[4] = b.x; tmp[5] = b.y; tmp[6] = b.z; tmp[7] = b.w; }
#pragma unroll
  for (int k = 0; k < K; ++k) ck[k] = tmp[k];
}

// Pixel-group addressing shared by every kernel in this file: `bid` is the block's index within its map (the
// two-map kernels of the MPSCL step run one map per segment of their grid).
template <int VEC>
__device__ __forceinline__ bool locate_at(const ProtoArgs& a, int64_t bid, int64_t& pix, int64_t& offset) {
  int64_t g = bid * blockDim.x + threadIdx.x;
  int64_t groups_per_image = a.pixels / VEC;
  if (g >= a.batch * groups_per_image) { pix = 0; offset = 0; return false; }
  int64_t b = g / groups_per_image;
  int64_t p = (g - b * groups_per_image) * VEC;
  pix = b * a.pixels + p;
  offset = b * a.sb + p * a.sp;
  return true;
}
template <int VEC>
__device__ __forceinline__ bool locate(const ProtoArgs& a, int64_t& pix, int64_t& offset) {
  const int64_t bid = a.reverse ? (int64_t)(gridDim.x - 1 - blockIdx.x) : (int64_t)blockIdx.x;
  return locate_at<VEC>(a, bid, pix, offset);
}

// Which block of its map this block is, evaluated where the kernel needs it.  WholeGrid: the grid is the map
// (walked back to front with a.reverse); Segment: blocks [first, first + n) of the grid are the map.
struct WholeGrid {
  __device__ __forceinline__ int64_t bid(const ProtoArgs& a) const {
    return a.reverse ? (int64_t)(gridDim.x - 1 - blockIdx.x) : (int64_t)blockIdx.x;
  }
  __device__ __forceinline__ unsigned int slot(const ProtoArgs& a) const {
    return a.reverse ? gridDim.x - 1 - blockIdx.x : blockIdx.x;
  }
};
struct Segment {
  unsigned int first, n;
  __device__ __forceinline__ unsigned int slot(const ProtoArgs& a) const {
    return a.reverse ? first + n - 1 - blockIdx.x : blockIdx.x - first;
  }
  __device__ __forceinline__ int64_t bid(const ProtoArgs& a) const { return (int64_t)slot(a); }
};

// Accumulate squared norm and K dot products over all channels.
template <int K, int VEC>
__device__ __forceinline__ void channel_pass(const float* base, int64_t sc, int C, const float* sC,
                                             float (&nrm)[VEC], float (&dot)[K][VEC], uint64_t pol) {
#pragma unroll
  for (int v = 0; v < VEC; ++v) {
    nrm[v] = 0.f;
#pragma unroll
    for (int k = 0; k < K; ++k) dot[k][v] = 0.f;
  }
  int c = 0;
  for (; c + kUnroll <= C; c += kUnroll) {
    float x[kUnroll][VEC];
#pragma unroll
    for (int u = 0; u < kUnroll; ++u) Vec<VEC>::load_pol(base + (int64_t)(c + u) * sc, x[u], pol);
#pragma unroll
    for (int u = 0; u < kUnroll; ++u) {
      float ck[K];
      centre_row<K>(sC, c + u, ck);
#pragma unroll
      for (int v = 0; v < VEC; ++v) {
        nrm[v] = fmaf(x[u][v], x[u][v], nrm[v]);
#pragma unroll
        for (int k = 0; k < K; ++k) dot[k][v] = fmaf(x[u][v], ck[k], dot[k][v]);
      }
    }
  }
  for (; c < C; ++c) {
    float x[VEC];
    Vec<VEC>::load_pol(base + (int64_t)c * sc, x, pol);
    float ck[K];
    centre_row<K>(sC, c, ck);
#pragma unroll
    for (int v = 0; v < VEC; ++v) {
      nrm[v] = fmaf(x[v], x[v], nrm[v]);
#pragma unroll
      for (int k = 0; k < K; ++k) dot[k][v] = fmaf(x[v], ck[k], dot[k][v]);
    }
  }
}

// ---------------------------------------------------------------------------
// forward: loss rows + stash
// ---------------------------------------------------------------------------
// One block's pixels of one map (the centres already in sC): loss rows, stash, and the block's partial, indexed by its
// pixel range.
template <int K, int VEC, class Blk>
__device__ __forceinline__ void proto_fwd_block(const ProtoArgs& a, const float* sC, double (*red)[kThreads / 32], int C,
                                                Blk blk) {
  int64_t pix, off;
  const bool active = locate_at<VEC>(a, blk.bid(a), pix, off);
  double loss_acc = 0.0, sel_acc = 0.0;
  if (active) {
    float nrm[VEC], dot[K][VEC];
    channel_pass<K, VEC>(a.feat + off, a.sc, C, sC, nrm, dot, l2_policy(a.keep_l2 != 0));

    float selv[VEC];
    if (a.sel != nullptr) Vec<VEC>::load_keep(a.sel + pix, selv);
    else {
#pragma unroll
      for (int v = 0; v < VEC; ++v) selv[v] = 1.0f;
    }
    long long lab[VEC];
    if (a.labels != nullptr) {
      if constexpr (VEC == 4) {
        const longlong2* lp = reinterpret_cast<const longlong2*>(a.labels + pix);
        longlong2 l0 = lp[0], l1 = lp[1];
        lab[0] = l0.x; lab[1] = l0.y; lab[2] = l1.x; lab[3] = l1.y;
      } else {
        lab[0] = a.labels[pix];
      }
    }
    if (a.fused_target) {
      // generate_pseudo_label (utils/utils_.py:597-624) on the cosines already in registers: same
      // arithmetic as pseudo_label_kernel (dot / n, strict >, first index wins ties)
#pragma unroll
      for (int v = 0; v < VEC; ++v) {
        const float n = fmaxf(sqrtf(nrm[v]), 1e-12f);
        float t1 = -INFINITY, t2 = -INFINITY;
        int best = 0;
#pragma unroll
        for (int k = 0; k < K; ++k) {
          const float cs = dot[k][v] / n;
          if (cs > t1) { t2 = t1; t1 = cs; best = k; }
          else if (cs > t2) { t2 = cs; }
        }
        lab[v] = best;
        selv[v] = (t1 - t2 > a.sel_threshold) ? 1.0f : 0.0f;
      }
      if constexpr (VEC == 4) {
        longlong2* lp = reinterpret_cast<longlong2*>(a.out_label + pix);
        lp[0] = make_longlong2(lab[0], lab[1]);
        lp[1] = make_longlong2(lab[2], lab[3]);
      } else {
        a.out_label[pix] = lab[0];
      }
      Vec<VEC>::store_keep(a.out_sel + pix, selv);
    }
    // soft positives (caller-supplied mask [N,K] row-major, :516-517): the VEC pixels of this thread own VEC*K consecutive
    // floats -- fetched as 128-bit loads (the first version gathered them one float at a time with a stride of K)
    float msoft[VEC * K];
    if (a.labels == nullptr && !a.fused_target) {
      const float* mp = a.soft_mask + pix * K;
      if constexpr (VEC == 4) {
#pragma unroll
        for (int q = 0; q < K; ++q) {
          const float4 t = *reinterpret_cast<const float4*>(mp + 4 * q);
          msoft[4 * q] = t.x; msoft[4 * q + 1] = t.y; msoft[4 * q + 2] = t.z; msoft[4 * q + 3] = t.w;
        }
      } else {
#pragma unroll
        for (int q = 0; q < K; ++q) msoft[q] = mp[q];
      }
    }
    float out[K + 1][VEC];
#pragma unroll
    for (int v = 0; v < VEC; ++v) {
      const float n = a.mc.normalize ? fmaxf(sqrtf(nrm[v]), 1e-12f) : 1.0f;   // F.normalize eps (:595)
      const float inv_n = 1.0f / n;
      float cosv[K], M[K], coef[K + 1];
#pragma unroll
      for (int k = 0; k < K; ++k) {
        cosv[k] = dot[k][v] * inv_n;
        if (!(a.labels == nullptr && !a.fused_target)) M[k] = (lab[v] == (long long)k) ? 1.0f : 0.0f;   // :513
        else M[k] = msoft[v * K + k];                                                  // :517
      }
      float row = margin_row<K>(cosv, M, selv[v], inv_n, a.mc, coef);
      loss_acc += (double)(selv[v] * row);
      sel_acc += (double)selv[v];
#pragma unroll
      for (int k = 0; k <= K; ++k) out[k][v] = coef[k];
    }
#pragma unroll
    for (int k = 0; k <= K; ++k) Vec<VEC>::store_keep(a.stash + (int64_t)k * a.n_total + pix, out[k]);
  }
  // deterministic block partial
  loss_acc = warp_sum(loss_acc);
  sel_acc = warp_sum(sel_acc);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (lane == 0) { red[0][warp] = loss_acc; red[1][warp] = sel_acc; }
  __syncthreads();
  if (threadIdx.x == 0) {
    double l = 0.0, s = 0.0;
#pragma unroll
    for (int w = 0; w < kThreads / 32; ++w) { l += red[0][w]; s += red[1][w]; }
    a.partial[blk.slot(a)] = make_double2(l, s);      // indexed by pixel range
  }
}

template <int K, int VEC>
__global__ void __launch_bounds__(kThreads, (K <= 5 && VEC == 4) ? SLCL_FWD_MINBLK : 1) proto_fwd_kernel(const ProtoArgs a) {
  pdl_trigger();
  pdl_wait();
  extern __shared__ __align__(16) float sC[];
  __shared__ double red[2][kThreads / 32];
  const int C = (int)a.channels;
  load_centres_smem<K>(sC, a.cstate, C);
  __syncthreads();
  proto_fwd_block<K, VEC>(a, sC, red, C, WholeGrid{});
}

// Blocks per SM of the two-map kernels: the single-map kernels' 3 where both bodies fit the 80 registers that leaves
// without spilling (ptxas -v), else 2.
constexpr int mpscl_fwd_minblk(int K, int VEC) { return VEC == 4 && K <= 5 ? ((K == 2 || K == 4) ? SLCL_FWD_MINBLK : 2) : 1; }
constexpr int mpscl_bwd_minblk(int K, int VEC) { return VEC == 4 && K <= 5 ? (K == 4 ? 2 : SLCL_BWD_MINBLK) : 1; }

// The MPSCL step's prototype forward over BOTH maps in one launch: blocks [0, nb_s) run the source map `s` (hard labels,
// source margin constants), blocks [nb_s, nb_s + nb_t) the fused target map `t` (pseudo label and mask written out,
// target constants).  Each map keeps the block decomposition, partial indexing and walk direction proto_fwd_kernel gives
// it, so each map's sums are the single-map launch's.  Both maps share the centres (one cstate).

template <int K, int VEC>
__global__ void __launch_bounds__(kThreads, mpscl_fwd_minblk(K, VEC))
    mpscl_fwd_kernel(const ProtoArgs s, const ProtoArgs t, int nb_s, int nb_t) {
  pdl_trigger();
  pdl_wait();
  extern __shared__ __align__(16) float sC[];
  __shared__ double red[2][kThreads / 32];
  const int C = (int)s.channels;
  load_centres_smem<K>(sC, s.cstate, C);
  __syncthreads();
  if (blockIdx.x < (unsigned int)nb_s) proto_fwd_block<K, VEC>(s, sC, red, C, Segment{0u, (unsigned int)nb_s});
  else proto_fwd_block<K, VEC>(t, sC, red, C, Segment{(unsigned int)nb_s, (unsigned int)nb_t});
}

// Sums the block partials in index order (deterministic) and writes
// scal = {loss, coefficient, weight sum, weighted row-loss sum}.
// Data-parallel (pc.world > 1): the pair {weight sum, weighted row-loss sum} is exchanged with the other ranks right
// here, through the NVLink peer mailboxes (peer.cuh) -- the same words slcl_proto_rescale_peer would send, added in the
// same rank order -- so the forward needs no extra launch (and no collective) to return the GLOBAL loss.
// split != 0: SEND only -- scal[2..3] keep the LOCAL pair, the epoch goes to mailbox word 4, and proto_bwd_kernel
// (launched with the same mailboxes) receives, adds and publishes: the exchange latency hides behind its launch + prologue.
// The block partials of one map summed in index order (deterministic); the totals are valid on thread 0.
__device__ __forceinline__ void sum_partials(const double2* partial, int n_blocks, double (*red)[kThreads / 32], double& l,
                                             double& s) {
  l = 0.0; s = 0.0;
  for (int i = threadIdx.x; i < n_blocks; i += kThreads) { double2 p = partial[i]; l += p.x; s += p.y; }
  l = warp_sum(l); s = warp_sum(s);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (lane == 0) { red[0][warp] = l; red[1][warp] = s; }
  __syncthreads();
  if (threadIdx.x == 0) {
    l = 0.0; s = 0.0;
    for (int w = 0; w < kThreads / 32; ++w) { l += red[0][w]; s += red[1][w]; }
  }
}

// scal = {loss, coefficient, weight sum, weighted row-loss sum} from the (global) pair.
__device__ __forceinline__ void write_scal(float* scal, int has_sel, float wsum, float lsum) {
  // with pixel_sel_loc: sum / (sum(sel) + 1e-4) (:565); else mean over N (:571)
  const float coef = has_sel ? 1.0f / (wsum + 1e-4f) : 1.0f / wsum;
  scal[0] = lsum * coef;
  scal[1] = coef;
  scal[2] = wsum;
  scal[3] = lsum;
}

__global__ void __launch_bounds__(kThreads) proto_finalize_kernel(const double2* partial, int n_blocks, int64_t n_total,
                                                                   int has_sel, float* scal, const PeerCtx pc, int split) {
  pdl_trigger();
  pdl_wait();
  __shared__ double red[2][kThreads / 32];
  __shared__ float s_pair[2];
  __shared__ float s_vals[2 * kMaxPeers];
  __shared__ int s_bad;
  double l, s;
  sum_partials(partial, n_blocks, red, l, s);
  if (threadIdx.x == 0) {
    s_pair[0] = has_sel ? (float)s : (float)n_total;
    s_pair[1] = (float)l;
    s_bad = 0;
  }
  __syncthreads();
  float wsum = s_pair[0], lsum = s_pair[1];
  if (pc.world > 1 && split) {
    const unsigned int e = peer_epoch_begin(pc);
    const int t = threadIdx.x;
    if (t < 2 * pc.world) peer_send(pc, e, t >> 1, t & 1, __float_as_uint(s_pair[t & 1]));
    if (t == 0) pc.boxes[pc.rank][4] = (unsigned long long)e;           // pending: completed by the backward kernel
  } else if (pc.world > 1) {
    const unsigned int e = peer_epoch_begin(pc);
    const int t = threadIdx.x;
    if (t < 2 * pc.world) {
      bool ok;
      const unsigned int got = peer_send_recv(pc, e, t >> 1, t & 1, __float_as_uint(s_pair[t & 1]), ok);
      s_vals[t] = __uint_as_float(got);
      if (!ok) s_bad = 1;
    }
    __syncthreads();
    if (t == 0) {
      wsum = 0.f; lsum = 0.f;
      for (int r = 0; r < pc.world; ++r) { wsum += s_vals[2 * r]; lsum += s_vals[2 * r + 1]; }
      if (s_bad) { wsum = __uint_as_float(0x7FC00000u); lsum = wsum; }      // a peer never arrived: poison, do not hang
      peer_epoch_end(pc, e, 1u);
    }
  }
  if (threadIdx.x == 0) write_scal(scal, has_sel, wsum, lsum);
}

// The MPSCL step's finaliser: both maps' partials summed as proto_finalize_kernel sums them, then ONE exchange of both
// pairs (thread 4p+v sends word v of {source weight sum, source row-loss sum, target weight sum, target row-loss sum}
// to rank p), added in rank order as proto_finalize_kernel adds them.  The source has no pixel selection (its weight sum
// is its pixel count), the target is weighted by its mask.  pairs != null (the NCCL route): the LOCAL quadruple goes
// there for the caller's all-reduce and mpscl_finish_kernel, and scal is left alone.
__global__ void __launch_bounds__(kThreads) mpscl_finalize_kernel(const double2* part_s, int nb_s, int64_t n_s,
                                                                   const double2* part_t, int nb_t, float* scal_s,
                                                                   float* scal_t, float* pairs, const PeerCtx pc) {
  pdl_trigger();
  pdl_wait();
  __shared__ double red_s[2][kThreads / 32], red_t[2][kThreads / 32];
  __shared__ float s_q[4];
  __shared__ float s_vals[4 * kMaxPeers];
  __shared__ int s_bad;
  double l, s;
  sum_partials(part_s, nb_s, red_s, l, s);
  if (threadIdx.x == 0) { s_q[0] = (float)n_s; s_q[1] = (float)l; }
  sum_partials(part_t, nb_t, red_t, l, s);
  if (threadIdx.x == 0) { s_q[2] = (float)s; s_q[3] = (float)l; s_bad = 0; }
  __syncthreads();
  float q[4] = {s_q[0], s_q[1], s_q[2], s_q[3]};
  if (pc.world > 1) {
    const unsigned int e = peer_epoch_begin(pc);
    const int t = threadIdx.x;
    if (t < 4 * pc.world) {
      bool ok;
      const unsigned int got = peer_send_recv(pc, e, t >> 2, t & 3, __float_as_uint(s_q[t & 3]), ok);
      s_vals[t] = __uint_as_float(got);
      if (!ok) s_bad = 1;
    }
    __syncthreads();
    if (t == 0) {
      for (int v = 0; v < 4; ++v) q[v] = 0.f;
      for (int r = 0; r < pc.world; ++r)
        for (int v = 0; v < 4; ++v) q[v] += s_vals[4 * r + v];
      if (s_bad)       // a peer never arrived: poison, do not hang
        for (int v = 0; v < 4; ++v) q[v] = __uint_as_float(0x7FC00000u);
      peer_epoch_end(pc, e, 1u);
    }
  }
  if (threadIdx.x == 0) {
    if (pairs != nullptr) {
      for (int v = 0; v < 4; ++v) pairs[v] = q[v];
    } else {
      write_scal(scal_s, 0, q[0], q[1]);
      write_scal(scal_t, 1, q[2], q[3]);
    }
  }
}

// NCCL route: after the caller's all-reduce of the four pair words, the two global quadruples.
__global__ void mpscl_finish_kernel(const float* pairs, float* scal_s, float* scal_t) {
  pdl_trigger();
  pdl_wait();
  if (threadIdx.x == 0 && blockIdx.x == 0) {
    write_scal(scal_s, 0, pairs[0], pairs[1]);
    write_scal(scal_t, 1, pairs[2], pairs[3]);
  }
}

// After a cross-rank all-reduce of scal[2..3] (weight sum, weighted row-loss sum):
// recompute the global loss and coefficient in place.
__global__ void proto_rescale_kernel(float* scal, int has_sel) {
  pdl_trigger();
  pdl_wait();
  if (threadIdx.x == 0 && blockIdx.x == 0) {
    float coef = has_sel ? 1.0f / (scal[2] + 1e-4f) : 1.0f / scal[2];
    scal[0] = scal[3] * coef;
    scal[1] = coef;
  }
}

// The same exchange + rescale as ONE kernel over NVLink peer memory (no NCCL launch between forward and backward):
// protocol and mailbox layout in peer.cuh.  Thread 2p+v sends value v (0 = weight sum, 1 = weighted row-loss sum) to
// rank p's mailbox and waits for rank p's value v in its own; thread 0 then adds in rank order (identical on every
// rank) and writes scal[0..3].
__global__ void __launch_bounds__(64) proto_rescale_peer_kernel(float* scal, int has_sel, const PeerCtx pc) {
  pdl_trigger();
  pdl_wait();
  __shared__ float vals[2 * kMaxPeers];
  __shared__ int s_bad;
  const unsigned int e = peer_epoch_begin(pc);
  const int t = threadIdx.x;
  if (t == 0) s_bad = 0;
  __syncthreads();
  if (t < 2 * pc.world) {
    bool ok;
    const unsigned int got = peer_send_recv(pc, e, t >> 1, t & 1, __float_as_uint(scal[2 + (t & 1)]), ok);
    vals[t] = __uint_as_float(got);
    if (!ok) s_bad = 1;
  }
  __syncthreads();
  if (t == 0) {
    float wsum = 0.f, lsum = 0.f;
    for (int r = 0; r < pc.world; ++r) { wsum += vals[2 * r]; lsum += vals[2 * r + 1]; }
    if (s_bad) { wsum = __uint_as_float(0x7FC00000u); lsum = wsum; }      // a peer never arrived: poison, do not hang
    const float coef = has_sel ? 1.0f / (wsum + 1e-4f) : 1.0f / wsum;
    scal[0] = lsum * coef;
    scal[1] = coef;
    scal[2] = wsum;
    scal[3] = lsum;
    peer_epoch_end(pc, e, 1u);
  }
}

// In-place all-reduce (sum) of n doubles across the ranks: one warp per element.
__global__ void __launch_bounds__(256) peer_allreduce_f64_kernel(double* buf, long long n, const PeerCtx pc) {
  const unsigned int e = peer_epoch_begin(pc);
  const long long idx = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
  if (idx < n) {
    const double t = peer_warp_allreduce(pc, e, idx, buf[idx]);
    if ((threadIdx.x & 31) == 0) buf[idx] = t;
  }
  __syncthreads();
  if (threadIdx.x == 0) peer_epoch_end(pc, e, gridDim.x);
}

// ---------------------------------------------------------------------------
// backward: dF = gamma * ( sum_k a_k chat_k - b x )
// ---------------------------------------------------------------------------
// One block's pixels of one map (block `bid` of that map; the centres already in sC), a_k and b from the stash.
// gamma = grad_out[0] * (*coef), coef in shared memory.
template <int K, int VEC, class Blk>
__device__ __forceinline__ void proto_bwd_block(const ProtoArgs& a, const float* sC, int C, Blk blk, const float* grad_out,
                                                const float* coef_, float* dfeat) {
  int64_t pix, off;
  if (!locate_at<VEC>(a, blk.bid(a), pix, off)) return;
  const float gamma = grad_out[0] * *coef_;
  float coef[K + 1][VEC];
#pragma unroll
  for (int k = 0; k <= K; ++k) {
    Vec<VEC>::load(a.stash + (int64_t)k * a.n_total + pix, coef[k]);
#pragma unroll
    for (int v = 0; v < VEC; ++v) coef[k][v] *= gamma;
  }
  const float* src = a.feat + off;
  float* dst = dfeat + off;
  int c = 0;
  for (; c + kUnrollBwd <= C; c += kUnrollBwd) {
    float x[kUnrollBwd][VEC];
#pragma unroll
    for (int u = 0; u < kUnrollBwd; ++u) Vec<VEC>::load(src + (int64_t)(c + u) * a.sc, x[u]);
#pragma unroll
    for (int u = 0; u < kUnrollBwd; ++u) {
      float ck[K];
      centre_row<K>(sC, c + u, ck);
      float o[VEC];
#pragma unroll
      for (int v = 0; v < VEC; ++v) {
        float acc = -coef[K][v] * x[u][v];
#pragma unroll
        for (int k = 0; k < K; ++k) acc = fmaf(coef[k][v], ck[k], acc);
        o[v] = acc;
      }
      Vec<VEC>::store(dst + (int64_t)(c + u) * a.sc, o);
    }
  }
  for (; c < C; ++c) {
    float x[VEC], ck[K], o[VEC];
    Vec<VEC>::load(src + (int64_t)c * a.sc, x);
    centre_row<K>(sC, c, ck);
#pragma unroll
    for (int v = 0; v < VEC; ++v) {
      float acc = -coef[K][v] * x[v];
#pragma unroll
      for (int k = 0; k < K; ++k) acc = fmaf(coef[k][v], ck[k], acc);
      o[v] = acc;
    }
    Vec<VEC>::store(dst + (int64_t)c * a.sc, o);
  }
}

template <int K, int VEC>
__global__ void __launch_bounds__(kThreads, (K <= 5 && VEC == 4) ? SLCL_BWD_MINBLK : 1) proto_bwd_kernel(const ProtoArgs a, float* scal, const float* grad_out,
                                                             float* dfeat, const PeerCtx pc, int has_sel) {
  pdl_trigger();
  pdl_wait();
  extern __shared__ __align__(16) float sC[];
  __shared__ float s_coef;
  __shared__ float s_vals[2 * kMaxPeers];
  const int C = (int)a.channels;
  load_centres_smem<K>(sC, a.cstate, C);
  if (pc.world > 1) {
    // second half of a split-phase exchange (proto_finalize_kernel sent this rank's pair and left the epoch in word 4):
    // block 0 receives every rank's pair, adds in rank order, rewrites scal and publishes the epoch in word 3; the other
    // blocks wait for that word.  By now the wire latency has been overlapped with this kernel's launch and prologue.
    unsigned long long* mine = pc.boxes[pc.rank];
    const unsigned int e = (unsigned int)(*reinterpret_cast<volatile unsigned long long*>(mine + 4));
    const int t = threadIdx.x;
    if (blockIdx.x == 0) {
      bool ok = true;
      if (t < 2 * pc.world) s_vals[t] = __uint_as_float(peer_recv(pc, e, t >> 1, t & 1, ok));
      const int bad = __syncthreads_or(!ok);
      if (t == 0) {
        float wsum = 0.f, lsum = 0.f;
        for (int r = 0; r < pc.world; ++r) { wsum += s_vals[2 * r]; lsum += s_vals[2 * r + 1]; }
        if (bad) { wsum = __uint_as_float(0x7FC00000u); lsum = wsum; }
        const float coef = has_sel ? 1.0f / (wsum + 1e-4f) : 1.0f / wsum;
        scal[0] = lsum * coef; scal[1] = coef; scal[2] = wsum; scal[3] = lsum;
        s_coef = coef;
        __threadfence();
        *reinterpret_cast<volatile unsigned long long*>(mine + 3) = (unsigned long long)e;       // ready
        peer_epoch_end(pc, e, 1u);
      }
    } else if (t == 0) {
      while ((unsigned int)(*reinterpret_cast<volatile unsigned long long*>(mine + 3)) != e) { }
      __threadfence();
      s_coef = *reinterpret_cast<volatile float*>(scal + 1);
    }
  } else if (threadIdx.x == 0) {
    s_coef = scal[1];
  }
  __syncthreads();
  proto_bwd_block<K, VEC>(a, sC, C, WholeGrid{}, grad_out, &s_coef, dfeat);
}

// The MPSCL step's backward over both maps in one launch: blocks [0, nb_s) write dF_s from the source stash and scal_s,
// blocks [nb_s, nb_s + nb_t) dF_t from the target's; both maps share the centres.  A map whose loss got no gradient is
// launched with no blocks.
template <int K, int VEC>
__global__ void __launch_bounds__(kThreads, mpscl_bwd_minblk(K, VEC))
    mpscl_bwd_kernel(const ProtoArgs s, const ProtoArgs t, int nb_s, int nb_t, const float* scal_s, const float* scal_t,
                     const float* grad_s, const float* grad_t, float* dfeat_s, float* dfeat_t) {
  pdl_trigger();
  pdl_wait();
  extern __shared__ __align__(16) float sC[];
  __shared__ float s_coef;
  const int C = (int)s.channels;
  load_centres_smem<K>(sC, s.cstate, C);
  const bool src = blockIdx.x < (unsigned int)nb_s;
  if (threadIdx.x == 0) s_coef = src ? scal_s[1] : scal_t[1];
  __syncthreads();
  if (src) proto_bwd_block<K, VEC>(s, sC, C, Segment{0u, (unsigned int)nb_s}, grad_s, &s_coef, dfeat_s);
  else proto_bwd_block<K, VEC>(t, sC, C, Segment{(unsigned int)nb_s, (unsigned int)nb_t}, grad_t, &s_coef, dfeat_t);
}

// ---------------------------------------------------------------------------
// auxiliary backward: d loss / d soft mask [N,K] and d loss / d pixel_sel_loc [N]  (utils/loss.py:516-517, :558-565 take
// both as tensors; no reference caller differentiates them, so this is a pass of its own that recomputes the cosines
// instead of widening the stash of the hot path)
//   dmask_ik = g coef sel_i dl_i/dM_ik          dsel_i = g coef (l_i - L)        coef = scal[1], L = scal[0]
// ---------------------------------------------------------------------------
template <int K, int VEC>
__global__ void __launch_bounds__(kThreads) proto_aux_bwd_kernel(const ProtoArgs a, const float* scal, const float* grad_out,
                                                                 float* dmask, float* dsel) {
  extern __shared__ __align__(16) float sC[];
  const int C = (int)a.channels;
  load_centres_smem<K>(sC, a.cstate, C);
  __syncthreads();
  int64_t pix, off;
  if (!locate<VEC>(a, pix, off)) return;
  float nrm[VEC], dot[K][VEC];
  channel_pass<K, VEC>(a.feat + off, a.sc, C, sC, nrm, dot, l2_policy(false));
  const float gc = grad_out[0] * scal[1], loss = scal[0];
#pragma unroll
  for (int v = 0; v < VEC; ++v) {
    const float n = a.mc.normalize ? fmaxf(sqrtf(nrm[v]), 1e-12f) : 1.0f;
    const float inv_n = 1.0f / n;
    const float selv = a.sel != nullptr ? a.sel[pix + v] : 1.0f;
    float cosv[K], M[K], dM[K];
#pragma unroll
    for (int k = 0; k < K; ++k) {
      cosv[k] = dot[k][v] * inv_n;
      if (a.labels != nullptr) M[k] = (a.labels[pix + v] == (long long)k) ? 1.0f : 0.0f;
      else M[k] = a.soft_mask[(pix + v) * K + k];
    }
    const float row = margin_row_aux<K>(cosv, M, a.mc, dM);
    if (dsel != nullptr) dsel[pix + v] = gc * (row - loss);
    if (dmask != nullptr) {
#pragma unroll
      for (int k = 0; k < K; ++k) dmask[(pix + v) * K + k] = gc * selv * dM[k];
    }
  }
}

// ---------------------------------------------------------------------------
// pseudo labels: argmax_k cos and (top1 - top2 > th)
// ---------------------------------------------------------------------------
template <int K, int VEC>
__global__ void __launch_bounds__(kThreads) pseudo_label_kernel(const ProtoArgs a) {
  extern __shared__ __align__(16) float sC[];
  const int C = (int)a.channels;
  load_centres_smem<K>(sC, a.cstate, C);
  __syncthreads();
  int64_t pix, off;
  if (!locate<VEC>(a, pix, off)) return;
  float nrm[VEC], dot[K][VEC];
  channel_pass<K, VEC>(a.feat + off, a.sc, C, sC, nrm, dot, l2_policy(a.keep_l2 != 0));
  long long lab[VEC];
  float selv[VEC];
#pragma unroll
  for (int v = 0; v < VEC; ++v) {
    float n = fmaxf(sqrtf(nrm[v]), 1e-12f);                      // utils_.py:615
    float t1 = -INFINITY, t2 = -INFINITY;
    int best = 0;
#pragma unroll
    for (int k = 0; k < K; ++k) {
      float cs = dot[k][v] / n;
      if (cs > t1) { t2 = t1; t1 = cs; best = k; }               // strict >: first index wins ties (:621)
      else if (cs > t2) { t2 = cs; }
    }
    lab[v] = best;
    selv[v] = (t1 - t2 > a.sel_threshold) ? 1.0f : 0.0f;         // :608-609
  }
  if constexpr (VEC == 4) {
    longlong2* lp = reinterpret_cast<longlong2*>(a.out_label + pix);
    lp[0] = make_longlong2(lab[0], lab[1]);
    lp[1] = make_longlong2(lab[2], lab[3]);
  } else {
    a.out_label[pix] = lab[0];
  }
  Vec<VEC>::store_keep(a.out_sel + pix, selv);
}

// Unit centres + norms: cstate[k*C+c] = c_k[c] / max(||c_k||, 1e-12), cstate[K*C+k] = max(||c_k||, 1e-12).
__global__ void __launch_bounds__(kThreads) prep_centres_kernel(const float* centres, int C, int K, int normalize,
                                                                float* cstate) {
  pdl_trigger();
  pdl_wait();
  __shared__ float red[kThreads / 32];
  __shared__ float s_norm;
  const int k = blockIdx.x;
  const float* row = centres + (int64_t)k * C;
  float ss = 0.f;
  for (int c = threadIdx.x; c < C; c += kThreads) ss = fmaf(row[c], row[c], ss);
  ss = warp_sum(ss);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = ss;
  __syncthreads();
  if (threadIdx.x == 0) {
    float t = 0.f;
    for (int w = 0; w < kThreads / 32; ++w) t += red[w];
    s_norm = normalize ? fmaxf(sqrtf(t), 1e-12f) : 1.0f;
    cstate[(int64_t)K * C + k] = s_norm;
  }
  __syncthreads();
  const float n = s_norm;
  for (int c = threadIdx.x; c < C; c += kThreads) cstate[(int64_t)k * C + c] = row[c] / n;
}

// dcentre_k = gamma * (G_k - chat_k (chat_k . G_k)) / nu_k   (A.1), G from the class-sum kernel (fp64 [K, C+1]).
__global__ void __launch_bounds__(kThreads) centre_grad_kernel(const double* sums, const float* cstate, const float* scal,
                                                               const float* grad_out, int C, int K, int normalize,
                                                               float* dcentres) {
  __shared__ double red[kThreads / 32];
  __shared__ double s_dot;
  const int k = blockIdx.x;
  const double* g = sums + (int64_t)k * (C + 1);
  const float* ch = cstate + (int64_t)k * C;
  double d = 0.0;
  for (int c = threadIdx.x; c < C; c += kThreads) d += g[c] * (double)ch[c];
  d = warp_sum(d);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = d;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
    for (int w = 0; w < kThreads / 32; ++w) t += red[w];
    s_dot = t;
  }
  __syncthreads();
  const double gamma = (double)grad_out[0] * (double)scal[1];
  const double nu = (double)cstate[(int64_t)K * C + k];
  for (int c = threadIdx.x; c < C; c += kThreads) {
    double v = normalize ? (g[c] - (double)ch[c] * s_dot) / nu : g[c];
    dcentres[(int64_t)k * C + c] = (float)(gamma * v);
  }
}

// ------------------------------ host side ----------------------------------
struct Plan {
  int vec;
  int64_t n_total;
  int n_blocks;
  size_t smem;
};

bool validate_map(const slcl_map_t* m) {
  return m && m->batch > 0 && m->channels > 0 && m->pixels > 0 && m->stride_c >= 0 && m->stride_p >= 0;
}

Plan make_plan(const slcl_map_t* m, int K, std::initializer_list<const void*> ptrs16) {
  Plan p;
  p.n_total = m->batch * m->pixels;
  bool vec4 = (m->stride_p == 1) && (m->pixels % 4 == 0) && (m->stride_c % 4 == 0) && (m->stride_b % 4 == 0);
  for (const void* q : ptrs16) vec4 = vec4 && (q == nullptr || aligned16(q));
  p.vec = vec4 ? 4 : 1;
  p.n_blocks = (int)ceil_div<int64_t>(p.n_total / p.vec, kThreads);
  p.smem = (size_t)m->channels * (K <= 4 ? 4 : 8) * sizeof(float);
  return p;
}

ProtoArgs base_args(const float* feat, const slcl_map_t* m, const float* cstate) {
  ProtoArgs a{};
  a.feat = feat;
  a.batch = m->batch; a.channels = m->channels; a.pixels = m->pixels;
  a.sb = m->stride_b; a.sc = m->stride_c; a.sp = m->stride_p;
  a.n_total = m->batch * m->pixels;
  a.cstate = cstate;
  { const char* e = getenv("SLCL_L2_KEEP"); const bool off = e && atoi(e) == 0;
    a.keep_l2 = (!off && (size_t)a.n_total * (size_t)a.channels * sizeof(float) <= kL2KeepBytes) ? 1 : 0; }
  return a;
}

MarginConst make_const(const slcl_proto_params_t* p) { return make_margin_const(p); }

template <typename Kern>
int ensure_smem(Kern kern, size_t smem) {
  if (smem > 200 * 1024) return SLCL_ERR_UNSUPPORTED;
  if (smem > 48 * 1024) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) { set_cuda_error(e, "cudaFuncSetAttribute"); return SLCL_ERR_CUDA; }
  }
  return SLCL_OK;
}

#define SLCL_DISPATCH_K(K_, VEC_, ...)                                           \
  switch (K_) {                                                                  \
    case 2: { constexpr int KK = 2; if (VEC_ == 4) { constexpr int VV = 4; __VA_ARGS__ } else { constexpr int VV = 1; __VA_ARGS__ } } break; \
    case 3: { constexpr int KK = 3; if (VEC_ == 4) { constexpr int VV = 4; __VA_ARGS__ } else { constexpr int VV = 1; __VA_ARGS__ } } break; \
    case 4: { constexpr int KK = 4; if (VEC_ == 4) { constexpr int VV = 4; __VA_ARGS__ } else { constexpr int VV = 1; __VA_ARGS__ } } break; \
    case 5: { constexpr int KK = 5; if (VEC_ == 4) { constexpr int VV = 4; __VA_ARGS__ } else { constexpr int VV = 1; __VA_ARGS__ } } break; \
    case 6: { constexpr int KK = 6; if (VEC_ == 4) { constexpr int VV = 4; __VA_ARGS__ } else { constexpr int VV = 1; __VA_ARGS__ } } break; \
    case 7: { constexpr int KK = 7; if (VEC_ == 4) { constexpr int VV = 4; __VA_ARGS__ } else { constexpr int VV = 1; __VA_ARGS__ } } break; \
    case 8: { constexpr int KK = 8; if (VEC_ == 4) { constexpr int VV = 4; __VA_ARGS__ } else { constexpr int VV = 1; __VA_ARGS__ } } break; \
    default: return SLCL_ERR_INVALID_ARGUMENT;                                   \
  }

}  // namespace

// launch helpers for the fused target tile kernel (class_sums.cu)
void launch_prep_centres(const float* centres, int C, int K, int normalize, float* cstate, cudaStream_t stream) {
  launch_pdl(prep_centres_kernel, dim3(K), dim3(kThreads), 0, stream, centres, C, K, normalize, cstate);
}
void launch_proto_finalize(const void* partial, int n_blocks, int64_t n_total, int has_sel, float* scal,
                           const slcl_peer_t* peer, cudaStream_t stream) {
  launch_pdl(proto_finalize_kernel, dim3(1), dim3(kThreads), 0, stream, reinterpret_cast<const double2*>(partial), n_blocks,
             n_total, has_sel, scal, peer_ctx(peer), 0);
}
}  // namespace slcl

using namespace slcl;

extern "C" size_t slcl_proto_workspace_bytes(int64_t n_pixels) {
  if (n_pixels <= 0) return 0;
  return (size_t)ceil_div<int64_t>(n_pixels, kThreads) * sizeof(double2) + 256;
}

extern "C" int slcl_proto_fwd_peer(const float* feat, const slcl_map_t* map, const int64_t* labels, const float* soft_mask,
                                   const float* sel, const float* centres, const slcl_proto_params_t* params, float* stash,
                                   float* cstate, float* scal, const slcl_peer_t* peer, int split_phase, void* workspace,
                                   size_t workspace_bytes, slcl_stream_t stream_) {
  if (!feat || !validate_map(map) || !centres || !params || !stash || !cstate || !scal || !workspace)
    return SLCL_ERR_INVALID_ARGUMENT;
  if (peer != nullptr && !peer_valid(peer)) return SLCL_ERR_INVALID_ARGUMENT;
  if ((labels == nullptr) == (soft_mask == nullptr)) return SLCL_ERR_INVALID_ARGUMENT;   // exactly one (:502-505)
  const int K = params->n_class;
  if (K < 2 || K > kMaxK || !(params->temperature > 0.f) || !(params->base_temperature > 0.f))
    return SLCL_ERR_INVALID_ARGUMENT;
  cudaStream_t stream = (cudaStream_t)stream_;
  Plan plan = make_plan(map, K, {feat, labels, sel, stash, soft_mask});
  if (workspace_bytes < slcl_proto_workspace_bytes(plan.n_total)) return SLCL_ERR_WORKSPACE;
  if (!aligned16(workspace)) return SLCL_ERR_INVALID_ARGUMENT;

  ProtoArgs a = base_args(feat, map, cstate);
  a.labels = labels; a.soft_mask = soft_mask; a.sel = sel; a.stash = stash;
  a.partial = reinterpret_cast<double2*>(workspace);
  a.mc = make_const(params);
  a.reverse = a.keep_l2;

  launch_pdl(prep_centres_kernel, dim3(K), dim3(kThreads), 0, stream, centres, (int)map->channels, K, params->normalize, cstate);
  SLCL_DISPATCH_K(K, plan.vec, {
    int st = ensure_smem(proto_fwd_kernel<KK, VV>, plan.smem);
    if (st != SLCL_OK) return st;
    launch_pdl(proto_fwd_kernel<KK, VV>, dim3(plan.n_blocks), dim3(kThreads), plan.smem, stream, a);
  })
  launch_pdl(proto_finalize_kernel, dim3(1), dim3(kThreads), 0, stream, (const double2*)a.partial, plan.n_blocks, plan.n_total, (int)(sel != nullptr), scal, peer_ctx(peer), split_phase);
  return check_launch("slcl_proto_fwd");
}

extern "C" int slcl_proto_fwd(const float* feat, const slcl_map_t* map, const int64_t* labels, const float* soft_mask,
                              const float* sel, const float* centres, const slcl_proto_params_t* params, float* stash,
                              float* cstate, float* scal, void* workspace, size_t workspace_bytes,
                              slcl_stream_t stream_) {
  return slcl_proto_fwd_peer(feat, map, labels, soft_mask, sel, centres, params, stash, cstate, scal, nullptr, 0, workspace,
                             workspace_bytes, stream_);
}

extern "C" int slcl_proto_fwd_target_peer(const float* feat, const slcl_map_t* map, const float* centres,
                                          const slcl_proto_params_t* params, float sel_threshold, int64_t* label, float* sel,
                                          float* stash, float* cstate, float* scal, const slcl_peer_t* peer, void* workspace,
                                          size_t workspace_bytes, slcl_stream_t stream_) {
  if (!feat || !validate_map(map) || !centres || !params || !label || !sel || !stash || !cstate || !scal || !workspace)
    return SLCL_ERR_INVALID_ARGUMENT;
  if (peer != nullptr && !peer_valid(peer)) return SLCL_ERR_INVALID_ARGUMENT;
  const int K = params->n_class;
  if (K < 2 || K > kMaxK || !(params->temperature > 0.f) || !(params->base_temperature > 0.f) || !params->normalize)
    return SLCL_ERR_INVALID_ARGUMENT;
  cudaStream_t stream = (cudaStream_t)stream_;
  Plan plan = make_plan(map, K, {feat, label, sel, stash});
  if (workspace_bytes < slcl_proto_workspace_bytes(plan.n_total)) return SLCL_ERR_WORKSPACE;
  if (!aligned16(workspace)) return SLCL_ERR_INVALID_ARGUMENT;
  ProtoArgs a = base_args(feat, map, cstate);
  a.stash = stash;
  a.partial = reinterpret_cast<double2*>(workspace);
  a.mc = make_const(params);
  a.fused_target = 1; a.sel_threshold = sel_threshold; a.out_label = label; a.out_sel = sel;
  a.reverse = a.keep_l2;
  launch_pdl(prep_centres_kernel, dim3(K), dim3(kThreads), 0, stream, centres, (int)map->channels, K, 1, cstate);
  SLCL_DISPATCH_K(K, plan.vec, {
    int st = ensure_smem(proto_fwd_kernel<KK, VV>, plan.smem);
    if (st != SLCL_OK) return st;
    launch_pdl(proto_fwd_kernel<KK, VV>, dim3(plan.n_blocks), dim3(kThreads), plan.smem, stream, a);
  })
  launch_pdl(proto_finalize_kernel, dim3(1), dim3(kThreads), 0, stream, (const double2*)a.partial, plan.n_blocks, plan.n_total, 1, scal, peer_ctx(peer), 0);
  return check_launch("slcl_proto_fwd_target");
}

extern "C" int slcl_proto_fwd_target(const float* feat, const slcl_map_t* map, const float* centres,
                                     const slcl_proto_params_t* params, float sel_threshold, int64_t* label, float* sel,
                                     float* stash, float* cstate, float* scal, void* workspace, size_t workspace_bytes,
                                     slcl_stream_t stream_) {
  return slcl_proto_fwd_target_peer(feat, map, centres, params, sel_threshold, label, sel, stash, cstate, scal, nullptr,
                                    workspace, workspace_bytes, stream_);
}

extern "C" int slcl_proto_rescale(float* scal, int has_sel, slcl_stream_t stream_) {
  if (!scal) return SLCL_ERR_INVALID_ARGUMENT;
  launch_pdl(proto_rescale_kernel, dim3(1), dim3(32), 0, (cudaStream_t)stream_, scal, has_sel);
  return check_launch("slcl_proto_rescale");
}

extern "C" size_t slcl_peer_mailbox_bytes(int world, int64_t capacity_words) {
  if (world < 1 || world > kMaxPeers || capacity_words < kPeerMinCapacity) return 0;
  return (size_t)(kPeerHeaderWords + 2 * (size_t)world * (size_t)capacity_words) * sizeof(unsigned long long);
}

extern "C" int slcl_proto_rescale_peer(float* scal, int has_sel, const slcl_peer_t* peer, slcl_stream_t stream_) {
  if (!scal || !peer_valid(peer)) return SLCL_ERR_INVALID_ARGUMENT;
  launch_pdl(proto_rescale_peer_kernel, dim3(1), dim3(64), 0, (cudaStream_t)stream_, scal, has_sel, peer_ctx(peer));
  return check_launch("slcl_proto_rescale_peer");
}

extern "C" int slcl_peer_allreduce_f64(double* buf, int64_t n, const slcl_peer_t* peer, slcl_stream_t stream_) {
  if (!buf || n < 1 || !peer_valid(peer) || 2 * n > peer->capacity_words) return SLCL_ERR_INVALID_ARGUMENT;
  peer_allreduce_f64_kernel<<<(unsigned)ceil_div<int64_t>(n, 8), 256, 0, (cudaStream_t)stream_>>>(buf, (long long)n,
                                                                                                peer_ctx(peer));
  return check_launch("slcl_peer_allreduce_f64");
}

extern "C" int slcl_proto_bwd_peer(const float* feat, const slcl_map_t* map, const float* stash, const float* cstate,
                                   float* scal, const float* grad_out, const slcl_proto_params_t* params, float* dfeat,
                                   const slcl_peer_t* peer, int has_sel, slcl_stream_t stream_) {
  if (!feat || !validate_map(map) || !stash || !cstate || !scal || !grad_out || !params || !dfeat)
    return SLCL_ERR_INVALID_ARGUMENT;
  if (peer != nullptr && !peer_valid(peer)) return SLCL_ERR_INVALID_ARGUMENT;
  const int K = params->n_class;
  if (K < 2 || K > kMaxK) return SLCL_ERR_INVALID_ARGUMENT;
  cudaStream_t stream = (cudaStream_t)stream_;
  Plan plan = make_plan(map, K, {feat, stash, dfeat});
  ProtoArgs a = base_args(feat, map, cstate);
  a.stash = const_cast<float*>(stash);
  a.mc = make_const(params);
  SLCL_DISPATCH_K(K, plan.vec, {
    int st = ensure_smem(proto_bwd_kernel<KK, VV>, plan.smem);
    if (st != SLCL_OK) return st;
    launch_pdl(proto_bwd_kernel<KK, VV>, dim3(plan.n_blocks), dim3(kThreads), plan.smem, stream, a, const_cast<float*>(scal),
               grad_out, dfeat, peer_ctx(peer), has_sel);
  })
  return check_launch("slcl_proto_bwd");
}

extern "C" int slcl_proto_bwd_aux(const float* feat, const slcl_map_t* map, const int64_t* labels, const float* soft_mask,
                                  const float* sel, const float* cstate, const float* scal, const float* grad_out,
                                  const slcl_proto_params_t* params, float* dmask, float* dsel, slcl_stream_t stream_) {
  if (!feat || !validate_map(map) || !cstate || !scal || !grad_out || !params || (!dmask && !dsel)) return SLCL_ERR_INVALID_ARGUMENT;
  if ((labels == nullptr) == (soft_mask == nullptr)) return SLCL_ERR_INVALID_ARGUMENT;
  if (dmask && !soft_mask) return SLCL_ERR_INVALID_ARGUMENT;          // the one-hot mask of `labels` is not an input
  if (dsel && !sel) return SLCL_ERR_INVALID_ARGUMENT;
  const int K = params->n_class;
  if (K < 2 || K > kMaxK) return SLCL_ERR_INVALID_ARGUMENT;
  cudaStream_t stream = (cudaStream_t)stream_;
  Plan plan = make_plan(map, K, {feat});
  ProtoArgs a = base_args(feat, map, cstate);
  a.labels = labels; a.soft_mask = soft_mask; a.sel = sel;
  a.mc = make_const(params);
  SLCL_DISPATCH_K(K, plan.vec, {
    int st = ensure_smem(proto_aux_bwd_kernel<KK, VV>, plan.smem);
    if (st != SLCL_OK) return st;
    proto_aux_bwd_kernel<KK, VV><<<plan.n_blocks, kThreads, plan.smem, stream>>>(a, scal, grad_out, dmask, dsel);
  })
  return check_launch("slcl_proto_bwd_aux");
}

extern "C" int slcl_proto_bwd(const float* feat, const slcl_map_t* map, const float* stash, const float* cstate,
                              const float* scal, const float* grad_out, const slcl_proto_params_t* params,
                              float* dfeat, slcl_stream_t stream_) {
  return slcl_proto_bwd_peer(feat, map, stash, cstate, const_cast<float*>(scal), grad_out, params, dfeat, nullptr, 0, stream_);
}

extern "C" int slcl_pseudo_label(const float* feat, const slcl_map_t* map, const float* centres, int n_class,
                                 float threshold, int64_t* label, float* sel, void* workspace, size_t workspace_bytes,
                                 slcl_stream_t stream_) {
  if (!feat || !validate_map(map) || !centres || !label || !sel || !workspace) return SLCL_ERR_INVALID_ARGUMENT;
  const int K = n_class;
  if (K < 2 || K > kMaxK) return SLCL_ERR_INVALID_ARGUMENT;
  // workspace holds the unit centres [K*C + K]
  if (workspace_bytes < ((size_t)K * map->channels + K) * sizeof(float)) return SLCL_ERR_WORKSPACE;
  cudaStream_t stream = (cudaStream_t)stream_;
  float* cstate = reinterpret_cast<float*>(workspace);
  Plan plan = make_plan(map, K, {feat, label, sel});
  ProtoArgs a = base_args(feat, map, cstate);
  a.out_label = label; a.out_sel = sel; a.sel_threshold = threshold;
  launch_pdl(prep_centres_kernel, dim3(K), dim3(kThreads), 0, stream, centres, (int)map->channels, K, 1, cstate);
  SLCL_DISPATCH_K(K, plan.vec, {
    int st = ensure_smem(pseudo_label_kernel<KK, VV>, plan.smem);
    if (st != SLCL_OK) return st;
    pseudo_label_kernel<KK, VV><<<plan.n_blocks, kThreads, plan.smem, stream>>>(a);
  })
  return check_launch("slcl_pseudo_label");
}

// Weighted sums G_k = sum_i a_ik x_i come from the class-sum kernel (class_sums.cu).
namespace slcl {
int class_sums_planar_weights(const float* feat, const slcl_map_t* map, const float* weights, int n_cols,
                              double* sums, void* workspace, size_t workspace_bytes, cudaStream_t stream);
size_t class_sums_ws_bytes(int64_t batch, int64_t channels, int64_t pixels, int n_cols);
}

extern "C" size_t slcl_proto_bwd_centres_workspace_bytes(int64_t n_pixels, int64_t channels, int n_class) {
  if (n_pixels <= 0 || channels <= 0 || n_class <= 0) return 0;
  size_t sums = align_up((size_t)n_class * (channels + 1) * sizeof(double), 256);
  return sums + class_sums_ws_bytes(1, channels, n_pixels, n_class);
}

extern "C" int slcl_proto_bwd_centres(const float* feat, const slcl_map_t* map, const float* stash,
                                      const float* cstate, const float* scal, const float* grad_out,
                                      const slcl_proto_params_t* params, float* dcentres, void* workspace,
                                      size_t workspace_bytes, slcl_stream_t stream_) {
  if (!feat || !validate_map(map) || !stash || !cstate || !scal || !grad_out || !params || !dcentres || !workspace)
    return SLCL_ERR_INVALID_ARGUMENT;
  const int K = params->n_class;
  if (K < 2 || K > kMaxK) return SLCL_ERR_INVALID_ARGUMENT;
  const int64_t n = map->batch * map->pixels;
  if (workspace_bytes < slcl_proto_bwd_centres_workspace_bytes(n, map->channels, K)) return SLCL_ERR_WORKSPACE;
  cudaStream_t stream = (cudaStream_t)stream_;
  double* sums = reinterpret_cast<double*>(workspace);
  size_t off = align_up((size_t)K * (map->channels + 1) * sizeof(double), 256);
  int st = class_sums_planar_weights(feat, map, stash, K, sums, (char*)workspace + off, workspace_bytes - off, stream);
  if (st != SLCL_OK) return st;
  centre_grad_kernel<<<K, kThreads, 0, stream>>>(sums, cstate, scal, grad_out, (int)map->channels, K,
                                                  params->normalize, dcentres);
  return check_launch("slcl_proto_bwd_centres");
}

// ---------------------------------------------------------------------------
// The MPSCL loss section (trainer/Trainer_MPSCL.py:133-147) in one forward and one backward call:
//   centres = update_class_center_iter(F_s, labels_s, old, m)          class-sum sweep + reduce/exchange/EMA (class_sums.cu)
//   hard, mask = generate_pseudo_label(F_t, centres, th)                \  prep_centres_kernel, then mpscl_fwd_kernel over
//   loss_s = mpcl_loss_calc(F_s, labels_s, centres, mpcl_src)           |  both maps and mpscl_finalize_kernel (one
//   loss_t = mpcl_loss_calc(F_t, hard, centres, mpcl_trg, mask)        /   exchange of both loss pairs)
// Workspace: [class sums K x (C+1) fp64 | source block partials | target block partials | class-sum sweep workspace].
// ---------------------------------------------------------------------------
namespace slcl {
namespace {

struct MpsclWs {
  double* sums;
  double2* part_s;
  double2* part_t;
  void* cs;
  size_t cs_bytes;
};

bool dense_nchw(const slcl_map_t* m) {
  return validate_map(m) && m->stride_p == 1 && m->stride_c == m->pixels && m->stride_b == m->channels * m->pixels;
}

size_t mpscl_cs_bytes(const slcl_map_t* s, int K) { return class_sums_ws_bytes(s->batch, s->channels, s->pixels, K); }

size_t mpscl_ws_layout(const slcl_map_t* s, const slcl_map_t* t, int K, void* base, MpsclWs* ws) {
  const size_t sums = align_up((size_t)K * (s->channels + 1) * sizeof(double), 256);
  const size_t ps = align_up(slcl_proto_workspace_bytes(s->batch * s->pixels), 256);
  const size_t pt = align_up(slcl_proto_workspace_bytes(t->batch * t->pixels), 256);
  const size_t cs = mpscl_cs_bytes(s, K);
  if (ws != nullptr) {
    char* b = reinterpret_cast<char*>(base);
    ws->sums = reinterpret_cast<double*>(b);
    ws->part_s = reinterpret_cast<double2*>(b + sums);
    ws->part_t = reinterpret_cast<double2*>(b + sums + ps);
    ws->cs = b + sums + ps + pt;
    ws->cs_bytes = cs;
  }
  return sums + ps + pt + cs;
}

// The checks every entry point makes before anything is launched.
int mpscl_check_maps(const float* feat_s, const slcl_map_t* map_s, const float* feat_t, const slcl_map_t* map_t,
                     const slcl_proto_params_t* ps, const slcl_proto_params_t* pt) {
  if (!feat_s || !feat_t || !ps || !pt || !dense_nchw(map_s) || !dense_nchw(map_t)) return SLCL_ERR_INVALID_ARGUMENT;
  if (map_s->channels != map_t->channels || map_s->pixels != map_t->pixels) return SLCL_ERR_INVALID_ARGUMENT;
  const int K = ps->n_class;
  if (K < 2 || K > kMaxK || pt->n_class != K) return SLCL_ERR_INVALID_ARGUMENT;
  return SLCL_OK;
}

int mpscl_check_params(const slcl_proto_params_t* p) {
  return (p->temperature > 0.f && p->base_temperature > 0.f && p->normalize) ? SLCL_OK : SLCL_ERR_INVALID_ARGUMENT;
}

// Prototype forward of both maps (mpscl_fwd_kernel; one launch per map when their load widths differ) and the finaliser.
int mpscl_proto_fwd(const float* feat_s, const slcl_map_t* map_s, const int64_t* labels_s, const float* feat_t,
                    const slcl_map_t* map_t, const float* centres, const slcl_proto_params_t* ps,
                    const slcl_proto_params_t* pt, float sel_threshold, float* cstate, float* stash_s, float* stash_t,
                    int64_t* label_t, float* sel_t, float* scal_s, float* scal_t, float* pairs, const slcl_peer_t* peer,
                    const MpsclWs& ws, cudaStream_t stream) {
  const int K = ps->n_class;
  const int C = (int)map_s->channels;
  // the plans, walk directions and L2 policies of the single-map calls (slcl_proto_fwd, slcl_proto_fwd_target)
  const Plan plan_s = make_plan(map_s, K, {feat_s, labels_s, nullptr, stash_s, nullptr});
  const Plan plan_t = make_plan(map_t, K, {feat_t, label_t, sel_t, stash_t});
  ProtoArgs s = base_args(feat_s, map_s, cstate);
  s.labels = labels_s; s.stash = stash_s; s.partial = ws.part_s; s.mc = make_const(ps);
  s.reverse = s.keep_l2;
  ProtoArgs t = base_args(feat_t, map_t, cstate);
  t.stash = stash_t; t.partial = ws.part_t; t.mc = make_const(pt);
  t.fused_target = 1; t.sel_threshold = sel_threshold; t.out_label = label_t; t.out_sel = sel_t;
  // Both maps together larger than L2 (the cfg4 8-GPU shard: 2 x 98 MiB): only the source map, which the backward reads
  // first, is loaded with evict_last -- measured faster than keeping both (DESIGN §3); building with
  // -DSLCL_MPSCL_L2_BOTH=1 keeps the single-map policy for both maps instead.
  const size_t bytes_s = (size_t)s.n_total * C * sizeof(float), bytes_t = (size_t)t.n_total * C * sizeof(float);
  if (!SLCL_MPSCL_L2_BOTH && s.keep_l2 && t.keep_l2 && bytes_s + bytes_t > kL2KeepBytes) t.keep_l2 = 0;
  t.reverse = 0;             // the target segment follows the source segment's last block (the start of F_s)
  launch_pdl(prep_centres_kernel, dim3(K), dim3(kThreads), 0, stream, centres, C, K, 1, cstate);
  SLCL_DISPATCH_K(K, plan_s.vec, {
    int st = ensure_smem(mpscl_fwd_kernel<KK, VV>, plan_s.smem);
    if (st != SLCL_OK) return st;
    if (plan_t.vec == VV) {
      launch_pdl(mpscl_fwd_kernel<KK, VV>, dim3(plan_s.n_blocks + plan_t.n_blocks), dim3(kThreads), plan_s.smem, stream, s, t,
                 plan_s.n_blocks, plan_t.n_blocks);
    } else {
      launch_pdl(mpscl_fwd_kernel<KK, VV>, dim3(plan_s.n_blocks), dim3(kThreads), plan_s.smem, stream, s, t, plan_s.n_blocks, 0);
      constexpr int VT = VV == 4 ? 1 : 4;
      st = ensure_smem(mpscl_fwd_kernel<KK, VT>, plan_t.smem);
      if (st != SLCL_OK) return st;
      launch_pdl(mpscl_fwd_kernel<KK, VT>, dim3(plan_t.n_blocks), dim3(kThreads), plan_t.smem, stream, s, t, 0, plan_t.n_blocks);
    }
  })
  launch_pdl(mpscl_finalize_kernel, dim3(1), dim3(kThreads), 0, stream, (const double2*)ws.part_s, plan_s.n_blocks,
             plan_s.n_total, (const double2*)ws.part_t, plan_t.n_blocks, scal_s, scal_t, pairs, peer_ctx(peer));
  return SLCL_OK;
}

}  // namespace
}  // namespace slcl

extern "C" size_t slcl_mpscl_step_workspace_bytes(const slcl_map_t* map_s, const slcl_map_t* map_t, int n_class) {
  if (!validate_map(map_s) || !validate_map(map_t) || n_class < 2 || n_class > kMaxK) return 0;
  return mpscl_ws_layout(map_s, map_t, n_class, nullptr, nullptr);
}

extern "C" int slcl_mpscl_step_fwd(const float* feat_s, const slcl_map_t* map_s, const int64_t* labels_s, const float* feat_t,
                                   const slcl_map_t* map_t, const float* old_centres, float momentum,
                                   const slcl_proto_params_t* params_s, const slcl_proto_params_t* params_t,
                                   float sel_threshold, float* centres, float* cstate, float* stash_s, float* stash_t,
                                   int64_t* label_t, float* sel_t, float* scal_s, float* scal_t, const slcl_peer_t* peer,
                                   void* workspace, size_t workspace_bytes, slcl_stream_t stream_) {
  int st = mpscl_check_maps(feat_s, map_s, feat_t, map_t, params_s, params_t);
  if (st != SLCL_OK) return st;
  if (mpscl_check_params(params_s) != SLCL_OK || mpscl_check_params(params_t) != SLCL_OK) return SLCL_ERR_INVALID_ARGUMENT;
  if (!labels_s || !old_centres || !centres || !cstate || !stash_s || !stash_t || !label_t || !sel_t || !scal_s || !scal_t ||
      !workspace)
    return SLCL_ERR_INVALID_ARGUMENT;
  const int K = params_s->n_class;
  if (peer != nullptr && (!peer_valid(peer) || 2 * (int64_t)K * (map_s->channels + 1) > peer->capacity_words))
    return SLCL_ERR_INVALID_ARGUMENT;
  MpsclWs ws;
  if (workspace_bytes < mpscl_ws_layout(map_s, map_t, K, workspace, &ws)) return SLCL_ERR_WORKSPACE;
  if (!aligned16(workspace)) return SLCL_ERR_INVALID_ARGUMENT;
  cudaStream_t stream = (cudaStream_t)stream_;
  // update_class_center_iter: the sweep and the reduce [+ exchange] + EMA kernels of slcl_class_centres_update, unchanged
  st = slcl_class_centres_update(feat_s, map_s->batch, map_s->channels, map_s->pixels, labels_s, K, old_centres, momentum,
                                 centres, ws.sums, peer, ws.cs, ws.cs_bytes, stream_);
  if (st != SLCL_OK) return st;
  st = mpscl_proto_fwd(feat_s, map_s, labels_s, feat_t, map_t, centres, params_s, params_t, sel_threshold, cstate, stash_s,
                       stash_t, label_t, sel_t, scal_s, scal_t, nullptr, peer, ws, stream);
  if (st != SLCL_OK) return st;
  return check_launch("slcl_mpscl_step_fwd");
}

extern "C" int slcl_mpscl_step_fwd_local(const float* feat_s, const slcl_map_t* map_s, const int64_t* labels_s,
                                         const float* feat_t, const slcl_map_t* map_t, const float* centres,
                                         const slcl_proto_params_t* params_s, const slcl_proto_params_t* params_t,
                                         float sel_threshold, float* cstate, float* stash_s, float* stash_t, int64_t* label_t,
                                         float* sel_t, float* pairs, void* workspace, size_t workspace_bytes,
                                         slcl_stream_t stream_) {
  int st = mpscl_check_maps(feat_s, map_s, feat_t, map_t, params_s, params_t);
  if (st != SLCL_OK) return st;
  if (mpscl_check_params(params_s) != SLCL_OK || mpscl_check_params(params_t) != SLCL_OK) return SLCL_ERR_INVALID_ARGUMENT;
  if (!labels_s || !centres || !cstate || !stash_s || !stash_t || !label_t || !sel_t || !pairs || !workspace)
    return SLCL_ERR_INVALID_ARGUMENT;
  MpsclWs ws;
  if (workspace_bytes < mpscl_ws_layout(map_s, map_t, params_s->n_class, workspace, &ws)) return SLCL_ERR_WORKSPACE;
  if (!aligned16(workspace)) return SLCL_ERR_INVALID_ARGUMENT;
  st = mpscl_proto_fwd(feat_s, map_s, labels_s, feat_t, map_t, centres, params_s, params_t, sel_threshold, cstate, stash_s,
                       stash_t, label_t, sel_t, nullptr, nullptr, pairs, nullptr, ws, (cudaStream_t)stream_);
  if (st != SLCL_OK) return st;
  return check_launch("slcl_mpscl_step_fwd_local");
}

extern "C" int slcl_mpscl_step_finish(const float* pairs, float* scal_s, float* scal_t, slcl_stream_t stream_) {
  if (!pairs || !scal_s || !scal_t) return SLCL_ERR_INVALID_ARGUMENT;
  launch_pdl(mpscl_finish_kernel, dim3(1), dim3(32), 0, (cudaStream_t)stream_, pairs, scal_s, scal_t);
  return check_launch("slcl_mpscl_step_finish");
}

extern "C" int slcl_mpscl_step_bwd(const float* feat_s, const slcl_map_t* map_s, const float* feat_t, const slcl_map_t* map_t,
                                   const float* stash_s, const float* stash_t, const float* cstate, const float* scal_s,
                                   const float* scal_t, const float* grad_s, const float* grad_t,
                                   const slcl_proto_params_t* params_s, const slcl_proto_params_t* params_t, float* dfeat_s,
                                   float* dfeat_t, slcl_stream_t stream_) {
  int st = mpscl_check_maps(feat_s, map_s, feat_t, map_t, params_s, params_t);
  if (st != SLCL_OK) return st;
  if (!cstate || (!grad_s && !grad_t)) return SLCL_ERR_INVALID_ARGUMENT;
  if (grad_s && (!stash_s || !scal_s || !dfeat_s)) return SLCL_ERR_INVALID_ARGUMENT;
  if (grad_t && (!stash_t || !scal_t || !dfeat_t)) return SLCL_ERR_INVALID_ARGUMENT;
  const int K = params_s->n_class;
  cudaStream_t stream = (cudaStream_t)stream_;
  // the plans of slcl_proto_bwd for each map; a map without an upstream gradient gets no blocks
  const Plan plan_s = make_plan(map_s, K, {feat_s, stash_s, dfeat_s});
  const Plan plan_t = make_plan(map_t, K, {feat_t, stash_t, dfeat_t});
  const int nb_s = grad_s ? plan_s.n_blocks : 0, nb_t = grad_t ? plan_t.n_blocks : 0;
  ProtoArgs s = base_args(feat_s, map_s, cstate);
  s.stash = const_cast<float*>(stash_s);
  ProtoArgs t = base_args(feat_t, map_t, cstate);
  t.stash = const_cast<float*>(stash_t);
  s.reverse = t.reverse = 0;
  SLCL_DISPATCH_K(K, (nb_s ? plan_s.vec : plan_t.vec), {
    st = ensure_smem(mpscl_bwd_kernel<KK, VV>, plan_s.smem);
    if (st != SLCL_OK) return st;
    if (nb_s == 0 || nb_t == 0 || plan_t.vec == plan_s.vec) {
      launch_pdl(mpscl_bwd_kernel<KK, VV>, dim3(nb_s + nb_t), dim3(kThreads), plan_s.smem, stream, s, t, nb_s, nb_t, scal_s,
                 scal_t, grad_s, grad_t, dfeat_s, dfeat_t);
    } else {
      launch_pdl(mpscl_bwd_kernel<KK, VV>, dim3(nb_s), dim3(kThreads), plan_s.smem, stream, s, t, nb_s, 0, scal_s, scal_t,
                 grad_s, grad_t, dfeat_s, dfeat_t);
      constexpr int VT = VV == 4 ? 1 : 4;
      st = ensure_smem(mpscl_bwd_kernel<KK, VT>, plan_t.smem);
      if (st != SLCL_OK) return st;
      launch_pdl(mpscl_bwd_kernel<KK, VT>, dim3(nb_t), dim3(kThreads), plan_t.smem, stream, s, t, 0, nb_t, scal_s, scal_t,
                 grad_s, grad_t, dfeat_s, dfeat_t);
    }
  })
  return check_launch("slcl_mpscl_step_bwd");
}
