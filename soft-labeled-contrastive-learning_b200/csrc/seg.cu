// seg.cu -- segmentation losses on the logits that sit right before / after the contrastive path
// (SURVEY.md section 8(f)-2): cross entropy + Jaccard + Dice in ONE pass over the logits, their fused
// backward, and the weighted self-information map.
//
// Replaces (reference, file:line):
//   loss_calc        utils/loss.py:46-66    nn.CrossEntropyLoss (+ jaccard_loss when jaccard=True)
//   jaccard_loss     utils/loss.py:11-43    softmax, one-hot, per-class intersection / union over (B,H,W)
//   dice_loss        utils/loss.py:69-103   softmax, one-hot, per-(image,class) 2 p.g / (p.p + g.g + 1e-5)
//   prob_2_entropy   utils/utils_.py:627-631   -p log2(p + 1e-7) / log2(C)
// Callers: trainer/Trainer_MPSCL.py:125,171-172, trainer/Trainer_MCCL.py:252.
//
// Roofline: HBM.  forward 4K + 8 B/px (logits + label), backward 8K + 8 B/px; the reference makes
// ~25 passes over [B,K,H,W]-sized temporaries (softmax, eye-indexed one-hot, products, sums per loss).
//
// Data-parallel form (group=): all three losses of the ranks' concatenated batches need only sums, so each rank reduces
// its partials into ONE fp64 vector [2K + 4] = {inter_k, card_k, n_valid, sum ce, sum dice_bk, n_images}, the ranks add
// the vectors (in the finaliser over NVLink peer mailboxes, or NCCL between two launches), and every rank finishes the
// same losses from the same global vector.  The backward reads its global coefficients from that vector: no exchange.
#include "common.cuh"
#include "peer.cuh"

#include <math.h>

namespace slcl {
namespace {

constexpr int kThreads = 256;
constexpr int kWarps = kThreads / 32;
constexpr int KM = SLCL_MAX_CLASSES;
constexpr int kStats = 4;          // per (image, class): sum p*g, sum p*p, sum g, sum p
constexpr int kVecTail = 4;        // global vector after inter_k, card_k: n_valid, sum ce, sum dice_bk, n_images

__host__ __device__ constexpr int seg_vec_len(int K) { return 2 * K + kVecTail; }

template <int VEC>
__device__ __forceinline__ void ldv(const float* p, float (&v)[VEC]) {
  if constexpr (VEC == 4) { float4 t = ld_stream4(p); v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w; }
  else v[0] = ld_stream1(p);
}
template <int VEC>
__device__ __forceinline__ void stv(float* p, const float (&v)[VEC]) {
  if constexpr (VEC == 4) st_stream4(p, make_float4(v[0], v[1], v[2], v[3]));
  else st_stream1(p, v[0]);
}

// softmax over K planar logits of VEC pixels: probabilities and log-probabilities
template <int K, int VEC>
__device__ __forceinline__ void softmax_k(const float* img, int64_t hw, int64_t p, float (&prob)[K][VEC], float (&logp)[K][VEC]) {
#pragma unroll
  for (int k = 0; k < K; ++k) ldv<VEC>(img + (int64_t)k * hw + p, logp[k]);
#pragma unroll
  for (int v = 0; v < VEC; ++v) {
    float m = logp[0][v];
#pragma unroll
    for (int k = 1; k < K; ++k) m = fmaxf(m, logp[k][v]);
    float s = 0.f;
#pragma unroll
    for (int k = 0; k < K; ++k) { prob[k][v] = expf(logp[k][v] - m); s += prob[k][v]; }
    const float inv = 1.0f / s;
    const float lse = m + logf(s);
#pragma unroll
    for (int k = 0; k < K; ++k) { prob[k][v] *= inv; logp[k][v] -= lse; }
  }
}

// grid = (blocks_per_image, B); one block = kThreads*VEC consecutive pixels of one image
template <int K, int VEC>
__global__ void __launch_bounds__(kThreads) seg_fwd_kernel(const float* logits, const int64_t* labels, int64_t hw,
                                                           float* partial /* [B][bpi][K*4 + 1] */) {
  __shared__ float red[kWarps][K * kStats + 1];
  const int b = blockIdx.y;
  const int64_t p = ((int64_t)blockIdx.x * kThreads + threadIdx.x) * VEC;
  float acc[K * kStats + 1];
#pragma unroll
  for (int i = 0; i < K * kStats + 1; ++i) acc[i] = 0.f;
  if (p < hw) {
    const float* img = logits + (int64_t)b * K * hw;
    float prob[K][VEC], logp[K][VEC];
    softmax_k<K, VEC>(img, hw, p, prob, logp);
#pragma unroll
    for (int v = 0; v < VEC; ++v) {
      const long long lab = labels[(int64_t)b * hw + p + v];
#pragma unroll
      for (int k = 0; k < K; ++k) {
        const float g = (lab == k) ? 1.f : 0.f;
        acc[k * kStats + 0] += prob[k][v] * g;
        acc[k * kStats + 1] += prob[k][v] * prob[k][v];
        acc[k * kStats + 2] += g;
        acc[k * kStats + 3] += prob[k][v];
        if (lab == k) acc[K * kStats] -= logp[k][v];                            // -log softmax(z)_label (CrossEntropyLoss)
      }
    }
  }
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int i = 0; i < K * kStats + 1; ++i) {
    const float r = warp_sum(acc[i]);
    if (lane == 0) red[warp][i] = r;
  }
  __syncthreads();
  if (threadIdx.x < K * kStats + 1) {
    float t = 0.f;
    for (int w = 0; w < kWarps; ++w) t += red[w][threadIdx.x];
    partial[((int64_t)b * gridDim.x + blockIdx.x) * (K * kStats + 1) + threadIdx.x] = t;
  }
}

// stats[b][k][4] (fp32) and losses[3] = {cross entropy, dice, jaccard}; one block, fixed summation order
__global__ void __launch_bounds__(kThreads) seg_finalize_kernel(const float* partial, int B, int bpi, int K, int64_t hw,
                                                                float* stats, float* losses) {
  __shared__ double s_ce[kThreads];
  const int per = K * kStats + 1;
  double ce = 0.0;
  for (int idx = threadIdx.x; idx < B * per; idx += kThreads) {
    const int b = idx / per, i = idx % per;
    double t = 0.0;
    for (int j = 0; j < bpi; ++j) t += (double)partial[((int64_t)b * bpi + j) * per + i];
    if (i == K * kStats) ce += t;
    else stats[(int64_t)b * K * kStats + i] = (float)t;
  }
  s_ce[threadIdx.x] = ce;
  __syncthreads();
  if (threadIdx.x == 0) {
    double tot = 0.0;
    for (int i = 0; i < kThreads; ++i) tot += s_ce[i];
    // nn.CrossEntropyLoss (:63-64) averages over the pixels it does not ignore.  Labels outside [0, K) -- the
    // reference's ignore_index = -100 and anything else it would raise on -- have an all-zero one-hot row here: they add
    // nothing to any sum and are not counted (no host-visible error: that would need a synchronisation).
    double n_valid = 0.0;
    for (int i = 0; i < B * K; ++i) n_valid += (double)stats[(int64_t)i * kStats + 2];
    (void)hw;
    losses[0] = (float)(tot / n_valid);
    double dice = 0.0;
    for (int b = 0; b < B; ++b)
      for (int k = 0; k < K; ++k) {
        const float* s = stats + ((int64_t)b * K + k) * kStats;
        dice += 2.0 * (double)(s[0] / (s[1] + s[2] + 1e-5f));                          // :96-100
      }
    losses[1] = (float)(1.0 - dice / B / K);                                            // :102-103
    double jac = 0.0;
    for (int k = 0; k < K; ++k) {
      float inter = 0.f, card = 0.f;
      for (int b = 0; b < B; ++b) {
        const float* s = stats + ((int64_t)b * K + k) * kStats;
        inter += s[0]; card += s[3] + s[2];
      }
      jac += (double)(inter / (card - inter + 1e-7f));                                  // :39-42
    }
    losses[2] = (float)(1.0 - jac / K);
  }
}

// losses[3] from a global vector v[2K + 4] (seg_vec_len); one thread.  The peer finaliser and seg_finish_kernel (the
// NCCL route) both end here, so the two routes finish with the same arithmetic.
__device__ void seg_losses_from_vec(const double* v, int K, float* losses) {
  const double n_valid = v[2 * K], ce = v[2 * K + 1], dice = v[2 * K + 2], n_images = v[2 * K + 3];
  losses[0] = (float)(ce / n_valid);                                                    // CrossEntropyLoss, :63-64
  losses[1] = (float)(1.0 - dice / n_images / K);                                       // :102-103
  double jac = 0.0;
  for (int k = 0; k < K; ++k) jac += v[k] / (v[K + k] - v[k] + 1e-7);                   // :39-42 on global sums
  losses[2] = (float)(1.0 - jac / K);
}

// The finaliser of the data-parallel forward: stats[b][k][4] as seg_finalize_kernel writes them, and this rank's vector
// {inter_k, card_k, n_valid, sum ce, sum dice_bk, n_images} in fp64 -> vec.  PEER: the vector is then all-reduced over
// the ranks through the mailboxes (one warp per element, rank order: identical bits everywhere), vec holds the GLOBAL
// vector and losses[3] the global losses.  A peer that times out makes the whole vector and the losses NaN.
template <bool PEER>
__global__ void __launch_bounds__(kThreads) seg_finalize_vec_kernel(const float* partial, int B, int bpi, int K, float* stats,
                                                                    double* vec, float* losses, const PeerCtx pc) {
  __shared__ double s_ce[kThreads];
  __shared__ double s_vec[seg_vec_len(KM)];
  __shared__ int s_bad;
  unsigned int e = 0u;
  if constexpr (PEER) e = peer_epoch_begin(pc);
  const int per = K * kStats + 1, n = seg_vec_len(K);
  double ce = 0.0;
  for (int idx = threadIdx.x; idx < B * per; idx += kThreads) {
    const int b = idx / per, i = idx % per;
    double t = 0.0;
    for (int j = 0; j < bpi; ++j) t += (double)partial[((int64_t)b * bpi + j) * per + i];
    if (i == K * kStats) ce += t;
    else stats[(int64_t)b * K * kStats + i] = (float)t;
  }
  s_ce[threadIdx.x] = ce;
  if (threadIdx.x == 0) s_bad = 0;
  __syncthreads();
  if (threadIdx.x < K) {                      // per-class intersection and cardinality over this rank's images
    const int k = threadIdx.x;
    double inter = 0.0, card = 0.0;
    for (int b = 0; b < B; ++b) {
      const float* s = stats + ((int64_t)b * K + k) * kStats;
      inter += (double)s[0];
      card += (double)s[3] + (double)s[2];
    }
    s_vec[k] = inter;
    s_vec[K + k] = card;
  } else if (threadIdx.x == K) {              // pixels with a label inside [0, K): the cross entropy's denominator
    double n_valid = 0.0;
    for (int i = 0; i < B * K; ++i) n_valid += (double)stats[(int64_t)i * kStats + 2];
    s_vec[2 * K] = n_valid;
  } else if (threadIdx.x == K + 1) {
    double tot = 0.0;
    for (int i = 0; i < kThreads; ++i) tot += s_ce[i];
    s_vec[2 * K + 1] = tot;
  } else if (threadIdx.x == K + 2) {          // dice_bk exactly as the single-rank finaliser forms it, summed over images
    double dice = 0.0;
    for (int b = 0; b < B; ++b)
      for (int k = 0; k < K; ++k) {
        const float* s = stats + ((int64_t)b * K + k) * kStats;
        dice += 2.0 * (double)(s[0] / (s[1] + s[2] + 1e-5f));
      }
    s_vec[2 * K + 2] = dice;
    s_vec[2 * K + 3] = (double)B;
  }
  __syncthreads();
  if constexpr (PEER) {
    const int lane = threadIdx.x & 31;
    for (int i = threadIdx.x >> 5; i < n; i += kWarps) {
      const double t = peer_warp_allreduce(pc, e, i, s_vec[i]);
      if (lane == 0) {
        s_vec[i] = t;
        if (isnan(t)) s_bad = 1;
      }
    }
    __syncthreads();
    if (s_bad && threadIdx.x < n) s_vec[threadIdx.x] = __longlong_as_double(0x7FF8000000000000ll);
    __syncthreads();
  }
  if (threadIdx.x < n) vec[threadIdx.x] = s_vec[threadIdx.x];
  if constexpr (PEER) {
    if (threadIdx.x == 0) {
      seg_losses_from_vec(s_vec, K, losses);
      peer_epoch_end(pc, e, 1u);
    }
  }
}

// losses[3] from an all-reduced vector (the NCCL route's last launch)
__global__ void seg_finish_kernel(const double* vec, int K, float* losses) {
  if (threadIdx.x == 0) seg_losses_from_vec(vec, K, losses);
}

// dlogits for upstream gradients gout[3] = d/d{ce, dice, jaccard}.  GLOBAL: the loss is that of the ranks' concatenated
// batches; the CE pixel count, the image count of the Dice mean and Jaccard's per-class sums come from the global vector
// gvec (seg_vec_len), the per-image Dice stats from this rank's stats.  !GLOBAL is the single-rank kernel, unchanged.
template <int K, int VEC, bool GLOBAL>
__global__ void __launch_bounds__(kThreads) seg_bwd_kernel(const float* logits, const int64_t* labels, int64_t hw, int B,
                                                           const float* stats, const double* gvec, const float* gout,
                                                           float* dlogits) {
  __shared__ float s_dice_a[K], s_dice_b[K], s_jac_a[K], s_jac_b[K];
  __shared__ float s_red[kWarps];
  const int b = blockIdx.y;
  if constexpr (!GLOBAL) {   // pixels the cross entropy averages over = labels inside [0, K) = sum of the one-hot counts (exact in fp32 per entry)
    double cnt = 0.0;
    for (int i = threadIdx.x; i < B * K; i += kThreads) cnt += (double)stats[(int64_t)i * kStats + 2];
    cnt = warp_sum(cnt);
    if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = (float)cnt;
  }
  if (threadIdx.x < K) {
    const int k = threadIdx.x;
    const float* s = stats + ((int64_t)b * K + k) * kStats;
    const float D = s[1] + s[2] + 1e-5f;
    const float BK = GLOBAL ? (float)(gvec[2 * K + 3] * K) : (float)(B * K);
    // dice_bk = 2 num / D :  d/dp = 2 g / D - 4 num p / D^2 ;  loss = 1 - sum/(B K)
    s_dice_a[k] = -gout[1] * 2.0f / (D * BK);
    s_dice_b[k] = gout[1] * 4.0f * s[0] / (D * D * BK);
    float inter = 0.f, U;
    if constexpr (GLOBAL) {
      inter = (float)gvec[k];
      U = (float)(gvec[K + k] - gvec[k] + 1e-7);
    } else {
      float card = 0.f;
      for (int bb = 0; bb < B; ++bb) {
        const float* t = stats + ((int64_t)bb * K + k) * kStats;
        inter += t[0]; card += t[3] + t[2];
      }
      U = card - inter + 1e-7f;
    }
    // jac_k = I / U, U = card - I + eps : dI/dp = g, dU/dp = 1 - g  ->  d jac/dp = (g U - I (1 - g)) / U^2
    s_jac_a[k] = -gout[2] / ((float)K * U * U) * (U + inter);      // coefficient of g
    s_jac_b[k] = gout[2] * inter / ((float)K * U * U);              // constant term
  }
  __syncthreads();
  const int64_t p = ((int64_t)blockIdx.x * kThreads + threadIdx.x) * VEC;
  if (p >= hw) return;
  const float* img = logits + (int64_t)b * K * hw;
  float prob[K][VEC], logp[K][VEC];
  softmax_k<K, VEC>(img, hw, p, prob, logp);
  float n_valid = 0.f;
  if constexpr (GLOBAL) n_valid = (float)gvec[2 * K];
  else {
#pragma unroll
    for (int w = 0; w < kWarps; ++w) n_valid += s_red[w];
  }
  const float g_ce = gout[0] / n_valid;
  float out[K][VEC];
#pragma unroll
  for (int v = 0; v < VEC; ++v) {
    const long long lab = labels[(int64_t)b * hw + p + v];
    float dp[K];
    float dot = 0.f;
#pragma unroll
    for (int k = 0; k < K; ++k) {
      const float g = (lab == k) ? 1.f : 0.f;
      dp[k] = s_dice_a[k] * g + s_dice_b[k] * prob[k][v] + s_jac_a[k] * g + s_jac_b[k];
      dot = fmaf(dp[k], prob[k][v], dot);
    }
#pragma unroll
    for (int k = 0; k < K; ++k) {
      const float g = (lab == k) ? 1.f : 0.f;
      const float ce = (lab >= 0 && lab < K) ? g_ce * (prob[k][v] - g) : 0.f;      // ignored pixels carry no CE gradient
      out[k][v] = ce + prob[k][v] * (dp[k] - dot);                              // CE + softmax backward of the rest
    }
  }
#pragma unroll
  for (int k = 0; k < K; ++k) stv<VEC>(dlogits + ((int64_t)b * K + k) * hw + p, out[k]);
}

// prob_2_entropy (utils/utils_.py:627-631): e = -p log2(p + 1e-7) / log2(C); backward de/dp
__global__ void __launch_bounds__(kThreads) entropy_map_kernel(const float* prob, int64_t n, float inv_log2c, float* out,
                                                               const float* gout, float* dprob) {
  const int64_t i = (int64_t)blockIdx.x * kThreads + threadIdx.x;
  if (i >= n) return;
  const float p = prob[i];
  const float l2 = log2f(p + 1e-7f);
  if (out) out[i] = -p * l2 * inv_log2c;
  if (dprob) dprob[i] = -gout[i] * inv_log2c * (l2 + p / ((p + 1e-7f) * 0.6931471805599453f));
}

}  // namespace
}  // namespace slcl

using namespace slcl;

extern "C" size_t slcl_seg_workspace_bytes(int64_t batch, int64_t pixels, int n_class) {
  if (batch <= 0 || pixels <= 0 || n_class < 2 || n_class > KM) return 0;
  const int64_t bpi = ceil_div<int64_t>(pixels, kThreads);      // worst case (scalar path)
  return align_up((size_t)batch * bpi * (n_class * kStats + 1) * sizeof(float), 256);
}

#define SLCL_SEG_DISPATCH(K_, VEC4_, ...)                                                                                \
  switch (K_) {                                                                                                            \
    case 2: { constexpr int KK = 2; if (VEC4_) { constexpr int VV = 4; __VA_ARGS__ } else { constexpr int VV = 1; __VA_ARGS__ } } break; \
    case 3: { constexpr int KK = 3; if (VEC4_) { constexpr int VV = 4; __VA_ARGS__ } else { constexpr int VV = 1; __VA_ARGS__ } } break; \
    case 4: { constexpr int KK = 4; if (VEC4_) { constexpr int VV = 4; __VA_ARGS__ } else { constexpr int VV = 1; __VA_ARGS__ } } break; \
    case 5: { constexpr int KK = 5; if (VEC4_) { constexpr int VV = 4; __VA_ARGS__ } else { constexpr int VV = 1; __VA_ARGS__ } } break; \
    case 6: { constexpr int KK = 6; if (VEC4_) { constexpr int VV = 4; __VA_ARGS__ } else { constexpr int VV = 1; __VA_ARGS__ } } break; \
    case 7: { constexpr int KK = 7; if (VEC4_) { constexpr int VV = 4; __VA_ARGS__ } else { constexpr int VV = 1; __VA_ARGS__ } } break; \
    case 8: { constexpr int KK = 8; if (VEC4_) { constexpr int VV = 4; __VA_ARGS__ } else { constexpr int VV = 1; __VA_ARGS__ } } break; \
    default: return SLCL_ERR_INVALID_ARGUMENT;                                                                             \
  }

namespace {

// Argument checks shared by every forward entry (nothing is launched when they fail).
int seg_fwd_check(const float* logits, const int64_t* labels, int64_t batch, int n_class, int64_t pixels, const float* stats,
                  const void* workspace, size_t workspace_bytes) {
  if (!logits || !labels || batch <= 0 || pixels <= 0 || !stats || !workspace) return SLCL_ERR_INVALID_ARGUMENT;
  if (n_class < 2 || n_class > KM) return SLCL_ERR_INVALID_ARGUMENT;
  if (workspace_bytes < slcl_seg_workspace_bytes(batch, pixels, n_class) || !aligned16(workspace)) return SLCL_ERR_WORKSPACE;
  return SLCL_OK;
}

// The forward sweep into the per-block partials (workspace); returns blocks per image.
int seg_sweep(const float* logits, const int64_t* labels, int64_t batch, int n_class, int64_t pixels, float* partial,
              cudaStream_t stream) {
  const bool vec4 = (pixels % 4 == 0) && aligned16(logits);
  const int bpi = (int)ceil_div<int64_t>(pixels, (int64_t)kThreads * (vec4 ? 4 : 1));
  dim3 grid((unsigned)bpi, (unsigned)batch);
  SLCL_SEG_DISPATCH(n_class, vec4, { seg_fwd_kernel<KK, VV><<<grid, kThreads, 0, stream>>>(logits, labels, pixels, partial); })
  return bpi;
}

template <bool GLOBAL>
int seg_bwd_launch(const float* logits, const int64_t* labels, int64_t batch, int n_class, int64_t pixels, const float* stats,
                   const double* gvec, const float* grad_losses, float* dlogits, cudaStream_t stream) {
  const bool vec4 = (pixels % 4 == 0) && aligned16(logits) && aligned16(dlogits);
  const int bpi = (int)ceil_div<int64_t>(pixels, (int64_t)kThreads * (vec4 ? 4 : 1));
  dim3 grid((unsigned)bpi, (unsigned)batch);
  SLCL_SEG_DISPATCH(n_class, vec4, {
    seg_bwd_kernel<KK, VV, GLOBAL><<<grid, kThreads, 0, stream>>>(logits, labels, pixels, (int)batch, stats, gvec, grad_losses,
                                                                  dlogits);
  })
  return SLCL_OK;
}

}  // namespace

extern "C" int slcl_seg_fwd(const float* logits, const int64_t* labels, int64_t batch, int n_class, int64_t pixels,
                            float* stats, float* losses, void* workspace, size_t workspace_bytes, slcl_stream_t stream_) {
  if (!losses) return SLCL_ERR_INVALID_ARGUMENT;
  const int st = seg_fwd_check(logits, labels, batch, n_class, pixels, stats, workspace, workspace_bytes);
  if (st != SLCL_OK) return st;
  cudaStream_t stream = (cudaStream_t)stream_;
  float* partial = reinterpret_cast<float*>(workspace);
  const int bpi = seg_sweep(logits, labels, batch, n_class, pixels, partial, stream);
  seg_finalize_kernel<<<1, kThreads, 0, stream>>>(partial, (int)batch, bpi, n_class, pixels, stats, losses);
  return check_launch("slcl_seg_fwd");
}

extern "C" int slcl_seg_fwd_peer(const float* logits, const int64_t* labels, int64_t batch, int n_class, int64_t pixels,
                                 float* stats, double* vec, float* losses, const slcl_peer_t* peer, void* workspace,
                                 size_t workspace_bytes, slcl_stream_t stream_) {
  if (!vec || !losses || !peer_valid(peer)) return SLCL_ERR_INVALID_ARGUMENT;
  const int st = seg_fwd_check(logits, labels, batch, n_class, pixels, stats, workspace, workspace_bytes);
  if (st != SLCL_OK) return st;
  if (peer->capacity_words < 2 * (int64_t)seg_vec_len(n_class)) return SLCL_ERR_INVALID_ARGUMENT;
  cudaStream_t stream = (cudaStream_t)stream_;
  float* partial = reinterpret_cast<float*>(workspace);
  const int bpi = seg_sweep(logits, labels, batch, n_class, pixels, partial, stream);
  seg_finalize_vec_kernel<true><<<1, kThreads, 0, stream>>>(partial, (int)batch, bpi, n_class, stats, vec, losses,
                                                            peer_ctx(peer));
  return check_launch("slcl_seg_fwd_peer");
}

extern "C" int slcl_seg_fwd_local(const float* logits, const int64_t* labels, int64_t batch, int n_class, int64_t pixels,
                                  float* stats, double* vec, void* workspace, size_t workspace_bytes, slcl_stream_t stream_) {
  if (!vec) return SLCL_ERR_INVALID_ARGUMENT;
  const int st = seg_fwd_check(logits, labels, batch, n_class, pixels, stats, workspace, workspace_bytes);
  if (st != SLCL_OK) return st;
  cudaStream_t stream = (cudaStream_t)stream_;
  float* partial = reinterpret_cast<float*>(workspace);
  const int bpi = seg_sweep(logits, labels, batch, n_class, pixels, partial, stream);
  seg_finalize_vec_kernel<false><<<1, kThreads, 0, stream>>>(partial, (int)batch, bpi, n_class, stats, vec, nullptr,
                                                             PeerCtx{});
  return check_launch("slcl_seg_fwd_local");
}

extern "C" int slcl_seg_finish(const double* vec, int n_class, float* losses, slcl_stream_t stream_) {
  if (!vec || !losses || n_class < 2 || n_class > KM) return SLCL_ERR_INVALID_ARGUMENT;
  seg_finish_kernel<<<1, 32, 0, (cudaStream_t)stream_>>>(vec, n_class, losses);
  return check_launch("slcl_seg_finish");
}

extern "C" int slcl_seg_bwd(const float* logits, const int64_t* labels, int64_t batch, int n_class, int64_t pixels,
                            const float* stats, const float* grad_losses, float* dlogits, slcl_stream_t stream_) {
  if (!logits || !labels || batch <= 0 || pixels <= 0 || !stats || !grad_losses || !dlogits) return SLCL_ERR_INVALID_ARGUMENT;
  if (n_class < 2 || n_class > KM) return SLCL_ERR_INVALID_ARGUMENT;
  const int st = seg_bwd_launch<false>(logits, labels, batch, n_class, pixels, stats, nullptr, grad_losses, dlogits,
                                       (cudaStream_t)stream_);
  if (st != SLCL_OK) return st;
  return check_launch("slcl_seg_bwd");
}

extern "C" int slcl_seg_bwd_global(const float* logits, const int64_t* labels, int64_t batch, int n_class, int64_t pixels,
                                   const float* stats, const double* vec, const float* grad_losses, float* dlogits,
                                   slcl_stream_t stream_) {
  if (!logits || !labels || batch <= 0 || pixels <= 0 || !stats || !vec || !grad_losses || !dlogits)
    return SLCL_ERR_INVALID_ARGUMENT;
  if (n_class < 2 || n_class > KM) return SLCL_ERR_INVALID_ARGUMENT;
  const int st = seg_bwd_launch<true>(logits, labels, batch, n_class, pixels, stats, vec, grad_losses, dlogits,
                                      (cudaStream_t)stream_);
  if (st != SLCL_OK) return st;
  return check_launch("slcl_seg_bwd_global");
}

extern "C" int slcl_entropy_map(const float* prob, int64_t n_elems, int n_class, float* out, const float* grad_out,
                                float* dprob, slcl_stream_t stream_) {
  if (!prob || n_elems <= 0 || n_class < 2 || (!out && !dprob) || (dprob && !grad_out)) return SLCL_ERR_INVALID_ARGUMENT;
  const float inv_log2c = 1.0f / log2f((float)n_class);
  entropy_map_kernel<<<(unsigned)ceil_div<int64_t>(n_elems, kThreads), kThreads, 0, (cudaStream_t)stream_>>>(
      prob, n_elems, inv_log2c, out, grad_out, dprob);
  return check_launch("slcl_entropy_map");
}
