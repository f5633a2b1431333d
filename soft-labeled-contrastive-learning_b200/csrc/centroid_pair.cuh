// centroid_pair.cuh -- the centroid <-> centroid terms of one MCCL step as block-level device functions, shared by
// centroid_loss.cu (slcl_centroid_loss / slcl_mccl_losses) and the tail of the fused MCCL step in class_sums.cu
// (slcl_mccl_step_*), so both compute every term with the same arithmetic.
//
// Replaces (reference, file:line):
//   ContrastiveLoss.forward   utils/loss.py:241-275
//   inline CNR                trainer/Trainer_MCCL.py:303-315
// Closed form: SURVEY.md appendix A.5.  Every function here is called by all threads of one 256-thread block.
#pragma once

#include "common.cuh"

#include <math.h>

namespace slcl {
namespace cpair {

constexpr int kThreads = 256;
constexpr int kWarps = kThreads / 32;
constexpr int KM = SLCL_MAX_CLASSES;

__device__ __forceinline__ float row_dot(const float* a, const float* b, int C, int lane) {
  float t = 0.f;
  for (int c = lane; c < C; c += 32) t = fmaf(a[c], b[c], t);
  return warp_sum(t);
}

// mode 0/1: contrastive (plain / split); mode 2: CNR.  One thread block; d_s / d_t double as scratch.
__device__ __forceinline__ void centroid_pair(const float* __restrict__ s, const float* __restrict__ t, int K, int C, int mode,
                                              int first, int last, int norm, float* loss, float* d_s, float* d_t) {
  __shared__ float ns[KM], nt[KM];          // row norms
  __shared__ float U[KM][KM], V[KM][KM];    // t_hat.s_hat, t_hat.t_hat
  __shared__ float A[KM][KM], B[KM][KM];    // dL/dU, dL/dV
  __shared__ float ps[KM], pt[KM];          // x_hat . dx_hat  (normalisation backward)
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;

  for (int r = warp; r < 2 * K; r += kWarps) {
    const float* row = (r < K) ? s + (int64_t)r * C : t + (int64_t)(r - K) * C;
    float n = sqrtf(row_dot(row, row, C, lane));
    if (lane == 0) { if (r < K) ns[r] = n; else nt[r - K] = n; }
  }
  __syncthreads();

  if (mode == 2) {
    // CNR = mean_k (||t_k|| - ||s_k||)^2     (F.mse_loss of the row norms)
    if (threadIdx.x == 0) {
      float acc = 0.f;
      for (int k = 0; k < K; ++k) { float d = nt[k] - ns[k]; acc += d * d; }
      loss[0] = acc / (float)K;
    }
    for (int idx = threadIdx.x; idx < K * C; idx += kThreads) {
      int k = idx / C;
      float d = 2.0f * (nt[k] - ns[k]) / (float)K;
      d_t[idx] = nt[k] > 0.f ? d * t[idx] / nt[k] : 0.f;
      d_s[idx] = ns[k] > 0.f ? -d * s[idx] / ns[k] : 0.f;
    }
    return;
  }

  // scale factors of x_hat = x / (||x|| + 1e-7)   (utils/loss.py:242-246); 1 when norm == 0
  for (int pair = warp; pair < 2 * K * K; pair += kWarps) {
    int which = pair / (K * K), ij = pair % (K * K), i = ij / K, j = ij % K;
    const float* ti = t + (int64_t)i * C;
    const float* other = which == 0 ? s + (int64_t)j * C : t + (int64_t)j * C;
    float d = row_dot(ti, other, C, lane);
    if (lane == 0) {
      float si = norm ? 1.0f / (nt[i] + 1e-7f) : 1.0f;
      float sj = norm ? 1.0f / ((which == 0 ? ns[j] : nt[j]) + 1e-7f) : 1.0f;
      if (which == 0) U[i][j] = d * si * sj; else V[i][j] = d * si * sj;
    }
  }
  __syncthreads();

  if (threadIdx.x < K) {
    const int i = threadIdx.x;
    float den = 0.f;
    for (int j = 0; j < K; ++j) den += expf(U[i][j]);                 // :264, :267
    float den2 = 0.f;
    for (int j = 0; j < K; ++j) den2 += expf(V[i][j]);                // :265
    den = den + den2 + 1e-7f;
    const bool rowon = (i >= first && i < last);                      // :266
    const float eii = expf(U[i][i]), fii = expf(V[i][i]);
    float li = 0.f;
    if (rowon) {
      if (mode == 1) li = 0.5f * (-logf(eii / den) - logf(fii / den));   // :268-270
      else li = -logf((eii + fii) / den);                                // :272-273
    }
    ps[i] = li;                                                          // reuse as scratch for the row losses
    for (int j = 0; j < K; ++j) {
      float a = 0.f, b = 0.f;
      if (rowon) {
        a = expf(U[i][j]) / den;
        b = expf(V[i][j]) / den;
        if (j == i) {
          if (mode == 1) { a -= 0.5f; b -= 0.5f; }
          else { a -= eii / (eii + fii); b -= fii / (eii + fii); }
        }
      }
      A[i][j] = a; B[i][j] = b;
    }
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    float acc = 0.f;
    for (int i = 0; i < K; ++i) acc += ps[i];
    loss[0] = acc;
  }
  __syncthreads();

  // gradients w.r.t. the unit rows, written to the outputs as scratch
  for (int idx = threadIdx.x; idx < K * C; idx += kThreads) {
    const int k = idx / C, c = idx % C;
    const float sk = norm ? 1.0f / (ns[k] + 1e-7f) : 1.0f;
    const float tk = norm ? 1.0f / (nt[k] + 1e-7f) : 1.0f;
    float gs = 0.f, gt = 0.f;
    for (int i = 0; i < K; ++i) {
      const float ti_hat = t[(int64_t)i * C + c] * (norm ? 1.0f / (nt[i] + 1e-7f) : 1.0f);
      const float si_hat = s[(int64_t)i * C + c] * (norm ? 1.0f / (ns[i] + 1e-7f) : 1.0f);
      gs = fmaf(A[i][k], ti_hat, gs);                       // d s_hat_k = sum_i A_ik t_hat_i
      gt = fmaf(A[k][i], si_hat, gt);                       // d t_hat_k = sum_j A_kj s_hat_j
      gt = fmaf(B[k][i] + B[i][k], ti_hat, gt);             //           + sum_j (B_kj + B_jk) t_hat_j
    }
    d_s[idx] = gs;
    d_t[idx] = gt;
    (void)sk; (void)tk;
  }
  __syncthreads();
  if (!norm) return;
  // x_hat = x/(n+eps):  dx = dxh/(n+eps) - x (x.dxh) / (n (n+eps)^2)
  for (int r = warp; r < 2 * K; r += kWarps) {
    const bool is_s = r < K;
    const int k = is_s ? r : r - K;
    const float* x = (is_s ? s : t) + (int64_t)k * C;
    const float* g = (is_s ? d_s : d_t) + (int64_t)k * C;
    float d = row_dot(x, g, C, lane);
    if (lane == 0) { if (is_s) ps[k] = d; else pt[k] = d; }
  }
  __syncthreads();
  for (int idx = threadIdx.x; idx < K * C; idx += kThreads) {
    const int k = idx / C;
    {
      const float n = ns[k], ne = n + 1e-7f;
      const float corr = n > 0.f ? ps[k] / (n * ne * ne) : 0.f;
      d_s[idx] = d_s[idx] / ne - s[idx] * corr;
    }
    {
      const float n = nt[k], ne = n + 1e-7f;
      const float corr = n > 0.f ? pt[k] / (n * ne * ne) : 0.f;
      d_t[idx] = d_t[idx] / ne - t[idx] * corr;
    }
  }
}

// All centroid <-> centroid terms of one MCCL step (trainer/Trainer_MCCL.py:303-326): pair i evaluates, for the P target
// partitions T_p, inter = CL(s = S, t = T_p), intra = CL(s = T_p, t = A), cnr = CNR(S, T_p) into scratch
// {loss_i, ds_i, dt_i}; mccl_combine then forms the weighted total and the gradients w.r.t. S, every T_p and A (a sum
// of 2P+... tiny terms per element, fixed order).
struct McclArgs {
  const float* S; const float* T; const float* A;     // [K,C], [P*K,C], [K,C] (A may be null: no intra term)
  int P, K, C, split, first, norm;
  float inter_w, intra_w, cnr_w;
  float* scratch;                                      // [3P] x {loss (padded to 4 floats), ds [K*C], dt [K*C]}
  float* loss; float* dS; float* dT; float* dA;
};

__device__ __forceinline__ void mccl_pair(const McclArgs& a, int i) {
  const int kind = i / a.P, p = i % a.P;
  const int kc = a.K * a.C;
  float* out = a.scratch + (size_t)i * (4 + 2 * kc);
  const float* Tp = a.T + (size_t)p * kc;
  if (kind == 0) centroid_pair(a.S, Tp, a.K, a.C, a.split ? 1 : 0, a.first, a.K, a.norm, out, out + 4, out + 4 + kc);
  else if (kind == 1) {
    if (a.A != nullptr) centroid_pair(Tp, a.A, a.K, a.C, a.split ? 1 : 0, a.first, a.K, a.norm, out, out + 4, out + 4 + kc);
  } else centroid_pair(a.S, Tp, a.K, a.C, 2, 0, a.K, 0, out, out + 4, out + 4 + kc);
}

// The weighted total and the three terms (for logging) into loss[0..3], and every gradient element of d total / d
// {S, T_p, A}: spread over the grid (mccl_combine_kernel), or over the calling block alone (ONE_BLOCK: the MCCL step's
// tail, whose last block runs it).
template <bool ONE_BLOCK>
__device__ __forceinline__ void mccl_combine(const McclArgs& a) {
  const int kc = a.K * a.C;
  const size_t stride = 4 + 2 * (size_t)kc;
  const float wi = a.inter_w / a.P, wa = (a.A != nullptr) ? a.intra_w / a.P : 0.f, wc = a.cnr_w / a.P;
  auto slot = [&](int kind, int p) { return a.scratch + (size_t)(kind * a.P + p) * stride; };
  if (ONE_BLOCK ? threadIdx.x == 0 : (blockIdx.x == 0 && threadIdx.x == 0)) {
    float inter = 0.f, intra = 0.f, cnr = 0.f;
    for (int p = 0; p < a.P; ++p) { inter += slot(0, p)[0]; if (a.A) intra += slot(1, p)[0]; cnr += slot(2, p)[0]; }
    a.loss[0] = wi * inter + wa * intra + wc * cnr;
    a.loss[1] = inter / a.P; a.loss[2] = intra / a.P; a.loss[3] = cnr / a.P;      // the three terms, for logging
  }
  for (int idx = ONE_BLOCK ? threadIdx.x : blockIdx.x * kThreads + threadIdx.x; idx < kc;
       idx += ONE_BLOCK ? kThreads : gridDim.x * kThreads) {
    float ds = 0.f, da = 0.f;
    for (int p = 0; p < a.P; ++p) {
      const float* in = slot(0, p) + 4;
      const float* cn = slot(2, p) + 4;
      ds += wi * in[idx] + wc * cn[idx];
      float dt = wi * in[kc + idx] + wc * cn[kc + idx];
      if (a.A != nullptr) { const float* ia = slot(1, p) + 4; dt += wa * ia[idx]; da += wa * ia[kc + idx]; }
      a.dT[(size_t)p * kc + idx] = dt;
    }
    a.dS[idx] = ds;
    if (a.dA != nullptr) a.dA[idx] = da;
  }
}

}  // namespace cpair
}  // namespace slcl
