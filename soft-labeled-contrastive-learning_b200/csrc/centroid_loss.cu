// centroid_loss.cu -- centroid <-> centroid InfoNCE and the centroid-norm
// regulariser on [K,C] inputs: loss and both gradients in ONE launch.
//
// Replaces (reference, file:line):
//   ContrastiveLoss.forward   utils/loss.py:241-275   (~30 tiny launches fwd, as many bwd)
//   inline CNR                trainer/Trainer_MCCL.py:303-315
// Closed form: SURVEY.md appendix A.5 (the device functions: centroid_pair.cuh).  This op is launch-latency bound, not
// bandwidth bound: the whole problem (<= 8 x 2048 floats per operand) lives in
// one CTA; the product goal is 1 launch instead of ~60.
#include "centroid_pair.cuh"
#include "common.cuh"

#include <math.h>

namespace slcl {
namespace {

constexpr int kThreads = cpair::kThreads;
constexpr int KM = cpair::KM;
using cpair::McclArgs;

__global__ void __launch_bounds__(kThreads) centroid_loss_kernel(const float* __restrict__ s, const float* __restrict__ t,
                                                                 int K, int C, int mode, int first, int last, int norm,
                                                                 float* loss, float* d_s, float* d_t) {
  cpair::centroid_pair(s, t, K, C, mode, first, last, norm, loss, d_s, d_t);
}

// All centroid <-> centroid terms of one MCCL step in two launches: block i of mccl_pairs_kernel evaluates pair i
// (cpair::mccl_pair), mccl_combine_kernel forms the weighted total and every gradient (cpair::mccl_combine).
__global__ void __launch_bounds__(kThreads) mccl_pairs_kernel(const McclArgs a) { cpair::mccl_pair(a, blockIdx.x); }
__global__ void __launch_bounds__(kThreads) mccl_combine_kernel(const McclArgs a) {
  cpair::mccl_combine<false>(a);
}

}  // namespace
}  // namespace slcl

using namespace slcl;

extern "C" int slcl_centroid_loss(const float* centroid_s, const float* centroid_t, int n_class, int64_t channels,
                                  int mode, int first_row, int n_rows, int norm, float* loss, float* d_s, float* d_t,
                                  slcl_stream_t stream_) {
  if (!centroid_s || !centroid_t || !loss || !d_s || !d_t) return SLCL_ERR_INVALID_ARGUMENT;
  if (n_class < 1 || n_class > KM || channels <= 0 || mode < 0 || mode > 2) return SLCL_ERR_INVALID_ARGUMENT;
  if (mode != 2 && (first_row < 0 || n_rows > n_class || first_row > n_rows)) return SLCL_ERR_INVALID_ARGUMENT;
  centroid_loss_kernel<<<1, kThreads, 0, (cudaStream_t)stream_>>>(centroid_s, centroid_t, n_class, (int)channels, mode,
                                                                 first_row, n_rows, norm, loss, d_s, d_t);
  return check_launch("slcl_centroid_loss");
}

extern "C" size_t slcl_mccl_losses_workspace_bytes(int n_partitions, int n_class, int64_t channels) {
  if (n_partitions < 1 || n_class < 1 || channels <= 0) return 0;
  return align_up((size_t)3 * n_partitions * (4 + 2 * (size_t)n_class * channels) * sizeof(float), 256);
}

extern "C" int slcl_mccl_losses(const float* centroid_s, const float* centroid_t_parts, const float* centroid_t_aug,
                                int n_partitions, int n_class, int64_t channels, int split, int bg, int norm,
                                float inter_w, float intra_w, float cnr_w, float* losses, float* d_s, float* d_t_parts,
                                float* d_t_aug, void* workspace, size_t workspace_bytes, slcl_stream_t stream_) {
  if (!centroid_s || !centroid_t_parts || !losses || !d_s || !d_t_parts || !workspace) return SLCL_ERR_INVALID_ARGUMENT;
  if ((centroid_t_aug == nullptr) != (d_t_aug == nullptr)) return SLCL_ERR_INVALID_ARGUMENT;
  if (n_partitions < 1 || n_partitions > 16 || n_class < 1 || n_class > KM || channels <= 0) return SLCL_ERR_INVALID_ARGUMENT;
  if (workspace_bytes < slcl_mccl_losses_workspace_bytes(n_partitions, n_class, channels) || !aligned16(workspace))
    return SLCL_ERR_WORKSPACE;
  McclArgs a{};
  a.S = centroid_s; a.T = centroid_t_parts; a.A = centroid_t_aug;
  a.P = n_partitions; a.K = n_class; a.C = (int)channels; a.split = split; a.first = bg ? 0 : 1; a.norm = norm;
  a.inter_w = inter_w; a.intra_w = intra_w; a.cnr_w = cnr_w;
  a.scratch = reinterpret_cast<float*>(workspace);
  a.loss = losses; a.dS = d_s; a.dT = d_t_parts; a.dA = d_t_aug;
  cudaStream_t stream = (cudaStream_t)stream_;
  mccl_pairs_kernel<<<3 * n_partitions, kThreads, 0, stream>>>(a);
  const int kc = n_class * (int)channels;
  mccl_combine_kernel<<<ceil_div(kc, kThreads) < 8 ? ceil_div(kc, kThreads) : 8, kThreads, 0, stream>>>(a);
  return check_launch("slcl_mccl_losses");
}
