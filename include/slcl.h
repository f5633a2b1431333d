/*
 * slcl.h -- C ABI of libslcl.so: the B200 (sm_100a) implementation of the SLCL
 * contrastive-loss hot path.
 *
 * The reference (Dinhthixuanbinh/Soft-Labeled-Contrastive-Learning) has no FFI
 * layer: its boundary for this path is a set of Python callables
 * (utils/loss.py, utils/losses.py, utils/utils_.py:479-624).  Each entry point
 * below names the reference callable (file:line) whose arithmetic it
 * replaces; the Python package `slcl` keeps the reference signatures and
 * calls these functions through ctypes (see INTEGRATION.md).
 *
 * Conventions (all entry points):
 *   - plain pointers and sizes only; every pointer is a DEVICE pointer unless
 *     the parameter name ends in `_host`;
 *   - the caller owns and allocates every output and the workspace; nothing
 *     is allocated or freed inside the library;
 *   - launches are asynchronous on `stream` (a cudaStream_t passed as void*);
 *     no host synchronisation, no host read-back;
 *   - return value: 0 = SLCL_OK, negative = error (slcl_strerror()); errors
 *     are detected before any launch, outputs are then untouched;
 *   - no global mutable state besides cached device attributes, so any thread
 *     may call, one process per GPU;
 *   - "pixel order" is the reference's (b, h, w) order of an NCHW map:
 *     pixel i = b*HW + p.
 */
#ifndef SLCL_H_
#define SLCL_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SLCL_VERSION 115            /* major*100 + minor */
#define SLCL_MAX_CLASSES 8          /* K <= 8 (reference uses 4; MPCL defaults to 5) */
#define SLCL_MAX_WEIGHT_COLS 16     /* partitions * classes <= 16 for class sums */

enum {
  SLCL_OK = 0,
  SLCL_ERR_INVALID_ARGUMENT = -1,   /* null pointer, non-positive size, K out of range ... */
  SLCL_ERR_UNSUPPORTED = -2,        /* shape/stride combination without a kernel */
  SLCL_ERR_WORKSPACE = -3,          /* workspace_bytes smaller than slcl_*_workspace_bytes() */
  SLCL_ERR_CUDA = -4                /* launch failed; slcl_last_cuda_error() has the text */
};

typedef void* slcl_stream_t;        /* cudaStream_t */

int         slcl_version(void);
const char* slcl_strerror(int status);
const char* slcl_last_cuda_error(void);     /* thread-local text of the last SLCL_ERR_CUDA */

/* Strided view of a feature map: element (b, c, p) lives at
 * base[b*stride_b + c*stride_c + p*stride_p] (strides in elements).
 * NCHW contiguous: {C*HW, HW, 1}; rows [N,C] (reference MPCL.forward input,
 * utils/loss.py:484): B=1, HW=N, {0, 1, C}. */
typedef struct {
  int64_t batch;       /* B */
  int64_t channels;    /* C */
  int64_t pixels;      /* HW (pixels per image) */
  int64_t stride_b, stride_c, stride_p;
} slcl_map_t;

/* ---------------------------------------------------------------------------
 * Prototype path: pixel -> class-centre margin InfoNCE.
 * Replaces MPCL.forward (utils/loss.py:484-573) fused with the layout and
 * normalisation work of mpcl_loss_calc (utils/loss.py:592-601) and the
 * autograd backward of both.
 * ------------------------------------------------------------------------- */
typedef struct {
  int   n_class;           /* K, 2..SLCL_MAX_CLASSES          (MPCL.num_class) */
  float temperature;       /* T                                (utils/loss.py:472) */
  float base_temperature;  /* T_b                              (:473) */
  float margin;            /* m; cos_m, sin_m, th, mm derive from it (:475-480) */
  int   easy_margin;       /* :538-541 */
  int   normalize;         /* 1: L2-normalise pixels and centres (mpcl_loss_calc :595,:600);
                              0: inputs are already unit vectors (direct MPCL.forward call) */
} slcl_proto_params_t;

size_t slcl_proto_workspace_bytes(int64_t n_pixels);

/* Forward.  labels [N] int64 (values outside [0,K) give an all-zero positive
 * row, as torch.eq against arange(K) does at :513) OR soft_mask [N,K] fp32
 * row-major (:516-517); exactly one of them non-null.  sel [N] fp32 or null
 * (pixel_sel_loc, :558-565).  centres [K,C] fp32 row-major, raw (un-normalised
 * when params.normalize).
 * Outputs: stash [(K+1)*N] fp32 (per-pixel backward coefficients, planar),
 *          cstate [K*C + K] fp32 (unit centres, centre norms),
 *          scal [4] fp32 = {loss, d loss / d (sum of weighted rows), sum(sel) or N, sum(sel*row loss)}. */
int slcl_proto_fwd(const float* feat, const slcl_map_t* map,
                   const int64_t* labels, const float* soft_mask, const float* sel,
                   const float* centres, const slcl_proto_params_t* params,
                   float* stash, float* cstate, float* scal,
                   void* workspace, size_t workspace_bytes, slcl_stream_t stream);

/* Fused target step (SURVEY.md 8(f)-1): generate_pseudo_label (utils/utils_.py:597-624) and the target-side
 * mpcl_loss_calc forward (trainer/Trainer_MPSCL.py:135,144) in ONE read of the target feature map.  Writes
 * label [N] int64 and sel [N] fp32 exactly as slcl_pseudo_label would, and stash / cstate / scal exactly as
 * slcl_proto_fwd(labels = label, sel = sel) would.  params->normalize must be 1. */
int slcl_proto_fwd_target(const float* feat, const slcl_map_t* map, const float* centres,
                          const slcl_proto_params_t* params, float sel_threshold,
                          int64_t* label, float* sel, float* stash, float* cstate, float* scal,
                          void* workspace, size_t workspace_bytes, slcl_stream_t stream);

/* Data-parallel use (SURVEY.md 8(e)): each rank runs slcl_proto_fwd on its shard, the
 * caller all-reduces scal[2..3] (weight sum, weighted row-loss sum) across ranks, then this
 * call recomputes scal[0] (global loss) and scal[1] (global coefficient) in place. */
int slcl_proto_rescale(float* scal, int has_sel, slcl_stream_t stream);

/* ---------------------------------------------------------------------------
 * NVLink peer-memory mailboxes (SURVEY.md 8(e)): the small exchanges of the data-parallel path -- the loss pair
 * {sum sel, sum sel*row loss} and the per-class sums [sets*K, C+1] fp64 -- are done INSIDE our own kernels with P2P
 * stores into the peers' mailboxes instead of NCCL collectives.  Every rank owns a zero-initialised mailbox of
 * slcl_peer_mailbox_bytes(world, capacity_words) bytes in memory that all ranks of the box have mapped (e.g.
 * torch.distributed._symmetric_memory); mailboxes_dev is a DEVICE array of `world` pointers, entry r = rank r's
 * mailbox in this process' address space.  capacity_words = payload words per message (2 per double; >= 2).
 * Every rank must make the same sequence of peer calls, on one stream per mailbox set.  A peer that does not arrive
 * within timeout_s seconds (0 = wait for ever, like NCCL) poisons the result with NaN instead of hanging; mailbox
 * word 1 counts such time-outs.
 * ------------------------------------------------------------------------- */
typedef struct {
  const void* mailboxes_dev;
  int rank, world;            /* world <= 16 */
  int64_t capacity_words;
  double timeout_s;
} slcl_peer_t;

size_t slcl_peer_mailbox_bytes(int world, int64_t capacity_words);

/* slcl_proto_rescale with the exchange fused in: ONE kernel that sends scal[2..3] to every peer, waits for theirs,
 * adds in rank order and rewrites scal[0..3] exactly as all-reduce + slcl_proto_rescale would. */
int slcl_proto_rescale_peer(float* scal, int has_sel, const slcl_peer_t* peer, slcl_stream_t stream);

/* In-place sum over the ranks of buf[0..n) (fp64, added in rank order: identical bits on every rank); one kernel,
 * one warp per element.  2*n <= capacity_words. */
int slcl_peer_allreduce_f64(double* buf, int64_t n, const slcl_peer_t* peer, slcl_stream_t stream);

/* Data-parallel forms of the two forwards: with `peer` (may be null = the plain call) the finaliser kernel exchanges
 * {weight sum, weighted row-loss sum} with the other ranks through the mailboxes before it writes scal, so scal[0] is
 * the loss over the GLOBAL batch and scal[1] the global coefficient -- no slcl_proto_rescale(_peer) call, no extra launch
 * between forward and backward.  (slcl_target_step does the same with its `peer`.) */
int slcl_proto_fwd_peer(const float* feat, const slcl_map_t* map,
                        const int64_t* labels, const float* soft_mask, const float* sel,
                        const float* centres, const slcl_proto_params_t* params,
                        float* stash, float* cstate, float* scal, const slcl_peer_t* peer, int split_phase,
                        void* workspace, size_t workspace_bytes, slcl_stream_t stream);
/* split_phase != 0 (fused forward + backward steps that read the loss only afterwards): the forward's finaliser only
 * SENDS this rank's pair; the matching slcl_proto_bwd_peer call -- same mailboxes, same stream, MUST follow -- receives,
 * adds and rewrites scal (block 0) while its other blocks already stream their first loads, so the exchange latency
 * hides behind the backward's launch and prologue.  scal[0] (the global loss) is valid after that backward. */
int slcl_proto_bwd_peer(const float* feat, const slcl_map_t* map,
                        const float* stash, const float* cstate, float* scal, const float* grad_out,
                        const slcl_proto_params_t* params, float* dfeat,
                        const slcl_peer_t* peer, int has_sel, slcl_stream_t stream);
int slcl_proto_fwd_target_peer(const float* feat, const slcl_map_t* map, const float* centres,
                               const slcl_proto_params_t* params, float sel_threshold,
                               int64_t* label, float* sel, float* stash, float* cstate, float* scal,
                               const slcl_peer_t* peer, void* workspace, size_t workspace_bytes, slcl_stream_t stream);

/* The same fused target step PLUS the per-class sums of the target map under the pseudo labels it has just generated
 * (hard target centroids: cal_centroid with the map's own arg-max labels, utils/utils_.py:524-529; weights one-hot(label),
 * or one-hot(label) * sel when weight_by_sel) -- ONE pass over F_t: every pixel's channel vector sits in a shared-memory
 * stage, "pixel warps" derive label / sel / loss row / stash from it and the class-sum consumers read the same stage.
 * label, sel, stash, cstate are bit-identical to slcl_proto_fwd_target's; scal likewise up to the order of the fp64 block
 * partials.  sums [K, C+1] fp64, centroids [K, C] / inv_weight [K] as slcl_centroids_fwd (previous may be null; peer may be
 * null, else the sums are all-reduced through the mailboxes).  Contiguous NCHW maps with HW % 4 == 0 and C <= 128
 * (K <= 5 when C > 64); anything else returns SLCL_ERR_UNSUPPORTED and the caller uses the separate entry points. */
size_t slcl_target_step_workspace_bytes(int64_t channels, int n_class);
int slcl_target_step(const float* feat, int64_t batch, int64_t channels, int64_t pixels, const float* centres,
                     const slcl_proto_params_t* params, float sel_threshold, int weight_by_sel,
                     int64_t* label, float* sel, float* stash, float* cstate, float* scal, double* sums,
                     const float* previous, float momentum, float* centroids, float* inv_weight,
                     const slcl_peer_t* peer, void* workspace, size_t workspace_bytes, slcl_stream_t stream);

/* Backward w.r.t. the feature map.  grad_out: device scalar dL/dloss.
 * dfeat uses the strides of `map`. */
int slcl_proto_bwd(const float* feat, const slcl_map_t* map,
                   const float* stash, const float* cstate, const float* scal, const float* grad_out,
                   const slcl_proto_params_t* params, float* dfeat, slcl_stream_t stream);
/* Gradients of the same loss w.r.t. the two inputs no reference caller differentiates (utils/loss.py:516-517, :558-565):
 * dmask [N,K] = d loss / d soft_mask (needs soft_mask), dsel [N] = d loss / d pixel_sel_loc (needs sel); either may be
 * null.  A pass of its own over `feat` (cosines recomputed) with the forward's cstate and scal; dL/dloss = *grad_out. */
int slcl_proto_bwd_aux(const float* feat, const slcl_map_t* map, const int64_t* labels, const float* soft_mask,
                       const float* sel, const float* cstate, const float* scal, const float* grad_out,
                       const slcl_proto_params_t* params, float* dmask, float* dsel, slcl_stream_t stream);

/* Backward w.r.t. the raw centres [K,C] (only when they require grad; both
 * reference callers pass detached centres, trainer/Trainer_MPSCL.py:139,145). */
size_t slcl_proto_bwd_centres_workspace_bytes(int64_t n_pixels, int64_t channels, int n_class);
int slcl_proto_bwd_centres(const float* feat, const slcl_map_t* map,
                           const float* stash, const float* cstate, const float* scal, const float* grad_out,
                           const slcl_proto_params_t* params, float* dcentres,
                           void* workspace, size_t workspace_bytes, slcl_stream_t stream);

/* generate_pseudo_label (utils/utils_.py:597-624): label = argmax_k cos(x_i, c_k)
 * (first index on ties), sel = (top1 - top2 > threshold) ? 1 : 0. */
int slcl_pseudo_label(const float* feat, const slcl_map_t* map, const float* centres, int n_class,
                      float threshold, int64_t* label, float* sel,
                      void* workspace, size_t workspace_bytes, slcl_stream_t stream);

/* ---------------------------------------------------------------------------
 * Class sums: one pass over an NCHW map producing, per weight column j
 * (j = partition*K + class), sum_i w_ij * x_i  (C values) and sum_i w_ij.
 * Replaces the per-class masked sums of update_class_center_iter
 * (utils/utils_.py:580-590) and cal_centroid (utils/utils_.py:509-540).
 *
 * Weights:  hard   w_ik = [label_i == k]                              (labels != null)
 *           soft   w_ik = probs[b,k,p] * cert_i      (weighted & SLCL_SOFT_WEIGHTED)  (probs  != null)
 *           argmax w_ik = [argmax_k probs == k] * cert_i (weighted == 0)
 *           cert_i = [max_k probs >= threshold] if 0 < threshold < 1 else 1
 *           and, when part_id != null, times [part_id_i == partition].
 * `weighted` is a flags word.  SLCL_SOFT_LOGITS: `probs` holds the logits z [B,K,HW] and the kernels use
 * probs = softmax_k(z) (per pixel: zmax = max_k z_k, arg-max = its first index, s = sum_k expf(z_k - zmax),
 * p_k = expf(z_k - zmax) / s, max_k p_k = 1/s), the same weights as above from one read of z.  Soft labels only:
 * the flag with `labels`, or any other bit, returns SLCL_ERR_INVALID_ARGUMENT.
 * Output sums [P*K, C+1] fp64 row-major: columns 0..C-1 = weighted feature
 * sums, column C = weight sum (exact integer counts for hard labels).  This is
 * the buffer a multi-GPU caller all-reduces (SURVEY.md section 8(e)).
 * ------------------------------------------------------------------------- */
#define SLCL_SOFT_WEIGHTED 1          /* soft weights p_k * cert (else the arg-max one-hot) */
#define SLCL_SOFT_LOGITS   2          /* `probs` are logits; dprobs of slcl_centroid_bwd receives dL/dlogits */
size_t slcl_class_sums_workspace_bytes(int64_t batch, int64_t channels, int64_t pixels, int n_cols);
int slcl_class_sums(const float* feat, int64_t batch, int64_t channels, int64_t pixels,
                    const int64_t* labels, const float* probs, int weighted, float threshold,
                    const int32_t* part_id, int n_partitions, int n_class,
                    double* sums, void* workspace, size_t workspace_bytes, slcl_stream_t stream);

/* update_class_center_iter tail (utils/utils_.py:585-592): per class
 * batch = sum/count, or the old centre when count == 0 (decided on the
 * device, no host sync); new = m*old + (1-m)*batch. */
int slcl_ema_finalize(const double* sums, const float* old_centres, float m, int n_class, int64_t channels,
                      float* new_centres, slcl_stream_t stream);

/* cal_centroid tail (utils/utils_.py:520-523,538,552-563): centroid = sum/(weight+1e-7),
 * optional EMA with `previous` [K,C] (same tensor for every set) when non-null.
 * Outputs centroids [sets*K, C] fp32 and inv_weight [sets*K] fp32 = 1/(weight+1e-7). */
int slcl_centroid_finalize(const double* sums, const float* previous, float momentum, int n_sets, int n_class,
                           int64_t channels, float* centroids, float* inv_weight, slcl_stream_t stream);

/* Fused forms (two launches: the sweep, then ONE kernel that sums the per-block partials in fp64, optionally
 * all-reduces them across ranks through the peer mailboxes -- `peer` may be null -- and whose last block runs the
 * finaliser):
 *   slcl_class_centres_update = slcl_class_sums(hard labels) [+ all-reduce] + slcl_ema_finalize
 *                               (update_class_center_iter, utils/utils_.py:568-594, over the GLOBAL batch)
 *   slcl_centroids_fwd        = slcl_class_sums [+ all-reduce] + slcl_centroid_finalize
 *                               (cal_centroid, utils/utils_.py:479-565)
 * `sums` [P*K, C+1] fp64 is still written (the backward needs it); with `peer` it holds the GLOBAL sums, so class
 * counts match a single-GPU run bit for bit.  Workspace: slcl_class_sums_workspace_bytes(). */
int slcl_class_centres_update(const float* feat, int64_t batch, int64_t channels, int64_t pixels,
                              const int64_t* labels, int n_class, const float* old_centres, float m,
                              float* new_centres, double* sums, const slcl_peer_t* peer,
                              void* workspace, size_t workspace_bytes, slcl_stream_t stream);
int slcl_centroids_fwd(const float* feat, int64_t batch, int64_t channels, int64_t pixels,
                       const int64_t* labels, const float* probs, int weighted, float threshold,
                       const int32_t* part_id, int n_partitions, int n_class,
                       const float* previous, float momentum, float* centroids, float* inv_weight,
                       double* sums, const slcl_peer_t* peer,
                       void* workspace, size_t workspace_bytes, slcl_stream_t stream);

/* Backward of the (soft / hard) centroid of cal_centroid (SURVEY.md appendix A.4).
 * With gc_j = grad_centroids_j * ema_scale / (W_j + 1e-7) and mu_j = S_j / (W_j + 1e-7)
 * (S, W from `sums`, the same -- possibly all-reduced -- buffer the forward used):
 *   dfeat[b,c,p]  = sum_j w_ij * gc[j,c]
 *   dprobs[b,k,p] = cert_i * [part_i] * ( x_i . gc_j - mu_j . gc_j ),  j = part_i*K + k   (soft weighted only)
 * With SLCL_SOFT_LOGITS (`probs` = logits z, p = softmax_k(z) as in slcl_class_sums), with g_ik the value above:
 *   dprobs[b,k,p] = dL/dz_ik = p_ik * ( g_ik - sum_m p_im g_im )
 * ema_scale = 1 - momentum when the forward applied the EMA, else 1.
 * dprobs may be null (hard labels / arg-max weights: no gradient to the labels). */
size_t slcl_centroid_bwd_workspace_bytes(int64_t channels, int n_cols);
int slcl_centroid_bwd(const float* feat, int64_t batch, int64_t channels, int64_t pixels,
                      const int64_t* labels, const float* probs, int weighted, float threshold,
                      const int32_t* part_id, int n_partitions, int n_class,
                      const float* grad_centroids, const double* sums, float ema_scale,
                      float* dfeat, float* dprobs, void* workspace, size_t workspace_bytes, slcl_stream_t stream);

/* ---------------------------------------------------------------------------
 * Centroid <-> centroid InfoNCE and centroid-norm regulariser on [K,C].
 * Replaces ContrastiveLoss.forward (utils/loss.py:241-275; `tau` is unused
 * there and therefore absent here) and the inline CNR of
 * trainer/Trainer_MCCL.py:303-315.  One block; writes the loss and both
 * gradients (for dL/dloss = 1) in a single launch.
 *   mode 0: contrastive, rows [first_row, n_rows)   (n_rows is the reference's hard-coded 4)
 *   mode 1: contrastive, split form (:268-270)
 *   mode 2: CNR = mean_k (||t_k|| - ||s_k||)^2
 * ------------------------------------------------------------------------- */
int slcl_centroid_loss(const float* centroid_s, const float* centroid_t, int n_class, int64_t channels,
                       int mode, int first_row, int n_rows, int norm,
                       float* loss, float* d_s, float* d_t, slcl_stream_t stream);

/* All centroid <-> centroid terms of one MCCL adaptation step (trainer/Trainer_MCCL.py:303-326) in two launches:
 *   inter = sum_p ContrastiveLoss(s = S, t = T_p) / P       intra = sum_p ContrastiveLoss(s = T_p, t = A) / P
 *   cnr   = sum_p MSE(||T_p||, ||S||) / P                    total = inter_w inter + intra_w intra + cnr_w cnr
 * S = source centroids [K,C], T = the P target-partition centroids [P*K, C] (cal_centroid's output order), A = the
 * augmented-target centroids [K,C] or null (no intra term).  losses [4] = {total, inter, intra, cnr}; d_s, d_t_parts,
 * d_t_aug = d total / d S, T, A for d/dtotal = 1.  Same arithmetic per pair as slcl_centroid_loss. */
size_t slcl_mccl_losses_workspace_bytes(int n_partitions, int n_class, int64_t channels);
int slcl_mccl_losses(const float* centroid_s, const float* centroid_t_parts, const float* centroid_t_aug,
                     int n_partitions, int n_class, int64_t channels, int split, int bg, int norm,
                     float inter_w, float intra_w, float cnr_w, float* losses, float* d_s, float* d_t_parts,
                     float* d_t_aug, void* workspace, size_t workspace_bytes, slcl_stream_t stream);

/* The MCCL loss section from the decoder outputs to the loss with its gradients (trainer/Trainer_MCCL.py:275-326) in
 * one forward and one backward call, defined as this composition:
 *   S = slcl_centroids_fwd(feat_s, labels_s, previous_s, momentum)            hard labels; no gradient (:277)
 *   T = slcl_centroids_fwd(feat_t, pred_t, part_id, n_partitions, flags, threshold)   soft labels
 *   A = slcl_centroids_fwd(feat_a, pred_a, flags, threshold)                  P = 1; optional (feat_a = pred_a = null,
 *                                                                             batch_a = 0: no intra term)
 *   losses = slcl_mccl_losses(S, T, A, split, bg, norm, inter_w, intra_w, cnr_w)
 * All maps are contiguous fp32 NCHW with the same channels and pixels (h * w); labels_s int64 [batch_s * pixels],
 * pred_* [B, K, pixels] probabilities or, with flags & SLCL_SOFT_LOGITS, logits; 2 <= K <= 8, P * K <= 16.
 * Outputs: sums [rows, C+1] fp64 and centroids [rows, C] with rows = (P + 1 + has_aug) K in the order S | T | A (sums
 * bit-identical to the separate calls'), losses [4] = {total, inter, intra, cnr}, d_centroids [rows, C] = d total / d
 * centroids (saved for the backward).
 * slcl_mccl_step_fwd: one class-sum sweep per set, then one tail kernel (reduce of every set, with `peer` one exchange of
 * the whole sums matrix -- capacity_words >= 2 rows (C+1) --, centroids, every centroid term); peer may be null.
 * slcl_mccl_step_fwd_local writes this rank's sums only; the caller sums them over the ranks (e.g. NCCL) and
 * slcl_mccl_step_finish computes the rest with the same arithmetic (its workspace:
 * slcl_mccl_step_finish_workspace_bytes).
 * slcl_mccl_step_bwd: dfeat_t / dfeat_a and, for SLCL_SOFT_WEIGHTED, dpred_t / dpred_a (each may be null; dL/dlogits
 * with SLCL_SOFT_LOGITS) of grad_out[0] * total, from the forward's sums and d_centroids: three launches, no host sync.
 * Workspace: slcl_centroid_bwd_workspace_bytes(channels, rows - K). */
size_t slcl_mccl_step_workspace_bytes(int64_t batch_s, int64_t batch_t, int64_t batch_a, int64_t channels, int64_t pixels,
                                      int n_partitions, int n_class);
size_t slcl_mccl_step_finish_workspace_bytes(int has_aug, int64_t channels, int n_partitions, int n_class);
int slcl_mccl_step_fwd(const float* feat_s, const int64_t* labels_s, int64_t batch_s, const float* feat_t,
                       const float* pred_t, const int32_t* part_id, int64_t batch_t, const float* feat_a,
                       const float* pred_a, int64_t batch_a, int64_t channels, int64_t pixels, int n_partitions,
                       int n_class, int flags, float threshold, const float* previous_s, float momentum,
                       int split, int bg, int norm, float inter_w, float intra_w, float cnr_w, double* sums,
                       float* centroids, float* losses, float* d_centroids, const slcl_peer_t* peer,
                       void* workspace, size_t workspace_bytes, slcl_stream_t stream);
int slcl_mccl_step_fwd_local(const float* feat_s, const int64_t* labels_s, int64_t batch_s, const float* feat_t,
                             const float* pred_t, const int32_t* part_id, int64_t batch_t, const float* feat_a,
                             const float* pred_a, int64_t batch_a, int64_t channels, int64_t pixels,
                             int n_partitions, int n_class, int flags, float threshold, double* sums,
                             void* workspace, size_t workspace_bytes, slcl_stream_t stream);
int slcl_mccl_step_finish(const double* sums, int has_aug, int64_t channels, int n_partitions, int n_class,
                          const float* previous_s, float momentum, int split, int bg, int norm, float inter_w,
                          float intra_w, float cnr_w, float* centroids, float* losses, float* d_centroids,
                          void* workspace, size_t workspace_bytes, slcl_stream_t stream);
int slcl_mccl_step_bwd(const float* feat_t, const float* pred_t, const int32_t* part_id, int64_t batch_t,
                       const float* feat_a, const float* pred_a, int64_t batch_a, int64_t channels,
                       int64_t pixels, int n_partitions, int n_class, int flags, float threshold,
                       const double* sums, const float* d_centroids, const float* grad_out, float* dfeat_t,
                       float* dpred_t, float* dfeat_a, float* dpred_a, void* workspace, size_t workspace_bytes,
                       slcl_stream_t stream);

/* ---------------------------------------------------------------------------
 * The MPSCL loss section (trainer/Trainer_MPSCL.py:133-147) in one call:
 *   centres = update_class_center_iter(feat_s, labels_s, old_centres, momentum)
 *   hard, mask = generate_pseudo_label(feat_t, centres, sel_threshold)
 *   loss_s = mpcl_loss_calc(feat_s, labels_s, centres, mpcl_src)
 *   loss_t = mpcl_loss_calc(feat_t, hard, centres, mpcl_trg, pixel_sel_loc=mask)
 * Both maps are dense NCHW with the same channels and pixels (batches may differ); params_s / params_t carry each
 * loss's constants, the same n_class in [2, 8], and normalize = 1.  scal_s / scal_t are the quadruples of
 * slcl_proto_fwd (loss, coefficient, weight sum, weighted row-loss sum); label_t / sel_t are the pseudo labels and mask.
 * slcl_mpscl_step_fwd: the class-sum sweep and reduce [+ exchange through `peer`, capacity_words >= 2 K (C+1)] + EMA of
 * slcl_class_centres_update, the unit centres, ONE prototype forward over both maps and ONE finaliser that exchanges
 * both loss pairs in one mailbox epoch: 5 launches; peer may be null.
 * slcl_mpscl_step_fwd_local (NCCL route, after the caller has the global centres): the same forward without the
 * exchange; pairs[4] = this rank's {w_s, l_s, w_t, l_t}.  Sum pairs over the ranks, then slcl_mpscl_step_finish.
 * slcl_mpscl_step_bwd: dfeat_s = grad_s[0] d loss_s / d feat_s and dfeat_t likewise, one launch over both maps; a null
 * grad_s or grad_t skips that map.  Each map's load width follows its own alignment; maps of different widths take
 * one launch each. */
size_t slcl_mpscl_step_workspace_bytes(const slcl_map_t* map_s, const slcl_map_t* map_t, int n_class);
int slcl_mpscl_step_fwd(const float* feat_s, const slcl_map_t* map_s, const int64_t* labels_s, const float* feat_t,
                        const slcl_map_t* map_t, const float* old_centres, float momentum,
                        const slcl_proto_params_t* params_s, const slcl_proto_params_t* params_t, float sel_threshold,
                        float* centres, float* cstate, float* stash_s, float* stash_t, int64_t* label_t, float* sel_t,
                        float* scal_s, float* scal_t, const slcl_peer_t* peer, void* workspace, size_t workspace_bytes,
                        slcl_stream_t stream);
int slcl_mpscl_step_fwd_local(const float* feat_s, const slcl_map_t* map_s, const int64_t* labels_s, const float* feat_t,
                              const slcl_map_t* map_t, const float* centres, const slcl_proto_params_t* params_s,
                              const slcl_proto_params_t* params_t, float sel_threshold, float* cstate, float* stash_s,
                              float* stash_t, int64_t* label_t, float* sel_t, float* pairs, void* workspace,
                              size_t workspace_bytes, slcl_stream_t stream);
int slcl_mpscl_step_finish(const float* pairs, float* scal_s, float* scal_t, slcl_stream_t stream);
int slcl_mpscl_step_bwd(const float* feat_s, const slcl_map_t* map_s, const float* feat_t, const slcl_map_t* map_t,
                        const float* stash_s, const float* stash_t, const float* cstate, const float* scal_s,
                        const float* scal_t, const float* grad_s, const float* grad_t, const slcl_proto_params_t* params_s,
                        const slcl_proto_params_t* params_t, float* dfeat_s, float* dfeat_t, slcl_stream_t stream);

/* ---------------------------------------------------------------------------
 * Sampler: per-class compaction + gather (north_star item 1).
 * slcl_compact_by_class: stable compaction of pixel indices by label, order
 * bit-identical to torch.nonzero(labels == k) for every k.  counts [K] int64,
 * offsets [K+1] int64 (exclusive scan), index [N] int64 (class-major).
 * slcl_gather_unit_rows: rows pixel_idx of an NCHW map -> [R, C] fp32 and/or
 * [R, bf16_row_stride] bf16 row-major (columns >= C zero-filled: the tensor-core
 * kernel wants a multiple of 64), L2-normalised (eps 1e-12) when `normalize`;
 * inv_norm [R] = 1/max(||x||, 1e-12) is written in both cases.
 * ------------------------------------------------------------------------- */
size_t slcl_compact_workspace_bytes(int64_t n_pixels, int n_class);
int slcl_compact_by_class(const int64_t* labels, int64_t n_pixels, int n_class,
                          int64_t* counts, int64_t* offsets, int64_t* index,
                          void* workspace, size_t workspace_bytes, slcl_stream_t stream);
/* Class-balanced two-phase pick of the sampler (SURVEY 8(c)-3) from ONE permutation `perm` [N] of the pixel indices
 * (torch.randperm) and the label map `labels` [N]: class k contributes its first `per` pixels in permutation order
 * (class-major output); slots a short class leaves open take the next unpicked labelled pixels in permutation order.
 * Two quotas at once (anchors / contrast rows; per_b = 0: one): out_q [n_class * per_q] pixel indices, filled_q [1] =
 * slots actually filled (< n_class * per_q: too few labelled pixels, the open slots hold 0).  No host synchronisation. */
size_t slcl_sample_balanced_workspace_bytes(int64_t n_pixels, int n_class);
int slcl_sample_balanced(const int64_t* perm, const int64_t* labels, int64_t n_pixels, int n_class,
                         int64_t per_a, int64_t* out_a, int64_t* filled_a,
                         int64_t per_b, int64_t* out_b, int64_t* filled_b,
                         void* workspace, size_t workspace_bytes, slcl_stream_t stream);
/* Self-pair maps of the analytic pixel<->pixel mode for ids in [0, n_ids) (pixel indices), unique within each side:
 * a_selfcol [A] = contrast row carrying anchor i's id or -1, b_selfrow [M] = its inverse.  row_of_id [2, n_ids] int32
 * (caller-owned) receives the two lookup tables they are read from: row_of_id[0][id] = anchor row holding id or -1,
 * row_of_id[1][id] = contrast row -- for pixel ids exactly the maps slcl_scatter_rows_by_map wants. */
int slcl_self_maps(const int64_t* id_a, int64_t n_anchor, const int64_t* id_b, int64_t n_contrast, int64_t n_ids,
                   int32_t* a_selfcol, int32_t* b_selfrow, int32_t* row_of_id, slcl_stream_t stream);
/* Backward of slcl_gather_unit_rows driven from the pixel side (same arithmetic as slcl_scatter_rows_bwd): row_of_pixel_s
 * [batch * pixels] int32 = the row of set s gathered from that pixel, or -1; every element of dfeat is WRITTEN (zeros
 * where no row holds the pixel), coalesced, without atomics -- the faster route when the rows cover a good share of
 * the map.  Set b is optional (all three pointers null); the two sets are summed. */
int slcl_scatter_rows_by_map(const float* feat, int64_t batch, int64_t channels, int64_t pixels, int normalize,
                             const int32_t* row_of_pixel_a, const float* d_rows_a, const float* inv_norm_a,
                             const int32_t* row_of_pixel_b, const float* d_rows_b, const float* inv_norm_b,
                             float* dfeat, slcl_stream_t stream);
/* {label, id} rows of slcl_p2p_fwd straight from the label map: meta [pad64(R), 2] int32 = {labels[idx[r]], idx[r]},
 * pad rows {INT_MIN, INT_MIN}.  n_pixels <= INT_MAX. */
int slcl_rows_meta(const int64_t* labels, int64_t n_pixels, const int64_t* pixel_idx, int64_t n_rows, int32_t* meta,
                   slcl_stream_t stream);
/* Row weights of the SupCon family from the metadata rows (label != 0 = foreground): the rows are n_tiles equal tiles
 * of rows_per_tile rows; weight[r] = fg_r / (foreground rows of r's tile) / (tiles that have foreground) --
 * utils/loss.py:382-384 for one problem (n_tiles = 1), :445-448 folded into the rows for BlockConLoss.  zero_if_empty:
 * tiles (or a whole problem) without foreground weigh 0 (:405-407, :439-440); otherwise 0/0 stays NaN as in SupConLoss.
 * tile_fg [n_tiles] fp32 receives the per-tile foreground counts. */
int slcl_tile_weights(const int32_t* meta, int64_t n_tiles, int64_t rows_per_tile, int zero_if_empty, float* tile_fg,
                      float* weight, slcl_stream_t stream);
int slcl_gather_unit_rows(const float* feat, int64_t batch, int64_t channels, int64_t pixels,
                          const int64_t* pixel_idx, int64_t n_rows, int normalize,
                          void* rows_bf16, int64_t bf16_row_stride, float* rows_f32, float* inv_norm,
                          slcl_stream_t stream);
/* exp shift for un-normalised rows (SupConLoss does not normalise, utils/loss.py:342-349):
 * shift[i] = |a_i| * max_j |b_j| / temperature, from the inv_norm outputs of slcl_gather_unit_rows.
 * n_contrast <= 2^20 (SLCL_ERR_UNSUPPORTED beyond). */
int slcl_p2p_shift(const float* inv_norm_a, int64_t n_anchor, const float* inv_norm_b, int64_t n_contrast,
                   float temperature, float* shift, slcl_stream_t stream);
/* scatter-add of row gradients back into an NCHW gradient map, through the
 * normalisation backward: dx = (g - xhat (xhat.g)) * inv_norm. */
int slcl_scatter_rows_bwd(const float* feat, int64_t batch, int64_t channels, int64_t pixels,
                          const int64_t* pixel_idx, int64_t n_rows, int normalize,
                          const float* d_rows, const float* inv_norm, float* dfeat, slcl_stream_t stream);

/* ---------------------------------------------------------------------------
 * Segmentation losses on the logits (SURVEY.md 8(f)-2): loss_calc (utils/loss.py:46-66: CrossEntropyLoss
 * [+ jaccard_loss :11-43]) and dice_loss (:69-103) in ONE pass over logits [B,K,HW] fp32 + labels [B,HW]
 * int64, and their fused backward.  K >= 2 (the reference's num_classes == 1 sigmoid branch is not built).
 *   stats  [B,K,4] fp32 = per (image, class) {sum p*g, sum p*p, sum g, sum p}
 *   losses [3]     fp32 = {cross entropy (mean over pixels), dice, jaccard}
 *   backward: grad_losses [3] device fp32 = d/d{ce, dice, jaccard}; dlogits [B,K,HW].
 * slcl_entropy_map: prob_2_entropy (utils/utils_.py:627-631), out = -p log2(p+1e-7)/log2(K) and/or its
 * backward dprob = grad_out * d out / d p (either output pointer may be null).
 * ------------------------------------------------------------------------- */
size_t slcl_seg_workspace_bytes(int64_t batch, int64_t pixels, int n_class);
int slcl_seg_fwd(const float* logits, const int64_t* labels, int64_t batch, int n_class, int64_t pixels,
                 float* stats, float* losses, void* workspace, size_t workspace_bytes, slcl_stream_t stream);
int slcl_seg_bwd(const float* logits, const int64_t* labels, int64_t batch, int n_class, int64_t pixels,
                 const float* stats, const float* grad_losses, float* dlogits, slcl_stream_t stream);
/* The same losses over the global batch of data-parallel ranks (utils/loss.py:11-103 on the ranks' batches
 * concatenated in rank order; ranks may hold different B, H W and K must agree).  Each rank reduces its batch into
 *   vec [2K+4] fp64 = {inter_k (K), card_k (K), n_valid, sum ce, sum dice_bk over its images, n_images}
 * which is a sum over ranks.  slcl_seg_fwd_peer all-reduces it inside its finaliser through the peer mailboxes (rank
 * order: identical bits on every rank; capacity_words >= 2 (2K+4)) and writes the GLOBAL vec and losses; a peer that
 * times out makes both NaN.  slcl_seg_fwd_local writes this rank's vec (the caller sums it over the ranks, e.g. NCCL)
 * and slcl_seg_finish turns a summed vec into losses with the same arithmetic.  stats stays per local image.
 * slcl_seg_bwd_global: this rank's dlogits of the global losses, from its stats and the global vec (no exchange). */
int slcl_seg_fwd_peer(const float* logits, const int64_t* labels, int64_t batch, int n_class, int64_t pixels,
                      float* stats, double* vec, float* losses, const slcl_peer_t* peer,
                      void* workspace, size_t workspace_bytes, slcl_stream_t stream);
int slcl_seg_fwd_local(const float* logits, const int64_t* labels, int64_t batch, int n_class, int64_t pixels,
                       float* stats, double* vec, void* workspace, size_t workspace_bytes, slcl_stream_t stream);
int slcl_seg_finish(const double* vec, int n_class, float* losses, slcl_stream_t stream);
int slcl_seg_bwd_global(const float* logits, const int64_t* labels, int64_t batch, int n_class, int64_t pixels,
                        const float* stats, const double* vec, const float* grad_losses, float* dlogits,
                        slcl_stream_t stream);
int slcl_entropy_map(const float* prob, int64_t n_elems, int n_class, float* out, const float* grad_out,
                     float* dprob, slcl_stream_t stream);
/* prob_2_entropy (utils/utils_.py:627-631) of softmax(logits, 1), the map of trainer/Trainer_MPSCL.py:171-172, from
 * logits [B,K,HW] fp32 in one pass: p = softmax_k(z) (the seg losses' softmax), out = -p log2(p+1e-7)/log2(K) with
 * slcl_entropy_map's arithmetic.  With grad_out and dlogits [B,K,HW] (= d/d out): dlogits = p (t - sum_m p_m t_m),
 * t = grad_out * d out / d p, p recomputed from the logits.  out, the pair (grad_out, dlogits), or both; 2 <= K <= 8. */
int slcl_entropy_map_logits(const float* logits, int64_t batch, int n_class, int64_t pixels, float* out,
                            const float* grad_out, float* dlogits, slcl_stream_t stream);

/* ---------------------------------------------------------------------------
 * Pixel <-> pixel supervised contrastive loss (SupConLoss.forward,
 * utils/loss.py:327-387 = utils/losses.py:106-161, and its autograd backward;
 * rectangular anchors x contrast-rows generalisation of SURVEY.md 8(c)-3).
 * a [A, dp] anchors and b [M, dp] contrast rows: bf16 row-major, dp = dim_padded,
 * a multiple of 64 <= 256 (pad columns zero).  Similarities S = a b^T / T run on
 * tcgen05 tensor cores with fp32 TMEM accumulation; S is never written to memory.
 *   a_meta / b_meta: int32 pairs {label, id} per row, each array PADDED to a multiple of 64
 *     entries with {INT_MIN, INT_MIN} (the kernel fetches whole 64-entry tiles with bulk
 *     copies), 16-byte aligned.  Pairs with equal id are the
 *     self pairs (excluded, :365-371); pairs with equal label and different id are the
 *     positives (:352-354,:368).  Unlabelled mode (:359-361): pass the pixel index
 *     within the view as "label".
 *   shift  [A] fp32: any upper bound of S_ij over j (e.g. ||a_i|| max_j||b_j|| / T);
 *     exponentials are evaluated as exp(S - shift), the result is shift-invariant.
 *   weight [A] fp32: w_i of the final reduction (fg_i / sum fg, :382-384, or 1/A).
 *   n_class: 0 = general labels (any int32; positives are tested per element from the labels; self pairs are found by
 *     comparing ids per element, or -- when a_selfcol / b_selfrow are given (unique ids) -- treated as ordinary pairs in
 *     the sweeps and removed afterwards; warps whose 32 columns carry one label then skip all per-element integer work,
 *     so sorting the contrast rows by label pays).  bwd_state must be null.
 *     1..8 = "analytic" mode for class-index labels in [0, n_class) and UNIQUE ids, weights >= 0: the
 *     positive-pair terms are rank-n_class and are evaluated outside the tensor-core sweeps from per-class row
 *     sums, the self pair is removed afterwards with one dot product per anchor.  An anchor whose label is outside
 *     [0, n_class) has no class table: its row loss is 0/0 and the returned loss is NaN (whatever its weight).
 *     The ids inside the meta arrays are then unused; instead
 *       a_selfcol [A] int32: the contrast row holding anchor i's own pixel, or -1 (null: no anchor is a contrast row)
 *       b_selfrow [M] int32: its inverse (anchor whose pixel contrast row j is, or -1); both or none.
 *       bwd_state: optional caller-owned buffer of slcl_p2p_state_bytes() bytes (16-byte aligned) that the forward
 *         fills with what the backward can reuse -- the column-split partials of U_i = sum_j exp(S_ij - shift_i) b_j
 *         exactly as the sweep wrote them (the backward finish sums them and removes the self pair), the per-class row
 *         sums of both sides and the per-anchor constants.  Handing it back to slcl_p2p_bwd leaves the backward with
 *         ONE tensor-core sweep (dB) and one finishing kernel; with null the backward regenerates it (one more sweep).
 *     The per-class sums of the contrast rows, and beta~_i = w_i / (T n_i) with the class sums ABsum of the anchors
 *     (labels and weights only), do not depend on the sweep: they run on a side stream owned by the library (one per
 *     host thread and device, created on first use; fork/join by events, graph-capturable).  The forward on the
 *     caller's stream is the sweep plus ONE finishing launch (its last block totals the loss).
 *   n_batch: 1, or the number of equal BLOCK-DIAGONAL batches (either mode; the analytic mode keeps one table of
 *     per-class sums per batch): anchors [z A/n, (z+1) A/n) are
 *     contrasted with contrast rows [z M/n, (z+1) M/n) only -- BlockConLoss (utils/loss.py:416-466) as ONE launch per
 *     sweep instead of div_num^2 separate problems.  A/n and M/n must be multiples of 128.
 * Sizes: A and M below INT_MAX - 128 in either mode (row indices are 32-bit); every finishing and reduction stage
 * grid-strides or sizes its partials from A, so no other row bound applies.  The workspace and the kept state grow
 * linearly with A (U partials and dA split partials: about 4 A dp bytes each per column split).
 * forward : stats [A,3] = {sum_j exp(S_ij - shift_i), sum_pos S_ij * T, #pos},
 *           loss [1] = sum_i w_i (shift_i + log stats_i0 - stats_i1/(T stats_i2)).
 * backward: d_a [A, dim] and/or d_b [M, dim] fp32 = dL/da, dL/db for dL/dloss = *grad_out
 *           (either pointer may be null).
 * ------------------------------------------------------------------------- */
size_t slcl_p2p_workspace_bytes(int64_t n_anchor, int64_t n_contrast, int64_t dim_padded);
size_t slcl_p2p_state_bytes(int64_t n_anchor, int64_t dim_padded);
int slcl_p2p_fwd(const void* a_bf16, const void* b_bf16, int64_t n_anchor, int64_t n_contrast, int64_t dim_padded,
                 const int32_t* a_meta, const int32_t* b_meta, const int32_t* a_selfcol, int n_class, int n_batch,
                 const float* shift, const float* weight, float temperature, float* stats, float* loss,
                 void* bwd_state, void* workspace, size_t workspace_bytes, slcl_stream_t stream);
int slcl_p2p_bwd(const void* a_bf16, const void* b_bf16, int64_t n_anchor, int64_t n_contrast, int64_t dim_padded,
                 int64_t dim, const int32_t* a_meta, const int32_t* b_meta, const int32_t* a_selfcol,
                 const int32_t* b_selfrow, int n_class, int n_batch, const float* shift, const float* weight,
                 float temperature, const float* stats, const void* bwd_state, const float* grad_out, float* d_a, float* d_b,
                 void* workspace, size_t workspace_bytes, slcl_stream_t stream);

/* ---------------------------------------------------------------------------
 * Pixel <-> pixel losses over the GLOBAL batch of data-parallel ranks (SURVEY.md 8(e); the `group=` argument of
 * SupConLoss / LocalConLoss / sampled_supcon_loss).  Each rank sweeps its own anchors against the contrast rows of all
 * ranks (slcl_p2p_fwd, d_a of slcl_p2p_bwd), and the anchors of all ranks against its own contrast rows (d_b of
 * slcl_p2p_bwd), so per-rank tensor work is 8 A_local M_global d flop and nothing is computed twice.
 *
 * slcl_peer_allgather: every rank contributes a record of n_bytes (multiple of 16, <= slot_bytes) and receives all ranks'
 * records in rank order in out [world * n_bytes] -- a private buffer no later call touches.  Replaces the NCCL
 * all_gather_into_tensor of the same records.  regions_dev: device array of `world` pointers to the ranks' row regions of
 * slcl_peer_rows_region_bytes(slot_bytes) bytes each (zero-initialised, mapped by every rank like the mailboxes); the call
 * is one exchange of the mailbox sequence of `peer` (same epochs, same time-out).  The first 16 bytes of a record are its
 * key (sizes / shapes) and must be equal on every rank.  status [1] int32, in/out: bit 0 = a peer timed out (mailbox word 1
 * counts it), bit 1 = a peer's key differs (mailbox word 5 counts it).  With a non-zero status on entry (an earlier
 * exchange of the same result failed) or after a time-out waiting for a free slot, the call publishes nothing and waits
 * for nobody, so the peers time out too and every rank's result is NaN; it still reads the peers' slots and acks them.
 * Out is then undefined but never read past a slot.  The calls may interleave with the other exchanges of the mailbox in
 * any order.
 * ------------------------------------------------------------------------- */
size_t slcl_peer_rows_region_bytes(int64_t slot_bytes);
int slcl_peer_allgather(const void* record, int64_t n_bytes, void* out, int32_t* status, const slcl_peer_t* peer,
                        const void* regions_dev, int64_t slot_bytes, slcl_stream_t stream);
/* Byte offsets inside the analytic backward state of slcl_p2p_state_bytes(n_anchor, dim_padded):
 * offsets_host[7] = {U partials, Bsum, ABsum [K][d+1] fp32, colshift [pad64(A)] fp32, alpha~ [A] fp32, beta~ [A] fp32, total}.
 * Lets a data-parallel caller read a rank's per-anchor constants and ABsum table out of its forward state. */
int slcl_p2p_state_layout(int64_t n_anchor, int64_t dim_padded, int64_t* offsets_host);
/* Backward state for slcl_p2p_bwd(d_b only) over the anchors of all ranks, built from what each rank's forward left:
 * alpha / beta / colshift [n_anchor] fp32 = the ranks' per-anchor constants concatenated in rank order, absum_parts
 * [n_parts][n_class][dim_padded + 1] fp32 = the ranks' ABsum tables (summed in rank order).  Replaces the state a forward
 * over all anchors would have left (U, Bsum: not read by the d_b backward, left unset). */
int slcl_p2p_state_assemble(void* bwd_state, int64_t n_anchor, int64_t dim_padded, int n_class, const float* alpha,
                            const float* beta, const float* colshift, const float* absum_parts, int n_parts,
                            slcl_stream_t stream);
/* The same for n_batch block-diagonal batches (the d_b backward of a block-diagonal problem, BlockConLoss(group=)):
 * alpha / beta / colshift [n_anchor] are already in the global batch-major order the d_b sweep reads, and absum_parts is
 * [n_parts][n_batch][n_class][dim_padded + 1] (one ABsum table per batch and rank, summed in rank order).  n_batch > 1
 * needs n_anchor / n_batch a multiple of 128, as slcl_p2p_bwd does.  slcl_p2p_state_assemble is the n_batch = 1 case. */
int slcl_p2p_state_assemble_batched(void* bwd_state, int64_t n_anchor, int64_t dim_padded, int n_class, int n_batch,
                                    const float* alpha, const float* beta, const float* colshift, const float* absum_parts,
                                    int n_parts, slcl_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif  /* SLCL_H_ */
