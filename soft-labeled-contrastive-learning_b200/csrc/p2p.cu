// p2p.cu -- pixel <-> pixel supervised contrastive loss on the 5th-gen tensor cores.
//
// Replaces (reference, file:line):
//   SupConLoss.forward   utils/loss.py:327-387 (= utils/losses.py:106-161): the M x M Gram matrix
//                        via conv2d (:342-349), >= 6 materialised M x M fp32 temporaries (:352-380)
//   and its autograd backward (SURVEY.md appendix A.6), generalised to anchors x contrast rows
//   (SURVEY.md 8(c)-3).
//
// Roofline: tensor core.  Flash-attention style: the similarity matrix never exists in memory.
//   One CTA owns a 128-row tile of the "row operand" R (resident in TENSOR MEMORY as the A operand of
//   MMA1) and streams 64-row tiles of the "column operand" Cm through a TMA ring in shared memory.
//     MMA1 (tcgen05.mma, bf16 -> fp32 TMEM):  S[128 x 64] = R_tile . Cm_tile^T        (K = d)
//     epilogue warps (tcgen05.ld, one thread per row): exp2 of the scaled, shifted similarities ->
//       row sums (forward) and/or the bf16 tile G, written back INTO TENSOR MEMORY over the S columns it
//       was computed from (tcgen05.st)
//     MMA2:  D[128 x d] += G[128 x 64] . Cm_tile[64 x d]   (A = G from tensor memory, B = the Cm tile
//       re-read from shared memory as an MN-major operand; accumulators stay in TMEM for the whole sweep)
//   S is double-buffered in TMEM so MMA1 of tile t+1 overlaps the epilogue of tile t.
//
// Two families of sweeps share the kernel (template parameter MODE):
//   * "analytic" (labels are class indices 0..K-1, K <= 8; ids unique): the positive-pair terms of loss and
//     gradient are rank-K and are taken OUT of the sweep --
//         sum_{j in pos(i)} S_ij = a_i . Bsum[lab_i] - [self]            Bsum[k] = sum_{lab_j = k} b_j
//         dA_i = alpha_i U_i - beta_i (Bsum[lab_i] - [self] b_self)      U_i = sum_j e_ij b_j
//         dB_j = sum_i alpha_i e_ij a_i - ABsum[lab_j] + [self] ...      ABsum[k] = sum_{lab_i = k} beta_i a_i
//     so the epilogue is FFMA + EX2 (+ FADD) per element with no integer work, the forward sweep also
//     produces U (its MMA2), and the whole backward is ONE more sweep (dB).  Tensor work = 8 A M d flop,
//     exactly the algorithmic count (S is formed twice, not three times).
//   * "general" (arbitrary integer labels, e.g. the unlabelled SupCon mode where the label is the pixel
//     position): self pairs and positives are decided per element from {label, id} pairs.
#include "common.cuh"

#include <cuda.h>
#include <cuda_bf16.h>
#include <limits.h>
#include <algorithm>
#include <type_traits>
#include <stdlib.h>
#include <math.h>

namespace slcl {
namespace {

constexpr int BM = 128;            // rows per CTA (UMMA M)
constexpr int BN = 64;             // streamed rows (S tile columns) per step
constexpr int KCH = 64;            // bf16 elements per 128-byte swizzle row
constexpr int kStages = 6;
constexpr int kMaxD = 256;
constexpr int kEpiWarps = 8;       // warps 4..11; (warp % 4) selects the TMEM lane quarter
constexpr int kThreads = 32 * (4 + kEpiWarps);
constexpr int kTmemCols = 512;
constexpr int kColS = 0;           // S double buffer: columns [0,64) and [64,128); G(t) overwrites S(t) in place
constexpr int kColAcc = 128;       // MMA2 accumulators: columns [128, 128 + d)
constexpr int kColR = 384;         // resident row operand R (bf16 pairs): columns [384, 384 + d/2)
constexpr float kLog2e = 1.4426950408889634f;
constexpr int kMaxLabelClasses = 8;     // analytic sweeps: labels in [0, K), K <= 8
constexpr float kShiftOff = 1.0e30f;    // column shift that switches a column off (exp2(-1e30) = 0)

#ifdef SLCL_P2P_PROFILE
constexpr bool kProfile = true;
#else
constexpr bool kProfile = false;
#endif

enum Mode {
  kGenFwd = 0,    // general: row statistics {Zs, P_raw, n} with per-element {label, id} tests
  kGenRows = 1,   // general: dA sweep, statistics per row
  kGenCols = 2,   // general: dB sweep, statistics per column
  kAnaFwd = 3,    // analytic: row sums of exp only
  kAnaFwdU = 4,   // analytic: row sums of exp + U = E . B (MMA2)
  kAnaCols = 5    // analytic: dB sweep, G = exp2(s * scale - colshift)  (alpha folded into the shift)
};
template <int MODE> struct ModeTraits {
  static constexpr bool kMma2 = MODE == kGenRows || MODE == kGenCols || MODE == kAnaFwdU || MODE == kAnaCols;
  static constexpr bool kRowSums = MODE == kGenFwd || MODE == kAnaFwd || MODE == kAnaFwdU;
  static constexpr bool kColRing = MODE == kGenFwd || MODE == kGenRows || MODE == kGenCols || MODE == kAnaCols;
  static constexpr int kStatN = MODE == kGenFwd ? 3 : 1;      // floats per row and slot in stat_partial
};

struct P2PArgs {
  int n_rows, n_cols, d;              // d padded to a multiple of 64
  int cols_per_split;                 // CTA (x, y) sweeps columns [y * cols_per_split, ...)
  int rows_per_batch, cols_per_batch; // block-diagonal batches (grid.z): batch z contrasts rows [z rpb, (z+1) rpb) with columns
                                      // [z cpb, (z+1) cpb) only; rpb % 128 == 0 and cpb % 64 == 0.  One batch: the whole problem.
  float scale_log2;                   // log2(e) / T
  int self_by_id;                     // general modes: 1 = self pairs found by comparing ids per element; 0 = the caller gave
                                      // self maps (unique ids): the sweep treats them as ordinary pairs, they are removed afterwards
  const uint32_t* rows_u32;           // resident operand, bf16 row-major [n_rows, d] viewed as 32-bit words
  const int2* row_meta;               // general modes: {label, id}
  const int2* col_meta;
  const float* row_shift;             // kGenFwd / kAnaFwd / kAnaFwdU: shift [n_rows] in natural-log units
  const float4* row_stat;             // kGenRows: {shift*log2e, alpha, beta, -}
  const float4* col_stat;             // kGenCols: {shift*log2e, alpha, beta, -}, padded to 64 entries
  const float* col_shift;             // kAnaCols: shift*log2e - log2(alpha) per column, padded to 64 entries
  float* stat_partial;                // row sums: [n_slots][n_rows][kStatN]
  float* grad_partial;                // MMA2 modes: [n_splits][n_rows][d] fp32
  float* fused_out;                   // dB sweeps with one split: d_b [n_rows][ld_out] written by the drain itself (else null);
                                      // kAnaCols also folds in:
  int ld_out;                         //   out = g (Acc - ABsum[label of the row]);  ab_sums [K][d+1], row labels = row_meta
  int n_class;
  const float* ab_sums;
  const float* grad_out;
  unsigned long long* prof;           // bring-up: per-role wait-cycle counters of CTA (0,0), or null
};

// --------------------------- PTX wrappers ----------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "WAIT_LOOP:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra WAIT_DONE;\n\t"
      "bra WAIT_LOOP;\n\t"
      "WAIT_DONE:\n\t"
      "}\n" ::"r"(smem_u32(bar)), "r"(parity)
      : "memory");
}
// Bring-up instrumentation (per-role barrier-wait cycle counters, read by tools/p2p_prof.py) is compiled
// in only with -DSLCL_P2P_PROFILE; the shipped library waits without touching the clock.
#ifdef SLCL_P2P_PROFILE
__device__ __forceinline__ void mbar_wait_t(uint64_t* bar, uint32_t parity, unsigned long long& acc) {
  const long long t0 = clock64();
  mbar_wait(bar, parity);
  acc += (unsigned long long)(clock64() - t0);
}
#define SLCL_PROF_NOW() clock64()
#else
__device__ __forceinline__ void mbar_wait_t(uint64_t* bar, uint32_t parity, unsigned long long&) { mbar_wait(bar, parity); }
#define SLCL_PROF_NOW() 0ll
#endif
// one lane of a converged warp (elect.sync): the idiom the compiler recognises for single-thread
// issue of uniform-datapath instructions
__device__ __forceinline__ bool elect_one() {
  uint32_t pred = 0;
  asm volatile(
      "{\n\t"
      ".reg .pred px;\n\t"
      "elect.sync _|px, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, px;\n\t"
      "}\n"
      : "=r"(pred));
  return pred != 0;
}
// (pdl_trigger / pdl_wait / launch_pdl: common.cuh -- every p2p kernel uses programmatic dependent launch)
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(
          smem_u32(smem_dst)),
      "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}
// same, multicast: the box lands at the same CTA-relative offset (and signals the same CTA-relative
// mbarrier) in every CTA of `mask`
__device__ __forceinline__ void tma_load_2d_mc(void* smem_dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1,
                                               uint16_t mask) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster [%0], [%1, {%3, %4}], "
      "[%2], %5;" ::"r"(smem_u32(smem_dst)),
      "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "h"(mask)
      : "memory");
}
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// 1-D bulk copy global -> shared, completion on an mbarrier (bytes % 16 == 0, 16-byte aligned)
__device__ __forceinline__ void bulk_load_1d(void* smem_dst, const void* gsrc, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                   smem_u32(smem_dst)),
               "l"(reinterpret_cast<uint64_t>(gsrc)), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
// TMA store of a 3-D box shared -> global (bulk async-group completion)
__device__ __forceinline__ void tma_store_3d(const CUtensorMap* map, const void* smem_src, int c0, int c1, int c2) {
  asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%2, %3, %4}], [%1];" ::"l"(
                   reinterpret_cast<uint64_t>(map)),
               "r"(smem_u32(smem_src)), "r"(c0), "r"(c1), "r"(c2)
               : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory"); }
__device__ __forceinline__ void bulk_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* map) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(map)) : "memory");
}

__device__ __forceinline__ void tmem_alloc(uint32_t* smem_dst, uint32_t cols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)), "r"(cols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t addr, uint32_t cols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(addr), "r"(cols) : "memory");
}
// D[tmem] (+)= A[tmem] * B[smem desc]; issued by ONE thread.  The A operand is read from tensor memory (rows = lanes,
// bf16 pairs packed along K in 32-bit columns): no per-instruction shared-memory fetch of the 128 A rows, so a narrow-N
// MMA runs at its N/2-cycle floor
__device__ __forceinline__ void umma_bf16_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t"
      "}\n" ::"r"(tmem_d),
      "r"(tmem_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// arrives on the mbarrier once every previously issued tcgen05.mma of this thread has completed
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// same, arriving on the barrier at this CTA-relative offset in every CTA of `mask`
__device__ __forceinline__ void umma_commit_mc(uint64_t* bar, uint16_t mask) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
                   smem_u32(bar)),
               "h"(mask)
               : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
        "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
        "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_st32(uint32_t taddr, const uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
      "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};" ::"r"(taddr),
      "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]), "r"(v[9]),
      "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15]), "r"(v[16]), "r"(v[17]), "r"(v[18]),
      "r"(v[19]), "r"(v[20]), "r"(v[21]), "r"(v[22]), "r"(v[23]), "r"(v[24]), "r"(v[25]), "r"(v[26]), "r"(v[27]),
      "r"(v[28]), "r"(v[29]), "r"(v[30]), "r"(v[31])
      : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ float ex2_approx(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// Shared-memory matrix descriptor (SM100 UMMA), 128-byte swizzle.
//   bits [0,14)  start address >> 4      bits [16,30) leading byte offset >> 4
//   bits [32,46) stride byte offset >> 4 bits [46,48) version = 1     bits [61,64) layout = 2 (SWIZZLE_128B)
__device__ __forceinline__ uint64_t make_desc(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr >> 4) & 0x3FFF);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}
// Instruction descriptor, kind::f16: D fp32, A/B bf16, M = 128.
//   [4,6) c_format = 1 (F32)  [7,10) a_format = 1 (BF16)  [10,13) b_format = 1 (BF16)
//   [15] a_major (0 = K)  [16] b_major (0 = K, 1 = MN)  [17,23) N >> 3  [24,29) M >> 4
__device__ __forceinline__ uint32_t make_idesc(int n, int b_mn_major) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)b_mn_major << 16) | ((uint32_t)(n >> 3) << 17) |
         ((uint32_t)(BM >> 4) << 24);
}

__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};" ::"r"(taddr),
      "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]), "r"(v[9]),
      "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15])
      : "memory");
}
__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
  __nv_bfloat162 h = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&h);
}

// Column metadata of one 64-column tile.  The TMA producer brings it in with 1-D bulk copies into a
// kMetaSlots-deep ring of its own (the epilogue reads it after the tile's smem stage has already been
// handed back), so the epilogue warps never issue a global load.  The caller pads the metadata arrays
// to a multiple of 64 entries; pad entries carry id INT_MIN (masked) / shift kShiftOff.
// Column metadata reads by 32-bit SHARED address: the carve-up below goes through generic pointer arithmetic, and a plain
// C++ dereference of it compiles to a generic LD.E (address translation + long scoreboard) instead of LDS -- found in
// round 2 with cuobjdump (64-72 LD.E per epilogue instantiation, most of them inside the per-tile loop).
__device__ __forceinline__ int2 lds_int2(uint32_t addr) {
  int2 v;
  asm volatile("ld.shared.v2.s32 {%0, %1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(addr));
  return v;
}
__device__ __forceinline__ float4 lds_float4(uint32_t addr) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
  return v;
}
constexpr int kMetaSlots = 4;
struct __align__(128) ColMeta {
  float4 stat[BN];      // kGenCols: {shift*log2e, alpha, beta, -};  kAnaCols: the first 64 floats = column shifts
  int2 meta[BN];        // general modes: {label, id}
};

struct __align__(8) Barriers {
  uint64_t r_in, r_full;
  uint64_t c_full[kStages], c_empty[kStages];
  uint64_t s_full[2], s_empty[2];
  uint64_t g_full[2];
  uint64_t acc_full;
  uint64_t m_full[kMetaSlots], m_empty[kMetaSlots];
  uint32_t tmem_base;
};

// dynamic smem carve-up (1024-byte aligned tiles); R and G live in tensor memory
//   Cm  : [kStages][d/64][64 rows][128 B]
//   after the sweep the ring doubles as the drain's staging area: 8 warps x 2 x 4 KB
constexpr size_t kDrainBytes = 8 * 2 * 4096;
constexpr size_t kTableBytes = (size_t)kMaxLabelClasses * kMaxD * sizeof(float);      // fused dB drain: ABsum [K][d]
__host__ __device__ inline size_t ring_bytes_for(int d) {
  const size_t ring = (size_t)kStages * (d / KCH) * BN * 128;
  return ring > kDrainBytes ? ring : kDrainBytes;
}
__host__ __device__ inline size_t smem_bytes_for(int d) {
  return 1024 /*align slack*/ + ring_bytes_for(d) + kMetaSlots * sizeof(ColMeta) + kTableBytes + sizeof(Barriers) + 64;
}

// CS = thread-block-cluster size along the row-tile axis.  The CS CTAs of a cluster sweep the same
// column tiles in lock step: each one fetches 1/CS of every column tile and TMA-multicasts it to all,
// so the L2 -> SM traffic of the streamed operand drops CS-fold.
template <int CS, int MODE>
__global__ void __launch_bounds__(kThreads, 1)
p2p_kernel(const __grid_constant__ CUtensorMap map_rows, const __grid_constant__ CUtensorMap map_cols,
           const __grid_constant__ CUtensorMap map_out, const P2PArgs a) {
  using MT = ModeTraits<MODE>;
  extern __shared__ uint8_t smem_raw[];
  const int kc = a.d / KCH;
  uint8_t* base = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint8_t* sC = base;
  ColMeta* sMeta = reinterpret_cast<ColMeta*>(sC + ring_bytes_for(a.d));
  float* sTab = reinterpret_cast<float*>(sMeta + kMetaSlots);
  Barriers* bars = reinterpret_cast<Barriers*>(reinterpret_cast<uint8_t*>(sTab) + kTableBytes);

  const long long t_entry = SLCL_PROF_NOW();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int batch = blockIdx.z;
  const int row0 = batch * a.rows_per_batch + blockIdx.x * BM;
  const int row_end = min(a.n_rows, (batch + 1) * a.rows_per_batch);
  const int split = blockIdx.y;
  const int col0 = batch * a.cols_per_batch + split * a.cols_per_split;
  const int col_end = min(min(a.n_cols, (batch + 1) * a.cols_per_batch), col0 + a.cols_per_split);
  const int n_tiles = (col_end - col0 + BN - 1) / BN;
  // Every CTA sweeps the same column tiles; start each one at a different tile so the CTAs do not
  // all hit the same L2 lines at the same moment (the sums do not depend on the sweep order).
  const int rot = (int)(((blockIdx.x / CS) * 37u + blockIdx.y * 11u + blockIdx.z * 5u) % (unsigned)n_tiles);
  const uint32_t crank = (CS > 1) ? cluster_ctarank() : 0u;
  constexpr uint16_t kAllCtas = (uint16_t)((1u << CS) - 1u);
  auto tile_col = [&](int t) { int tt = t + rot; if (tt >= n_tiles) tt -= n_tiles; return col0 + tt * BN; };

  if (threadIdx.x == 0) {
    tma_prefetch_desc(&map_rows);
    tma_prefetch_desc(&map_cols);
    mbar_init(&bars->r_in, 1);                   // R tile landed in its staging stages (TMA)
    mbar_init(&bars->r_full, 4);                 // the four warps that move R's lane quarters into tensor memory
    for (int s = 0; s < kStages; ++s) { mbar_init(&bars->c_full[s], 1); mbar_init(&bars->c_empty[s], CS); }
    for (int s = 0; s < 2; ++s) {
      mbar_init(&bars->s_full[s], 1);
      mbar_init(&bars->s_empty[s], kEpiWarps);
      mbar_init(&bars->g_full[s], kEpiWarps);
    }
    mbar_init(&bars->acc_full, 1);
    for (int s = 0; s < kMetaSlots; ++s) { mbar_init(&bars->m_full[s], 1); mbar_init(&bars->m_empty[s], kEpiWarps); }
    fence_barrier_init();
  }
  if (warp == 2) tmem_alloc(&bars->tmem_base, kTmemCols);
  tc_fence_before();
  __syncthreads();
  if (CS > 1) cluster_sync_all();          // every CTA's barriers exist before any multicast / remote arrive
  tc_fence_after();
  const uint32_t tmem = bars->tmem_base;
  const long long t_setup = SLCL_PROF_NOW();
  pdl_trigger();
  pdl_wait();                              // nothing above reads or writes global memory
  const long long t_pdl = SLCL_PROF_NOW();

  // Producer and MMA roles run with the WHOLE warp in the loop (converged, warp-uniform control flow) and
  // elect one lane only around the asynchronous instructions.  Running them under `if (lane == 0)` makes
  // the compiler wrap every UTCHMMA / UTMALDG in an ELECT + R2UR waterfall loop (~100 cycles per MMA).
  if (warp == 0) {
    // ===================== TMA producer =====================
    unsigned long long w0 = 0, w1 = 0;
    const long long tstart = SLCL_PROF_NOW();
    // The resident operand R comes in first, staged in the last two ring stages (128 rows = two 64-row stages);
    // the ring starts with the other stages and takes these two over once R sits in tensor memory.
    if (elect_one()) {
      mbar_expect_tx(&bars->r_in, (uint32_t)kc * BM * 128);
      uint8_t* rdst = sC + (size_t)(kStages - 2) * kc * BN * 128;
      for (int c = 0; c < kc; ++c) tma_load_2d(rdst + (size_t)c * BM * 128, &map_rows, &bars->r_in, c * KCH, row0);
    }
    __syncwarp();
    for (int t = 0; t < n_tiles; ++t) {
      const int s = t % kStages;
      const int ms = t % kMetaSlots;
      // the two staging stages start "full" (of R): their first hand-over is a real phase, signalled by the MMA
      // warp of every CTA of the cluster once R sits in tensor memory, so their parity runs one phase behind
      mbar_wait_t(&bars->c_empty[s], ((t / kStages) & 1) ^ (s >= kStages - 2 ? 0 : 1), w0);
      if (MT::kColRing) mbar_wait_t(&bars->m_empty[ms], ((t / kMetaSlots) & 1) ^ 1, w1);
      if (elect_one()) {
        mbar_expect_tx(&bars->c_full[s], (uint32_t)kc * BN * 128);
        uint8_t* dst = sC + (size_t)s * kc * BN * 128;
        if (CS == 1) {
          for (int c = 0; c < kc; ++c) tma_load_2d(dst + (size_t)c * BN * 128, &map_cols, &bars->c_full[s], c * KCH, tile_col(t));
        } else {
          constexpr int kSlice = BN / CS;        // rows of the tile this CTA fetches for the whole cluster
          for (int c = 0; c < kc; ++c)
            tma_load_2d_mc(dst + (size_t)c * BN * 128 + (size_t)crank * kSlice * 128, &map_cols, &bars->c_full[s], c * KCH,
                           tile_col(t) + (int)crank * kSlice, kAllCtas);
        }
        if (MODE == kAnaCols) {
          mbar_expect_tx(&bars->m_full[ms], (uint32_t)(BN * sizeof(float)));
          bulk_load_1d(sMeta[ms].stat, a.col_shift + tile_col(t), BN * sizeof(float), &bars->m_full[ms]);
        } else if (MT::kColRing) {
          constexpr bool with_stat = MODE == kGenCols;
          mbar_expect_tx(&bars->m_full[ms], (uint32_t)(BN * sizeof(int2) + (with_stat ? BN * sizeof(float4) : 0)));
          bulk_load_1d(sMeta[ms].meta, a.col_meta + tile_col(t), BN * sizeof(int2), &bars->m_full[ms]);
          if (with_stat) bulk_load_1d(sMeta[ms].stat, a.col_stat + tile_col(t), BN * sizeof(float4), &bars->m_full[ms]);
        }
      }
      __syncwarp();
    }
    if (kProfile && a.prof && blockIdx.x == 0 && blockIdx.y == 0 && lane == 0) {
      a.prof[0] = (unsigned long long)(SLCL_PROF_NOW() - tstart); a.prof[1] = w0; a.prof[2] = w1;
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    const uint32_t idesc1 = make_idesc(BN, 0);
    const uint32_t idesc2 = make_idesc(a.d, 1);
    const uint32_t c_addr = smem_u32(sC);
    unsigned long long w0 = 0, w1 = 0, w2 = 0;
    const long long tstart = SLCL_PROF_NOW();
    mbar_wait(&bars->r_full, 0);
    tc_fence_after();
    if (elect_one()) {                       // R has left its staging stages: release them to the ring (in every CTA)
      for (int s = kStages - 2; s < kStages; ++s) {
        if (CS == 1) umma_commit(&bars->c_empty[s]); else umma_commit_mc(&bars->c_empty[s], kAllCtas);
      }
    }
    __syncwarp();
    // Descriptors are built once; inside the loops only the 14-bit start-address field moves
    // (all operand addresses are < 256 KB, so adding (bytes >> 4) to the low word never carries out).
    const uint64_t descC = make_desc(c_addr, 16, 1024);              // K-major view of a column tile (MMA1)
    const uint64_t descCmn = make_desc(c_addr, BN * 128, 1024);      // MN-major view of the same bytes (MMA2)
    const uint32_t stage_units = (uint32_t)(kc * BN * 128) >> 4;
    for (int t = 0; t <= n_tiles; ++t) {
      if (t < n_tiles) {
        const int s = t % kStages, buf = t & 1;
        mbar_wait_t(&bars->c_full[s], (t / kStages) & 1, w0);
        // S[buf] is free once the epilogue of tile t-2 has it in registers.  In the MMA2 modes that is implied:
        // MMA2(t-2), issued in the previous iteration, waited for G(t-2), which the epilogue writes after the read.
        if (!MT::kMma2) mbar_wait_t(&bars->s_empty[buf], ((t >> 1) & 1) ^ 1, w1);
        tc_fence_after();
        if (elect_one()) {
          // S[buf] = R . Cm_tile^T : A = R from tensor memory, B = column tile K-major, 16 bf16 of K per MMA
          const uint32_t d_tmem = tmem + kColS + buf * BN;
          uint32_t ta = tmem + kColR;                          // 16 bf16 of K = 8 tensor-memory columns per step
          uint64_t db = descC + (uint64_t)(s * stage_units);
          for (int c = 0; c < kc; ++c) {
#pragma unroll
            for (int k = 0; k < KCH / 16; ++k)
              umma_bf16_ts(d_tmem, ta + 8 * k, db + 2 * k, idesc1, (c | k) != 0);
            ta += KCH / 2;
            db += (BN * 128) >> 4;
          }
          umma_commit(&bars->s_full[buf]);
          if (!MT::kMma2) { if (CS == 1) umma_commit(&bars->c_empty[s]); else umma_commit_mc(&bars->c_empty[s], kAllCtas); }
        }
        __syncwarp();
      }
      if (MT::kMma2 && t > 0) {
        // D += G(t-1)[128 x 64] . Cm_tile(t-1)[64 x d] : A = G from tensor memory (the epilogue warp of column half h
        // left its 32 bf16 columns packed in S columns [32h, 32h+16)); B = Cm tile as MN-major operand
        const int tp = t - 1, sp = tp % kStages, bp = tp & 1;
        mbar_wait_t(&bars->g_full[bp], (tp >> 1) & 1, w2);
        tc_fence_after();
        if (elect_one()) {
          const uint32_t ga = tmem + kColS + bp * BN;
          const uint64_t dc = descCmn + (uint64_t)(sp * stage_units);
#pragma unroll
          for (int k = 0; k < BN / 16; ++k)
            umma_bf16_ts(tmem + kColAcc, ga + (k >> 1) * 32 + (k & 1) * 8, dc + k * (2048 >> 4), idesc2, (tp | k) != 0);
          if (CS == 1) umma_commit(&bars->c_empty[sp]); else umma_commit_mc(&bars->c_empty[sp], kAllCtas);
        }
        __syncwarp();
      }
    }
    if (MT::kMma2 && elect_one()) umma_commit(&bars->acc_full);
    __syncwarp();
    if (kProfile && a.prof && blockIdx.x == 0 && blockIdx.y == 0 && lane == 0) {
      a.prof[4] = (unsigned long long)(SLCL_PROF_NOW() - tstart); a.prof[5] = w0; a.prof[6] = w1; a.prof[7] = w2;
    }
  } else if (warp >= 4) {
    // ===================== epilogue: one thread per row, 32 of the 64 tile columns per warp =====================
    const int q = warp & 3;                       // TMEM lane quarter this warp may access
    const int half = (warp - 4) >> 2;             // column half of the S tile
    const int r_local = q * 32 + lane;
    const int row = row0 + r_local;
    const bool row_ok = row < row_end;
    int2 rm = make_int2(INT_MIN + 1, INT_MIN + 1);
    float4 rs = make_float4(0.f, 0.f, 0.f, 0.f);
    if (MODE == kGenFwd || MODE == kGenRows) { if (row_ok) rm = a.row_meta[row]; }
    if (MODE == kGenCols) { if (row_ok) rm = a.row_meta[row]; }
    if (MODE == kGenRows) { if (row_ok) rs = a.row_stat[row]; }
    if (MODE == kGenFwd || MODE == kAnaFwd || MODE == kAnaFwdU) { if (row_ok) rs.x = a.row_shift[row] * kLog2e; }
    float zs[4] = {0.f, 0.f, 0.f, 0.f};
    float praw = 0.f, npos = 0.f;
    unsigned long long w0 = 0, w1 = 0;
    const uint32_t lane_addr = ((uint32_t)(q * 32) << 16);
    // fused dB drain (kAnaCols, one split): fetch what the drain needs now, long before it is used
    const bool fused = (MODE == kAnaCols || MODE == kGenCols) && a.fused_out != nullptr;      // the drain writes d_b itself
    float gscale = 1.f;
    int lab = -1;
    if (MODE == kAnaCols && fused) {
      gscale = a.grad_out[0];
      if (row_ok) lab = a.row_meta[row].x;
      if (lab >= a.n_class) lab = -1;
      for (int idx = threadIdx.x - 128; idx < a.n_class * a.d; idx += 32 * kEpiWarps)
        sTab[idx] = a.ab_sums[((size_t)batch * a.n_class + (size_t)(idx / a.d)) * (a.d + 1) + idx % a.d];      // this batch's table
      asm volatile("bar.sync 1, %0;" ::"n"(32 * kEpiWarps) : "memory");         // the eight epilogue warps only
    }
    if (half == 0) {
      // resident operand: this thread's row of the staged tile (128-byte-swizzled rows of 64 bf16) -> tensor memory
      // lane r_local as packed bf16 pairs.  Rows past n_rows were zero-filled by TMA.
      mbar_wait(&bars->r_in, 0);
      const uint8_t* rsrc = sC + (size_t)(kStages - 2) * kc * BN * 128 + (size_t)r_local * 128;
      for (int c = 0; c < kc; ++c) {
        uint32_t v[32];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const uint4 t = *reinterpret_cast<const uint4*>(rsrc + (size_t)c * BM * 128 + ((i ^ (r_local & 7)) << 4));
          v[4 * i] = t.x; v[4 * i + 1] = t.y; v[4 * i + 2] = t.z; v[4 * i + 3] = t.w;
        }
        tmem_st32(tmem + lane_addr + kColR + c * 32, v);
      }
      tmem_st_wait();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&bars->r_full);
    }
    const long long tstart = SLCL_PROF_NOW();
    for (int t = 0; t < n_tiles; ++t) {
      const int buf = t & 1;
      const int ms = t % kMetaSlots;
      const uint32_t cstat_u32 = (uint32_t)__cvta_generic_to_shared(sMeta + ms);               // ColMeta::stat [BN] float4
      const uint32_t cmeta_u32 = cstat_u32 + (uint32_t)(BN * sizeof(float4));                    // ColMeta::meta [BN] int2
      if (MT::kColRing) mbar_wait_t(&bars->m_full[ms], (t / kMetaSlots) & 1, w0);
      mbar_wait_t(&bars->s_full[buf], (t >> 1) & 1, w1);
      tc_fence_after();
      uint32_t v[32];
      const uint32_t s_addr = tmem + lane_addr + kColS + buf * BN + half * 32;
      tmem_ld32(s_addr, v);
      tmem_ld_wait();
      if (!MT::kMma2) {
        // S buffer is free as soon as it sits in registers
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&bars->s_empty[buf]);
      }
      uint32_t packed[16];
      // general modes with self maps: is this warp's half tile label-uniform?  (one shared load, a shuffle and a vote)
      bool gen_fast = false, gen_same = false;
      if ((MODE == kGenFwd || MODE == kGenRows || MODE == kGenCols) && !a.self_by_id) {
        const int my_col_label = lds_int2(cmeta_u32 + (uint32_t)((half * 32 + lane) * 8)).x;
        const int tile_label = __shfl_sync(0xffffffffu, my_col_label, 0);
        gen_fast = __all_sync(0xffffffffu, my_col_label == tile_label);
        gen_same = rm.x == tile_label;
      }

      if (MODE == kAnaFwd || MODE == kAnaFwdU) {
        // e = exp2(s * scale - shift): four independent accumulation chains
#pragma unroll
        for (int jj = 0; jj < 32; jj += 2) {
          const float e0 = ex2_approx(fmaf(__uint_as_float(v[jj]), a.scale_log2, -rs.x));
          const float e1 = ex2_approx(fmaf(__uint_as_float(v[jj + 1]), a.scale_log2, -rs.x));
          zs[jj & 2] += e0;
          zs[(jj & 2) + 1] += e1;
          if (MODE == kAnaFwdU) packed[jj >> 1] = pack_bf16x2(e0, e1);
        }
      } else if (MODE == kAnaCols) {
        const uint32_t cs4 = cstat_u32 + (uint32_t)(half * 8 * 16);
#pragma unroll
        for (int jj = 0; jj < 32; jj += 4) {
          const float4 sh = lds_float4(cs4 + (uint32_t)((jj >> 2) * 16));
          const float e0 = ex2_approx(fmaf(__uint_as_float(v[jj]), a.scale_log2, -sh.x));
          const float e1 = ex2_approx(fmaf(__uint_as_float(v[jj + 1]), a.scale_log2, -sh.y));
          const float e2 = ex2_approx(fmaf(__uint_as_float(v[jj + 2]), a.scale_log2, -sh.z));
          const float e3 = ex2_approx(fmaf(__uint_as_float(v[jj + 3]), a.scale_log2, -sh.w));
          packed[jj >> 1] = pack_bf16x2(e0, e1);
          packed[(jj >> 1) + 1] = pack_bf16x2(e2, e3);
        }
      } else if (MODE == kGenFwd) {
        if (gen_fast) {
          // label-uniform half tile (the caller sorted the contrast rows by label) and no id tests: FFMA + EX2 + 2 FADD
          float tsum = 0.f;
#pragma unroll
          for (int jj = 0; jj < 32; ++jj) {
            const float sv = __uint_as_float(v[jj]);
            zs[jj & 3] += ex2_approx(fmaf(sv, a.scale_log2, -rs.x));
            tsum += sv;
          }
          if (gen_same) { praw += tsum; npos += 32.f; }
        } else {
          const int rid = a.self_by_id ? rm.y : INT_MIN + 2;      // self maps given: never equal to a column id
#pragma unroll
          for (int jj = 0; jj < 32; ++jj) {
            const int2 cm = lds_int2(cmeta_u32 + (uint32_t)((half * 32 + jj) * 8));
            const float s = __uint_as_float(v[jj]);
            const float e = ex2_approx(fmaf(s, a.scale_log2, -rs.x));
            // predicated adds spelled out in PTX: 2 compares + 3 predicated FADDs, no selects, no branches
            asm("{\n\t"
                ".reg .pred pv, pp;\n\t"
                "setp.ne.s32 pv, %5, %6;\n\t"
                "setp.eq.and.s32 pp, %7, %8, pv;\n\t"
                "@pv add.f32 %0, %0, %3;\n\t"
                "@pp add.f32 %1, %1, %4;\n\t"
                "@pp add.f32 %2, %2, 0f3F800000;\n\t"
                "}\n"
                : "+f"(zs[0]), "+f"(praw), "+f"(npos)
                : "f"(e), "f"(s), "r"(cm.y), "r"(rid), "r"(cm.x), "r"(rm.x));
          }
        }
      } else if (gen_fast) {
        // general backward on a label-uniform half tile: G = alpha e - [row label == tile label] beta, no integer work
#pragma unroll
        for (int jj = 0; jj < 32; jj += 2) {
          float g2[2];
#pragma unroll
          for (int u = 0; u < 2; ++u) {
            float sh = rs.x, al = rs.y, be = rs.z;
            if (MODE == kGenCols) {
              const float4 st = lds_float4(cstat_u32 + (uint32_t)((half * 32 + jj + u) * 16));
              sh = st.x; al = st.y; be = st.z;
            }
            const float e = ex2_approx(fmaf(__uint_as_float(v[jj + u]), a.scale_log2, -sh));
            g2[u] = fmaf(al, e, gen_same ? -be : 0.f);
          }
          packed[jj >> 1] = pack_bf16x2(g2[0], g2[1]);
        }
      } else {
        // general backward: G = alpha e - [same label] beta, zero for the self pair.  The statistics
        // {shift, alpha, beta} belong to the row (dA sweep) or to the column (dB sweep).
        const int rid = a.self_by_id ? rm.y : INT_MIN + 2;
#pragma unroll
        for (int jj = 0; jj < 32; jj += 2) {
          float g2[2];
#pragma unroll
          for (int u = 0; u < 2; ++u) {
            const int2 cm = lds_int2(cmeta_u32 + (uint32_t)((half * 32 + jj + u) * 8));
            float sh = rs.x, al = rs.y, be = rs.z;
            if (MODE == kGenCols) {
              const float4 st = lds_float4(cstat_u32 + (uint32_t)((half * 32 + jj + u) * 16));
              sh = st.x; al = st.y; be = st.z;
            }
            const float s = __uint_as_float(v[jj + u]);
            const float e = ex2_approx(fmaf(s, a.scale_log2, -sh));
            float g;
            asm("{\n\t"
                ".reg .pred pv, pp;\n\t"
                "setp.ne.s32 pv, %4, %5;\n\t"
                "setp.eq.s32 pp, %6, %7;\n\t"
                "mul.f32 %0, %1, %2;\n\t"
                "@pp sub.f32 %0, %0, %3;\n\t"
                "@!pv mov.f32 %0, 0f00000000;\n\t"
                "}\n"
                : "=&f"(g)
                : "f"(al), "f"(e), "f"(be), "r"(cm.y), "r"(rid), "r"(cm.x), "r"(rm.x));
            g2[u] = g;
          }
          packed[jj >> 1] = pack_bf16x2(g2[0], g2[1]);
        }
      }
      if (MT::kRowSums) {
        // Padding columns (beyond col_end; only the last tile of a sweep has them) were read as zero rows
        // by TMA (sentinel id/label in the general mode) and therefore entered zs as exp(0 - shift): take
        // them out analytically instead of testing every element.  Their G entries multiply zero rows.
        const int jb = tile_col(t) + half * 32;
        const int n_pad = max(0, min(32, jb + 32 - col_end));
        if (n_pad > 0) zs[0] -= (float)n_pad * ex2_approx(-rs.x);
      }
      if (MT::kMma2) {
        // G tile -> tensor memory, over the S columns this warp has just read: row = lane, 16 words of bf16 pairs
        tmem_st16(s_addr, packed);
        tmem_st_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&bars->g_full[buf]);
      }
      if (MT::kColRing) {
        __syncwarp();
        if (lane == 0) mbar_arrive(&bars->m_empty[ms]);
      }
    }

    if (kProfile && a.prof && blockIdx.x == 0 && blockIdx.y == 0 && lane == 0 && (warp == 4 || warp == 11)) {
      unsigned long long* pp = a.prof + (warp == 4 ? 8 : 12);
      pp[0] = (unsigned long long)(SLCL_PROF_NOW() - tstart); pp[1] = w0; pp[2] = w1;
      if (warp == 4) {
        a.prof[3] = (unsigned long long)(tstart - t_entry);          // set-up + R load
        a.prof[9] = (unsigned long long)(t_setup - t_entry);         // barrier init, TMEM allocation
        a.prof[10] = (unsigned long long)(t_pdl - t_setup);          // waiting for the kernel in front
      }
    }
    const long long t_drain = SLCL_PROF_NOW();
    if (MT::kRowSums) {
      if (row_ok) {
        float* out = a.stat_partial + ((size_t)(split * 2 + half) * a.n_rows + row) * MT::kStatN;
        out[0] = (zs[0] + zs[1]) + (zs[2] + zs[3]);
        if (MODE == kGenFwd) { out[1] = praw; out[2] = npos; }
      }
    }
    if (MT::kMma2) {
      // Accumulators -> global, 32 columns at a time; the warps of the two column halves interleave over d.
      // Each 32 x 32 block is transposed through a padded staging tile in shared memory (the operand ring is idle
      // now), so every store instruction writes one full 128-byte line of one row.
      mbar_wait(&bars->acc_full, 0);
      tc_fence_after();
      if (kProfile && a.prof && blockIdx.x == 0 && blockIdx.y == 0 && lane == 0 && warp == 4)
        a.prof[13] = (unsigned long long)(SLCL_PROF_NOW() - t_drain);             // waiting for the last MMA2
      // Each warp stages a 32-row x 32-column fp32 block (thread = row, 128 bytes, 16-byte chunks XOR-swizzled so
      // the 128-bit stores are conflict-free) in the idle operand ring and hands it to a TMA store; two staging
      // buffers per warp keep one store in flight while the next block is read out of tensor memory.
      uint8_t* stg = sC + (size_t)(warp - 4) * (2 * 4096);
      const float* tab = sTab;
      int nbuf = 0;
      for (int c = half * 32; c < a.d; c += 64, nbuf ^= 1) {
        uint32_t v[32];
        tmem_ld32(tmem + lane_addr + kColAcc + c, v);
        tmem_ld_wait();
        if (MODE == kAnaCols && fused) {
          // thread = row: subtract the row's class sum (rows of one label broadcast the same 16 bytes) and scale
          const float4* t4 = reinterpret_cast<const float4*>(tab + (size_t)max(lab, 0) * a.d + c);
          const float m = lab >= 0 ? 1.f : 0.f;
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const float4 t = t4[i];
            v[4 * i] = __float_as_uint(gscale * fmaf(-m, t.x, __uint_as_float(v[4 * i])));
            v[4 * i + 1] = __float_as_uint(gscale * fmaf(-m, t.y, __uint_as_float(v[4 * i + 1])));
            v[4 * i + 2] = __float_as_uint(gscale * fmaf(-m, t.z, __uint_as_float(v[4 * i + 2])));
            v[4 * i + 3] = __float_as_uint(gscale * fmaf(-m, t.w, __uint_as_float(v[4 * i + 3])));
          }
        }
        if (lane == 0) bulk_wait_read<1>();            // the store that last read this staging buffer is done with it
        __syncwarp();
        uint8_t* dst = stg + nbuf * 4096 + lane * 128;
#pragma unroll
        for (int i = 0; i < 8; ++i)
          *reinterpret_cast<uint4*>(dst + ((i ^ (lane & 7)) << 4)) = make_uint4(v[4 * i], v[4 * i + 1], v[4 * i + 2], v[4 * i + 3]);
        fence_proxy_async();
        __syncwarp();
        if (lane == 0) {
          tma_store_3d(&map_out, stg + nbuf * 4096, c, row0 + q * 32, fused ? 0 : split);
          bulk_commit();
        }
      }
      if (lane == 0) bulk_wait_all();
      __syncwarp();
      tc_fence_before();
    }
    if (kProfile && a.prof && blockIdx.x == 0 && blockIdx.y == 0 && lane == 0 && warp == 4) {
      a.prof[11] = (unsigned long long)(SLCL_PROF_NOW() - t_drain);               // accumulator drain
      a.prof[15] = (unsigned long long)(SLCL_PROF_NOW() - t_entry);               // whole CTA
    }
  }
  __syncthreads();
  if (CS > 1) cluster_sync_all();          // no CTA leaves while a peer may still multicast into it
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc(tmem, kTmemCols);
  }
}

// ---------------------------------------------------------------------------
// small helper kernels
// ---------------------------------------------------------------------------
// dot product of two bf16 rows (length d, multiple of 64) by one warp, fp32 accumulate
__device__ __forceinline__ float warp_dot_bf16(const __nv_bfloat16* x, const __nv_bfloat16* y, int d, int lane) {
  float acc = 0.f;
  for (int c = lane * 2; c < d; c += 64) {
    const float2 a2 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(x + c));
    const float2 b2 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(y + c));
    acc = fmaf(a2.x, b2.x, acc);
    acc = fmaf(a2.y, b2.y, acc);
  }
  return warp_sum(acc);
}
__device__ __forceinline__ float bf16_round(float x) { return __bfloat162float(__float2bfloat16_rn(x)); }

// ---- row groups: LPR = 8, 16 or 32 lanes per row (the finishing kernels; LPR = d / 8 so that one 16-byte load per lane
// covers a bf16 row, 32 / LPR rows per warp instruction).  The shuffles name only the group's lanes, so the groups of a
// warp may diverge.
template <int LPR>
__device__ __forceinline__ unsigned grp_mask(int lane) {
  return LPR == 32 ? 0xffffffffu : (((1u << (LPR & 31)) - 1u) << (lane & ~(LPR - 1)));
}
template <int LPR>
__device__ __forceinline__ float grp_sum(float v, unsigned mask) {
#pragma unroll
  for (int o = LPR / 2; o > 0; o >>= 1) v += __shfl_xor_sync(mask, v, o);
  return v;
}
__device__ __forceinline__ void bf16x8_to_float(const uint4& r, float (&x)[8]) {
  const uint32_t w[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    x[2 * k] = __uint_as_float(w[k] << 16);
    x[2 * k + 1] = __uint_as_float(w[k] & 0xFFFF0000u);
  }
}
template <int LPR>
__device__ __forceinline__ float grp_dot_bf16(const __nv_bfloat16* x, const __nv_bfloat16* y, int d, int lg, unsigned mask) {
  float acc = 0.f;
  for (int c = lg * 8; c < d; c += LPR * 8) {
    float xa[8], ya[8];
    bf16x8_to_float(*reinterpret_cast<const uint4*>(x + c), xa);
    bf16x8_to_float(*reinterpret_cast<const uint4*>(y + c), ya);
#pragma unroll
    for (int k = 0; k < 8; ++k) acc = fmaf(xa[k], ya[k], acc);
  }
  return grp_sum<LPR>(acc, mask);
}
inline int lanes_per_row(int d) { return d <= 64 ? 8 : (d <= 128 ? 16 : 32); }

// ---- general path -----------------------------------------------------------
// stats[i] = sum over slots of partial (deterministic order); also the per-block partial of
// sum_i w_i * (shift_i + log(Zs_i) - P_i / n_i),  P_i = P_raw_i / T     (utils/loss.py:371-386)
__global__ void __launch_bounds__(256) p2p_reduce_stats_kernel(const float* partial, int n_slots, int n_rows, const float* shift,
                                                               const float* weight, float inv_t, float* stats,
                                                               double* loss_partial) {
  pdl_trigger();
  pdl_wait();
  __shared__ double red[8];
  const int i = blockIdx.x * 256 + threadIdx.x;
  double acc = 0.0;
  if (i < n_rows) {
    float t[3] = {0.f, 0.f, 0.f};
    for (int s = 0; s < n_slots; ++s) {
      const float* p = partial + ((size_t)s * n_rows + i) * 3;
      t[0] += p[0]; t[1] += p[1]; t[2] += p[2];
    }
    stats[3 * i] = t[0]; stats[3 * i + 1] = t[1]; stats[3 * i + 2] = t[2];
    const float li = shift[i] + logf(t[0]) - (t[1] * inv_t) / t[2];     // n == 0 -> NaN, as 0/0 in the reference (:376-380)
    acc = (double)(weight[i] * li);
  }
  acc = warp_sum(acc);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
    for (int w = 0; w < 8; ++w) t += red[w];
    loss_partial[blockIdx.x] = t;
  }
}

__global__ void __launch_bounds__(256) p2p_loss_kernel(const double* loss_partial, int n_blocks, float* loss) {
  pdl_trigger();
  pdl_wait();
  __shared__ double red[8];
  double acc = 0.0;
  for (int i = threadIdx.x; i < n_blocks; i += 256) acc += loss_partial[i];
  acc = warp_sum(acc);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
    for (int w = 0; w < 8; ++w) t += red[w];
    loss[0] = (float)t;
  }
}

// per-anchor backward constants {shift*log2e, alpha, beta, 0}: alpha = g w /(T Zs), beta = g w /(T n)
__global__ void p2p_anchor_stat_kernel(const float* stats, const float* shift, const float* weight, const float* grad_out,
                                       int n, int n_padded, float inv_t, float4* out) {
  pdl_trigger();
  pdl_wait();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_padded) return;
  if (i >= n) { out[i] = make_float4(0.f, 0.f, 0.f, 0.f); return; }      // pad entries (bulk-copied as column stats)
  const float gw = grad_out[0] * weight[i] * inv_t;
  out[i] = make_float4(shift[i] * kLog2e, gw / stats[3 * i], gw / stats[3 * i + 2], 0.f);
}

// out[r][c] = sum over splits of partial[s][r][c]  (-  g_self * other[c] when the caller gave self maps: the sweep treated
// the self pair as an ordinary pair)
//   dA sweep: rows are anchors:       other row = b[a_selfcol[r]],  g_self = gself[r]
//   dB sweep: rows are contrast rows: anchor m = b_selfrow[r], other row = a[m], g_self = gself[m]
__global__ void p2p_reduce_grad_kernel(const float* partial, int n_splits, int64_t n_elems, int d_pad, int d, float* out,
                                       const float* gself, const int32_t* self_map, const __nv_bfloat16* other,
                                       int rows_are_anchors) {
  pdl_trigger();
  pdl_wait();
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= n_elems) return;
  const int64_t r = idx / d, c = idx % d;
  float t = 0.f;
  const int64_t stride = (n_elems / d) * d_pad;
  for (int s = 0; s < n_splits; ++s) t += partial[(size_t)s * stride + r * d_pad + c];
  if (self_map != nullptr) {
    const int m = self_map[r];
    if (m >= 0) t -= (rows_are_anchors ? gself[r] : gself[m]) * __bfloat162float(other[(size_t)m * d_pad + c]);
  }
  out[idx] = t;
}

// General sweeps with self maps, forward finish: one warp per anchor.  stats[i] = sum over slots (fixed order) minus the
// self pair  S_ii = a_i . b_selfcol(i):  Zs -= exp(S_ii / T - shift);  labels agree -> P_raw -= S_ii, n -= 1.
// Also the per-block partial of  sum_i w_i (shift_i + log Zs_i - P_raw_i / (T n_i))        (utils/loss.py:371-386)
__global__ void __launch_bounds__(256) p2p_reduce_stats_self_kernel(const float* partial, int n_slots, int n_rows,
                                                                    const float* shift, const float* weight, float inv_t,
                                                                    const __nv_bfloat16* a, const __nv_bfloat16* b, int d,
                                                                    const int2* a_meta, const int2* b_meta,
                                                                    const int32_t* a_selfcol, float* stats,
                                                                    double* loss_partial) {
  pdl_trigger();
  pdl_wait();
  __shared__ double red[8];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int i = blockIdx.x * 8 + warp;
  double acc = 0.0;
  if (i < n_rows) {
    float t[3] = {0.f, 0.f, 0.f};
    for (int s = lane; s < n_slots; s += 32) {
      const float* p = partial + ((size_t)s * n_rows + i) * 3;
      t[0] += p[0]; t[1] += p[1]; t[2] += p[2];
    }
    t[0] = warp_sum(t[0]); t[1] = warp_sum(t[1]); t[2] = warp_sum(t[2]);
    const int sc = a_selfcol[i];
    if (sc >= 0) {
      const float s_self = warp_dot_bf16(a + (size_t)i * d, b + (size_t)sc * d, d, lane);
      // The self term was summed by the sweep (tensor-core route) and is taken out here (fp32 route): when it dominates
      // the row -- small T, few or distant neighbours -- the difference is pure round-off and can come out <= 0.  Floor it
      // at the round-off level of the self term so log() and 1/Zs stay finite (the reference masks the diagonal exactly
      // and is finite there too; below this floor no fp32 evaluation of the row is meaningful).
      const float e_self = ex2_approx(fmaf(s_self, inv_t * kLog2e, -shift[i] * kLog2e));
      t[0] = fmaxf(t[0] - e_self, e_self * 1.1920929e-7f);
      if (a_meta[i].x == b_meta[sc].x) { t[1] -= s_self; t[2] -= 1.f; }
    }
    if (lane == 0) {
      stats[3 * i] = t[0]; stats[3 * i + 1] = t[1]; stats[3 * i + 2] = t[2];
      const float li = shift[i] + logf(t[0]) - (t[1] * inv_t) / t[2];     // n == 0 -> NaN, as 0/0 in the reference (:376-380)
      acc = (double)(weight[i] * li);
    }
  }
  if (lane == 0) red[warp] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    double tt = 0.0;
    for (int w = 0; w < 8; ++w) tt += red[w];
    loss_partial[blockIdx.x] = tt;
  }
}

// Self-pair entry of the gradient tile, exactly as the sweeps formed it (bf16-rounded):
// g_self[i] = bf16(alpha_i exp(S_ii / T - shift_i) - [labels agree] beta_i), 0 when anchor i has no self column.
__global__ void __launch_bounds__(256) p2p_gself_kernel(const float4* anchor_stat, float scale_log2, const __nv_bfloat16* a,
                                                        const __nv_bfloat16* b, int d, const int2* a_meta, const int2* b_meta,
                                                        const int32_t* a_selfcol, int n_rows, float* gself) {
  pdl_trigger();
  pdl_wait();
  const int lane = threadIdx.x & 31;
  const int i = blockIdx.x * 8 + (threadIdx.x >> 5);
  if (i >= n_rows) return;
  const int sc = a_selfcol[i];
  float g = 0.f;
  if (sc >= 0) {
    const float s_self = warp_dot_bf16(a + (size_t)i * d, b + (size_t)sc * d, d, lane);
    const float4 st = anchor_stat[i];
    g = bf16_round(fmaf(st.y, ex2_approx(fmaf(s_self, scale_log2, -st.x)), (a_meta[i].x == b_meta[sc].x) ? -st.z : 0.f));
  }
  if (lane == 0) gself[i] = g;
}

// General dB sweep whose drain wrote d_b directly (one column split), self maps given: take the self-pair entry out,
//   d_b[selfcol(i)] -= g_self[i] * a_i      (one warp per anchor; ids are unique, so no two warps touch the same row)
__global__ void __launch_bounds__(256) p2p_self_fix_kernel(const float* gself, const int32_t* a_selfcol, const __nv_bfloat16* a,
                                                           int d_pad, int dim, int n_anchor, float* d_b) {
  pdl_trigger();
  pdl_wait();
  const int lane = threadIdx.x & 31;
  const int i = blockIdx.x * 8 + (threadIdx.x >> 5);
  if (i >= n_anchor) return;
  const int sc = a_selfcol[i];
  if (sc < 0) return;
  const float g = gself[i];
  for (int c = lane; c < dim; c += 32) d_b[(size_t)sc * dim + c] -= g * __bfloat162float(a[(size_t)i * d_pad + c]);
}

// ---- analytic path ----------------------------------------------------------
// Label-indexed accumulation of one bf16 row into a warp-private table in shared memory: tab[lab][c] += coef * x[c]
// (lane = 8 consecutive columns, so the 32 lanes never collide), cnt[lab] += coef.
__device__ __forceinline__ void label_table_add(float* tab, float* cnt, int d, int lab, float coef, uint4 x, int lane) {
  if (lane * 8 < d) {
    float4* acc = reinterpret_cast<float4*>(tab + (size_t)lab * d + lane * 8);
    float4 a0 = acc[0], a1 = acc[1];
    a0.x = fmaf(coef, __uint_as_float(x.x << 16), a0.x); a0.y = fmaf(coef, __uint_as_float(x.x & 0xFFFF0000u), a0.y);
    a0.z = fmaf(coef, __uint_as_float(x.y << 16), a0.z); a0.w = fmaf(coef, __uint_as_float(x.y & 0xFFFF0000u), a0.w);
    a1.x = fmaf(coef, __uint_as_float(x.z << 16), a1.x); a1.y = fmaf(coef, __uint_as_float(x.z & 0xFFFF0000u), a1.y);
    a1.z = fmaf(coef, __uint_as_float(x.w << 16), a1.z); a1.w = fmaf(coef, __uint_as_float(x.w & 0xFFFF0000u), a1.w);
    acc[0] = a0; acc[1] = a1;
  }
  if (lane == 0) cnt[lab] += coef;
}
// fixed-order combine of the eight warp tables of a block -> partial[block][K][d], cnt[block][K]  (after __syncthreads)
__device__ __forceinline__ void label_tables_flush(const float* s_sum, const float* s_cnt, int n_class, int d, float* partial,
                                                   float* cnt) {
  const size_t blk = (size_t)blockIdx.y * gridDim.x + blockIdx.x;          // blockIdx.y = block-diagonal batch
  for (int idx = threadIdx.x; idx < n_class * d; idx += 256) {
    float t = 0.f;
#pragma unroll
    for (int w = 0; w < 8; ++w) t += s_sum[(size_t)w * n_class * d + idx];
    partial[blk * n_class * d + idx] = t;
  }
  if ((int)threadIdx.x < n_class) {
    float t = 0.f;
#pragma unroll
    for (int w = 0; w < 8; ++w) t += s_cnt[w * n_class + threadIdx.x];
    cnt[blk * n_class + threadIdx.x] = t;
  }
}

// Per-class row sums, stage 1:  sum[k] = sum_{rows r with label k} coef_r x_r,  cnt[k] = sum coef_r.
//   kBeta = false: coef = 1 (Bsum / class counts of the contrast rows);
//   kBeta = true : coef = beta~_r = w_r / (T n_r),  n_r = count[lab_r] - [row r is itself a contrast row with the same label]
//                  (0 when n_r == 0) -> ABsum of the anchors; the coefficients are also written to beta_out.  They depend on
//                  labels and weights only, so this runs on the side stream next to the forward sweep.
// A block owns kLabelRowsPerBlock rows at a time (grid-stride over the row blocks); a warp walks every 8th row of them with
// 16-byte loads, eight rows in flight.  Stage 2 (p2p_label_reduce_kernel) sums the blocks in fixed order.
constexpr int kLabelRowsPerBlock = 64;
template <bool kBeta>
__global__ void __launch_bounds__(256) p2p_label_part_kernel(const __nv_bfloat16* rows, int n_rows, int d, const int2* meta,
                                                             int n_class, float* partial, float* cnt, const float* weight,
                                                             float inv_t, const int32_t* selfcol, const int2* other_meta,
                                                             const float* other_sums, float* beta_out,
                                                             unsigned int* zero_ticket) {
  pdl_trigger();
  pdl_wait();
  if (zero_ticket != nullptr && blockIdx.x == 0 && blockIdx.y == 0 && threadIdx.x == 0) *zero_ticket = 0u;      // (see p2p_finish_fwd_kernel)
  // block-diagonal batches (gridDim.y > 1): batch z owns rows [z n_rows, (z+1) n_rows) and its own [K][d+1] tables;
  // n_rows is the per-batch row count, self columns stay global contrast-row indices
  {
    const size_t z = blockIdx.y;
    rows += z * (size_t)n_rows * d;
    meta += z * (size_t)n_rows;
    if (kBeta) {
      weight += z * (size_t)n_rows;
      beta_out += z * (size_t)n_rows;
      if (selfcol) selfcol += z * (size_t)n_rows;
      other_sums += z * (size_t)n_class * (d + 1);
    }
  }
  extern __shared__ float sm_lp[];                 // [8 warps][K][d] + [8][K]
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float* s_sum = sm_lp;
  float* s_cnt = sm_lp + (size_t)8 * n_class * d;
  float* my_sum = s_sum + (size_t)warp * n_class * d;
  float* my_cnt = s_cnt + warp * n_class;
  for (int idx = lane; idx < n_class * d; idx += 32) my_sum[idx] = 0.f;
  if (lane < n_class) my_cnt[lane] = 0.f;
  __syncwarp();
  constexpr int kInFlight = 8;
  for (int r0 = blockIdx.x * kLabelRowsPerBlock; r0 < n_rows; r0 += gridDim.x * kLabelRowsPerBlock) {
    const int r1 = min(n_rows, r0 + kLabelRowsPerBlock);
    for (int rb = r0 + warp; rb < r1; rb += 8 * kInFlight) {
      uint4 x[kInFlight];
      int lab[kInFlight];
      float coef[kInFlight];
#pragma unroll
      for (int u = 0; u < kInFlight; ++u) {
        const int r = rb + 8 * u;
        lab[u] = -1; x[u] = make_uint4(0u, 0u, 0u, 0u); coef[u] = 1.f;
        if (r < r1) {
          lab[u] = meta[r].x;
          if (lane * 8 < d) x[u] = __ldg(reinterpret_cast<const uint4*>(rows + (size_t)r * d) + lane);
        }
      }
      if (kBeta) {
#pragma unroll
        for (int u = 0; u < kInFlight; ++u) {
          const int r = rb + 8 * u;
          if (r < r1) {
            const bool ok = lab[u] >= 0 && lab[u] < n_class;
            float n = 0.f;
            if (ok) {
              n = __ldg(other_sums + (size_t)lab[u] * (d + 1) + d);
              const int sc = selfcol ? selfcol[r] : -1;
              if (sc >= 0 && other_meta[sc].x == lab[u]) n -= 1.f;
            }
            const float wt = weight[r] * inv_t;
            coef[u] = n > 0.f ? wt / n : 0.f;
            if (lane == 0) beta_out[r] = coef[u];
          }
        }
      }
#pragma unroll
      for (int u = 0; u < kInFlight; ++u)
        if (lab[u] >= 0 && lab[u] < n_class) label_table_add(my_sum, my_cnt, d, lab[u], coef[u], x[u], lane);      // warp-uniform
    }
  }
  __syncthreads();
  label_tables_flush(s_sum, s_cnt, n_class, d, partial, cnt);
}

// Stage 2: out[k][c] (row stride d + 1; column d = count) = sum over blocks, fixed order.  A block owns 32 outputs;
// 8 partial-lanes per output, combined through shared memory.
__global__ void __launch_bounds__(256) p2p_label_reduce_kernel(const float* partial, const float* cnt, int n_blocks,
                                                               int n_class, int d, float* out) {
  pdl_trigger();
  pdl_wait();
  __shared__ float red[8][33];
  partial += (size_t)blockIdx.y * n_blocks * n_class * d;          // blockIdx.y = block-diagonal batch
  cnt += (size_t)blockIdx.y * n_blocks * n_class;
  out += (size_t)blockIdx.y * n_class * (d + 1);
  const int o = threadIdx.x & 31, pl = threadIdx.x >> 5;
  const int n_out = n_class * (d + 1);
  const int idx = blockIdx.x * 32 + o;
  float t = 0.f;
  if (idx < n_out) {
    const int k = idx / (d + 1), c = idx % (d + 1);
    const float* src = c < d ? partial + (size_t)k * d + c : cnt + k;
    const size_t stride = c < d ? (size_t)n_class * d : (size_t)n_class;
    float t4[4] = {0.f, 0.f, 0.f, 0.f};
    int b = pl;
    for (; b + 24 < n_blocks; b += 32) {
#pragma unroll
      for (int u = 0; u < 4; ++u) t4[u] += src[(size_t)(b + 8 * u) * stride];
    }
    for (; b < n_blocks; b += 8) t4[0] += src[(size_t)b * stride];
    t = (t4[0] + t4[1]) + (t4[2] + t4[3]);
  }
  red[pl][o] = t;
  __syncthreads();
  if (pl == 0 && idx < n_out) {
    float s = 0.f;
#pragma unroll
    for (int w = 0; w < 8; ++w) s += red[w][o];
    out[idx] = s;
  }
}

// Forward finish, LPR lanes per anchor i (fixed summation orders throughout).  The per-class sums
// label_sums[K][d + 1] (last column = class count) are read through L1 (a 5 KB table every warp shares).
//   Zs_i   = sum_slots zs - e_self                      e_self = exp(S_i,self / T - shift_i) if anchor i is a contrast row
//   P_raw  = a_i . Bsum[lab_i] - [labels agree] S_i,self        n_i = count[lab_i] - [labels agree]
//   block partial of  sum_i w_i (shift_i + log Zs_i - P_raw_i / (T n_i))                  (utils/loss.py:371-386)
// With alpha_out (the forward keeps state for the backward) it also writes the per-anchor constants
//   alpha~_i = w_i / (T Zs_i),   colshift_i = shift_i log2e - log2 alpha~_i
// (beta~ and ABsum do not depend on the sweep: p2p_label_part_kernel<true> on the side stream; the split partials of U
// stay where the sweep wrote them and are summed by the backward finish).
// The block that finishes last adds the per-block loss partials in index order (ticket counter `done`, zeroed by the
// first side-stream kernel of the call and wrapped back to zero by atomicInc), so the forward ends with this launch.
constexpr int kFinWarps = 8;           // warps per block of the forward finish
template <int LPR>
__global__ void __launch_bounds__(32 * kFinWarps) p2p_finish_fwd_kernel(const float* zs_partial, int n_slots, int n_rows, const float* shift,
                                                             const float* weight, float inv_t, const __nv_bfloat16* a,
                                                             const __nv_bfloat16* b, int d, const int2* a_meta,
                                                             const int2* b_meta, const int32_t* a_selfcol,
                                                             const float* label_sums, int n_class, int rows_per_batch,
                                                             float* alpha_out,
                                                             float* colshift_out, int n_rows_padded, float* stats,
                                                             double* loss_partial, unsigned int* done, float* loss) {
  pdl_trigger();
  pdl_wait();
  const bool keep = alpha_out != nullptr;
  if (keep && blockIdx.x == 0)
    for (int r = n_rows + threadIdx.x; r < n_rows_padded; r += 32 * kFinWarps) colshift_out[r] = kShiftOff;
  __shared__ double red[kFinWarps];
  __shared__ bool s_last;
  constexpr int kRpw = 32 / LPR, kFinRows = kRpw * kFinWarps;          // rows per warp, per block and pass
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, grp = lane / LPR, l8 = lane % LPR;
  const unsigned om = grp_mask<LPR>(lane);
  double acc = 0.0;
  for (int base = blockIdx.x * kFinRows; base < n_rows; base += gridDim.x * kFinRows) {
    const int i = base + warp * kRpw + grp;
    if (i >= n_rows) continue;                      // whole groups leave together
    const __nv_bfloat16* ai = a + (size_t)i * d;
    const int lab = a_meta[i].x;
    const int sc = a_selfcol ? a_selfcol[i] : -1;
    const bool lab_ok = lab >= 0 && lab < n_class;
    float zp = 0.f;
    for (int s = l8; s < n_slots; s += LPR) zp += zs_partial[(size_t)s * n_rows + i];
    float zs = grp_sum<LPR>(zp, om);
    float praw = 0.f, n = 0.f;
    if (lab_ok) {
      const float* bs = label_sums + ((size_t)(i / rows_per_batch) * n_class + lab) * (d + 1);      // the tables of anchor i's batch
      float t = 0.f;
      for (int c = l8 * 8; c < d; c += LPR * 8) {
        float x[8];
        bf16x8_to_float(*reinterpret_cast<const uint4*>(ai + c), x);
#pragma unroll
        for (int k = 0; k < 8; ++k) t = fmaf(x[k], __ldg(bs + c + k), t);
      }
      praw = grp_sum<LPR>(t, om);
      n = __ldg(bs + d);
    }
    if (sc >= 0) {
      const float s_self = grp_dot_bf16<LPR>(ai, b + (size_t)sc * d, d, l8, om);
      const float e_self = ex2_approx(fmaf(s_self, inv_t * kLog2e, -shift[i] * kLog2e));
      zs = fmaxf(zs - e_self, e_self * 1.1920929e-7f);      // round-off floor, see p2p_reduce_stats_self_kernel
      if (lab_ok && lab == b_meta[sc].x) { praw -= s_self; n -= 1.f; }      // (a label outside [0, K): n stays 0 -> NaN)
    }
    if (l8 == 0) {
      if (keep) {
        const float al = weight[i] * inv_t / zs;
        alpha_out[i] = al;
        colshift_out[i] = al > 0.f ? shift[i] * kLog2e - log2f(al) : kShiftOff;
      }
      stats[3 * i] = zs; stats[3 * i + 1] = praw; stats[3 * i + 2] = n;
      const float li = shift[i] + logf(zs) - (praw * inv_t) / n;      // n == 0 -> NaN, as 0/0 in the reference (:376-380)
      acc += (double)(weight[i] * li);
    }
  }
  __syncwarp();
  {          // the group leaders of the warp, in lane order
    double t = 0.0;
#pragma unroll
    for (int gl = 0; gl < 32; gl += LPR) t += __shfl_sync(0xffffffffu, acc, gl);
    acc = t;
  }
  if (lane == 0) red[warp] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
    for (int w = 0; w < kFinWarps; ++w) t += red[w];
    loss_partial[blockIdx.x] = t;
    __threadfence();
    s_last = atomicInc(done, gridDim.x - 1) == gridDim.x - 1;
  }
  __syncthreads();
  if (s_last && warp == 0) {
    __threadfence();
    double t = 0.0;
    for (int bidx = lane; bidx < (int)gridDim.x; bidx += 32) t += __ldcg(loss_partial + bidx);
    t = warp_sum(t);
    if (lane == 0) loss[0] = (float)t;
  }
}

// Backward finish, eight lanes per output row (anchors first, then contrast rows), g = dL/dloss:
//   d_a[i] = g ( alpha~_i U_i - beta~_i (Bsum[lab_i] - [labels agree] b_self) )
//   d_b[j] = g ( sum_splits Acc_j - bf16(alpha~_i e_i,self) a_i - ABsum[lab_j] + [labels agree] beta~_i a_i ),  i = b_selfrow[j]
template <int LPR>
__global__ void __launch_bounds__(256) p2p_finish_bwd_kernel(int n_anchor, int n_contrast, int d, int dim,
                                                             const __nv_bfloat16* a, const __nv_bfloat16* b, const int2* a_meta,
                                                             const int2* b_meta, const int32_t* a_selfcol,
                                                             const int32_t* b_selfrow, const float* label_sums,
                                                             const float* ab_sums, int n_class, int rows_per_batch_a,
                                                             int rows_per_batch_b, const float* alpha,
                                                             const float* beta, const float* colshift, const float* shift,
                                                             float scale_log2, const float* u_partial, int n_splits_u,
                                                             const float* acc_partial, int n_splits,
                                                             int fused_db, const float* grad_out, float* d_a, float* d_b) {
  pdl_trigger();
  pdl_wait();
  // fused_db: the dB sweep already wrote d_b = g (Acc - ABsum[lab_j]); only the self-pair term is left, and it is
  // added here by the lane group of the anchor it belongs to (ids are unique, so no two groups touch the same row)
  const float g = grad_out[0];
  constexpr int kRpw = 32 / LPR, kStep = LPR * 8;          // rows per warp; channels per pass of a group
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, grp = lane / LPR, l8 = lane % LPR;
  const unsigned om = grp_mask<LPR>(lane);
  const bool vec = (dim & 3) == 0;          // 16-byte stores: every 4-channel group is wholly inside or outside [0, dim)
  const int r_begin = (d_a || fused_db) ? 0 : n_anchor, r_end = (d_b && !fused_db) ? n_anchor + n_contrast : n_anchor;
  for (int r = r_begin + blockIdx.x * (8 * kRpw) + warp * kRpw + grp; r < r_end; r += gridDim.x * (8 * kRpw)) {
    if (r < n_anchor) {
      const int i = r;
      const int lab = a_meta[i].x;
      const bool lab_ok = lab >= 0 && lab < n_class;
      const int sc = a_selfcol ? a_selfcol[i] : -1;
      const bool match = sc >= 0 && lab_ok && lab == b_meta[sc].x;
      const float al = alpha[i], be = lab_ok ? beta[i] : 0.f;
      const __nv_bfloat16* bs = b + (size_t)max(sc, 0) * d;
      const float* bsum = label_sums + ((size_t)(i / rows_per_batch_a) * n_class + (lab_ok ? lab : 0)) * (d + 1);
      const __nv_bfloat16* ai = a + (size_t)i * d;
      const float s_self = sc >= 0 ? grp_dot_bf16<LPR>(ai, bs, d, l8, om) : 0.f;
      if (fused_db && sc >= 0) {
        const float g_self = bf16_round(ex2_approx(fmaf(s_self, scale_log2, -colshift[i])));
        const float coef = g * ((match ? beta[i] : 0.f) - g_self);
        for (int c = l8 * 8; c < dim; c += kStep) {
          float x[8];
          bf16x8_to_float(*reinterpret_cast<const uint4*>(ai + c), x);
          float* dst = d_b + (size_t)sc * dim + c;
          if (vec) {
#pragma unroll
            for (int h = 0; h < 2; ++h)
              if (c + 4 * h < dim) {
                float4 o = *reinterpret_cast<float4*>(dst + 4 * h);
                o.x = fmaf(coef, x[4 * h], o.x); o.y = fmaf(coef, x[4 * h + 1], o.y);
                o.z = fmaf(coef, x[4 * h + 2], o.z); o.w = fmaf(coef, x[4 * h + 3], o.w);
                *reinterpret_cast<float4*>(dst + 4 * h) = o;
              }
          } else {
#pragma unroll
            for (int k = 0; k < 8; ++k)
              if (c + k < dim) dst[k] = fmaf(coef, x[k], dst[k]);
          }
        }
      }
      if (d_a == nullptr) continue;
      // U_i = sum_splits U_partial - bf16(e_self) b_self   (the sweep multiplied bf16-rounded exponentials)
      const float e_self_r = sc >= 0 ? bf16_round(ex2_approx(fmaf(s_self, scale_log2, -shift[i] * kLog2e))) : 0.f;
      const size_t split_stride = (size_t)n_anchor * d;
      for (int c = l8 * 8; c < dim; c += kStep) {
        const float* src = u_partial + (size_t)i * d + c;
        float uu[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
        for (int s = 0; s < n_splits_u; ++s) {                // summed in split order
          const float4 p0 = *reinterpret_cast<const float4*>(src + (size_t)s * split_stride);
          const float4 p1 = *reinterpret_cast<const float4*>(src + (size_t)s * split_stride + 4);
          uu[0] += p0.x; uu[1] += p0.y; uu[2] += p0.z; uu[3] += p0.w;
          uu[4] += p1.x; uu[5] += p1.y; uu[6] += p1.z; uu[7] += p1.w;
        }
        float x[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
        if (sc >= 0) bf16x8_to_float(*reinterpret_cast<const uint4*>(bs + c), x);
        float o[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) {
          const float u = fmaf(-e_self_r, x[k], uu[k]);
          float pk = lab_ok ? __ldg(bsum + c + k) : 0.f;
          if (match) pk -= x[k];
          o[k] = g * (al * u - be * pk);
        }
        float* dst = d_a + (size_t)i * dim + c;
        if (vec) {
          if (c < dim) *reinterpret_cast<float4*>(dst) = make_float4(o[0], o[1], o[2], o[3]);
          if (c + 4 < dim) *reinterpret_cast<float4*>(dst + 4) = make_float4(o[4], o[5], o[6], o[7]);
        } else {
#pragma unroll
          for (int k = 0; k < 8; ++k)
            if (c + k < dim) dst[k] = o[k];
        }
      }
    } else {
      const int j = r - n_anchor;
      const int lab = b_meta[j].x;
      const bool lab_ok = lab >= 0 && lab < n_class;
      const int i = b_selfrow ? b_selfrow[j] : -1;
      float g_self = 0.f, be_self = 0.f;
      const __nv_bfloat16* as = a + (size_t)max(i, 0) * d;
      if (i >= 0) {
        const float s_self = grp_dot_bf16<LPR>(as, b + (size_t)j * d, d, l8, om);
        g_self = bf16_round(ex2_approx(fmaf(s_self, scale_log2, -colshift[i])));
        if (a_meta[i].x == lab) be_self = beta[i];
      }
      const float* absum = ab_sums + ((size_t)(j / rows_per_batch_b) * n_class + (lab_ok ? lab : 0)) * (d + 1);
      for (int c = l8 * 8; c < dim; c += kStep) {
        float t[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
        for (int s = 0; s < n_splits; ++s) {
          const float* src = acc_partial + ((size_t)s * n_contrast + j) * d + c;
          const float4 p0 = *reinterpret_cast<const float4*>(src), p1 = *reinterpret_cast<const float4*>(src + 4);
          t[0] += p0.x; t[1] += p0.y; t[2] += p0.z; t[3] += p0.w;
          t[4] += p1.x; t[5] += p1.y; t[6] += p1.z; t[7] += p1.w;
        }
        float x[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
        if (i >= 0) bf16x8_to_float(*reinterpret_cast<const uint4*>(as + c), x);
        float o[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) {
          float tk = t[k];
          if (lab_ok) tk -= __ldg(absum + c + k);
          tk += (be_self - g_self) * x[k];          // x = 0 without a self pair
          o[k] = g * tk;
        }
        float* dst = d_b + (size_t)j * dim + c;
        if (vec) {
          if (c < dim) *reinterpret_cast<float4*>(dst) = make_float4(o[0], o[1], o[2], o[3]);
          if (c + 4 < dim) *reinterpret_cast<float4*>(dst + 4) = make_float4(o[4], o[5], o[6], o[7]);
        } else {
#pragma unroll
          for (int k = 0; k < 8; ++k)
            if (c + k < dim) dst[k] = o[k];
        }
      }
    }
  }
}

// ------------------------------ host side ----------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  }
  return fn;
}

// [rows, d] bf16 row-major, box = 64 elements (128 B) x box_rows, 128-byte swizzle, OOB rows read as zero
int make_map(CUtensorMap* m, const void* ptr, int64_t rows, int64_t d, int box_rows) {
  ensure_context_on_this_thread();
  EncodeTiledFn fn = encode_fn();
  if (!fn) return SLCL_ERR_CUDA;
  cuuint64_t dims[2] = {(cuuint64_t)d, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)d * 2};
  cuuint32_t box[2] = {(cuuint32_t)KCH, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(ptr), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    char what[160];
    snprintf(what, sizeof(what), "cuTensorMapEncodeTiled(rows=%lld, d=%lld, box_rows=%d, ptr%%16=%d, CUresult=%d)", (long long)rows,
             (long long)d, box_rows, (int)(reinterpret_cast<uintptr_t>(ptr) & 15), (int)r);
    set_cuda_error(cudaErrorInvalidValue, what);
    return SLCL_ERR_CUDA;
  }
  return SLCL_OK;
}

struct Sweep { int row_tiles, splits, cols_per_split, cluster; };

Sweep plan_sweep(int64_t n_rows, int64_t n_cols, int n_batch = 1, bool tail_split = false) {          // sizes are per batch
  Sweep s;
  s.row_tiles = (int)ceil_div<int64_t>(n_rows, BM);
  int col_tiles = (int)ceil_div<int64_t>(n_cols, BN);
  const int n_sm = sm_count(), R = s.row_tiles * n_batch;
  int want = max(1, n_sm / R);      // fill the SMs: batches x row tiles x column splits ~ #SMs
  s.splits = min(want, col_tiles);
  int tiles_per_split = ceil_div(col_tiles, s.splits);
  s.splits = ceil_div(col_tiles, tiles_per_split);
  // Uneven tail: R x want CTAs leave SMs idle (cfg3: 32 x 4 = 128 of 148).  One more, SHORT split per row tile puts them to
  // work: the long CTAs (launched first: blockIdx.y < want) shrink from ceil(T / want) to tp column tiles, the R short ones
  // take the remaining T - want tp tiles each and run on the (n_sm - R want) free SMs, in rounds.  tp is the smallest
  // value for which the rounds of short CTAs end before the long ones (kFixed ~ set-up + drain of a CTA in tile-steps).
  // Measured at cfg3: general sweeps 160 -> 155 us; the ANALYTIC forward gets slower (48 -> 52 us, 70 -> 76 us with U):
  // its table kernels run on the side stream and want those idle SMs, and a fifth split adds partial traffic -- so only
  // the general sweeps ask for it (tail_split).
  static const bool uneven = [] { const char* e = getenv("SLCL_P2P_UNEVEN"); return !(e && atoi(e) == 0); }();
  constexpr int kFixed = 7;
  if (tail_split && uneven && want >= 2 && s.splits == want && R * want < n_sm && col_tiles > 2 * want) {
    const int free_sms = n_sm - R * want, rounds = ceil_div(R, free_sms);
    for (int tp = ceil_div(col_tiles, want + 1); tp < tiles_per_split; ++tp) {
      const int tail = col_tiles - want * tp;
      if (tail < 1) break;
      if (rounds * (tail + kFixed) <= tp + kFixed) { tiles_per_split = tp; s.splits = want + 1; break; }
    }
  }
  s.cols_per_split = tiles_per_split * BN;
  // Cluster size of the multicast variant (1, 2 or 4 CTAs along the row tiles share every column tile).
  s.cluster = 1;
  { const char* e = getenv("SLCL_P2P_CLUSTER"); if (e) s.cluster = atoi(e) == 4 ? 4 : (atoi(e) == 2 ? 2 : 1); }
  return s;
}

// fp32 output of the MMA2 drain as a 3-D tensor [splits][rows][ld]: box = 32 columns (128 B) x 32 rows, 128-byte swizzle;
// rows past n_rows and columns past n_cols are clipped by the TMA unit
int make_out_map(CUtensorMap* m, const float* ptr, int64_t n_cols, int64_t ld, int64_t rows, int64_t splits) {
  ensure_context_on_this_thread();
  EncodeTiledFn fn = encode_fn();
  if (!fn) return SLCL_ERR_CUDA;
  cuuint64_t dims[3] = {(cuuint64_t)n_cols, (cuuint64_t)rows, (cuuint64_t)splits};
  cuuint64_t strides[2] = {(cuuint64_t)ld * 4, (cuuint64_t)rows * ld * 4};
  cuuint32_t box[3] = {32, 32, 1};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = fn(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<float*>(ptr), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    char what[200];
    snprintf(what, sizeof(what), "cuTensorMapEncodeTiled(out: cols=%lld, ld=%lld, rows=%lld, splits=%lld, ptr%%16=%d, CUresult=%d)",
             (long long)n_cols, (long long)ld, (long long)rows, (long long)splits, (int)(reinterpret_cast<uintptr_t>(ptr) & 15), (int)r);
    set_cuda_error(cudaErrorInvalidValue, what);
    return SLCL_ERR_CUDA;
  }
  return SLCL_OK;
}

template <int CS, int MODE>
int launch_one(const CUtensorMap& mr, const CUtensorMap& mc, const CUtensorMap& mo, const P2PArgs& a, const Sweep& sw, size_t smem,
               int n_batch, cudaStream_t stream) {
  static bool attr_set_dev[64] = {};     // per instantiation and per device (function attributes are per device)
  bool& attr_set = attr_set_dev[current_device_slot()];
  if (!attr_set) {
    cudaError_t e = cudaFuncSetAttribute(p2p_kernel<CS, MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_bytes_for(kMaxD));
    if (e != cudaSuccess) { set_cuda_error(e, "cudaFuncSetAttribute(p2p_kernel)"); return SLCL_ERR_CUDA; }
    attr_set = true;
  }
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3((unsigned)(ceil_div(sw.row_tiles, CS) * CS), (unsigned)sw.splits, (unsigned)n_batch);
  cfg.blockDim = dim3(kThreads, 1, 1);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cudaLaunchAttribute attr[2];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = (unsigned)CS;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[1].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 2;
  cudaError_t le = cudaLaunchKernelEx(&cfg, p2p_kernel<CS, MODE>, mr, mc, mo, a);
  if (le != cudaSuccess) { set_cuda_error(le, "cudaLaunchKernelEx(p2p_kernel)"); return SLCL_ERR_CUDA; }
  return check_launch("p2p_kernel");
}

template <int MODE>
int launch_sweep(const void* rows, int64_t n_rows, const void* cols, int64_t n_cols, int d, float inv_t, P2PArgs a,
                 const Sweep& sw, cudaStream_t stream, int n_batch = 1) {
  CUtensorMap mr, mc, mo;
  int st = make_map(&mr, rows, n_rows, d, BM);
  if (st != SLCL_OK) return st;
  st = make_map(&mc, cols, n_cols, d, BN / sw.cluster);
  if (st != SLCL_OK) return st;
  if (ModeTraits<MODE>::kMma2) {
    st = a.fused_out ? make_out_map(&mo, a.fused_out, a.ld_out, a.ld_out, n_rows, 1)
                     : make_out_map(&mo, a.grad_partial, d, d, n_rows, sw.splits);
    if (st != SLCL_OK) return st;
  } else {
    mo = mc;          // unused
  }
  a.n_rows = (int)n_rows; a.n_cols = (int)n_cols; a.d = d;
  a.rows_per_batch = (int)(n_rows / n_batch); a.cols_per_batch = (int)(n_cols / n_batch);
  a.cols_per_split = sw.cols_per_split;
  a.scale_log2 = inv_t * kLog2e;
  a.rows_u32 = reinterpret_cast<const uint32_t*>(rows);
#ifdef SLCL_P2P_PROFILE
  { const char* e = getenv("SLCL_P2P_PROF"); a.prof = e ? reinterpret_cast<unsigned long long*>(strtoull(e, nullptr, 0)) : nullptr; }
#endif
  const size_t smem = smem_bytes_for(d);
  if (sw.cluster == 4) return launch_one<4, MODE>(mr, mc, mo, a, sw, smem, n_batch, stream);
  if (sw.cluster == 2) return launch_one<2, MODE>(mr, mc, mo, a, sw, smem, n_batch, stream);
  return launch_one<1, MODE>(mr, mc, mo, a, sw, smem, n_batch, stream);
}

// State the analytic forward leaves for the backward (slcl_p2p_state_bytes): one caller-owned buffer.
struct P2PState {
  float* u;          // [splits][Na][d]  split partials of U_i = sum_j exp(S_ij - shift_i) b_j, as the forward sweep wrote them
                     //                  (splits <= max_splits(Na); summed, and the self pair removed, by the backward finish)
  float* bsum;       // [K][d+1]       per-class sums / counts of the contrast rows
  float* absum;      // [K][d+1]       sum_{lab_i = k} beta~_i a_i
  float* colshift;   // [pad64(Na)]    column shifts of the dB sweep
  float* alpha;      // [Na]
  float* beta;       // [Na]
  size_t total;
};
int max_splits(int64_t n_rows) {          // upper bound of plan_sweep(n_rows, any).splits (+1: the uneven tail split)
  return max(1, sm_count() / (int)ceil_div<int64_t>(n_rows, BM)) + 1;
}
P2PState carve_state(void* p, int64_t na, int d) {
  size_t off = 0;
  auto take = [&](size_t bytes) { size_t o = off; off += align_up(bytes, 256); return o; };
  const size_t K = kMaxLabelClasses * (size_t)ceil_div<int64_t>(na, BM);      // per-class tables for every possible block-diagonal batch
  size_t o0 = take((size_t)max_splits(na) * na * d * sizeof(float)), o1 = take(K * (d + 1) * sizeof(float)), o2 = take(K * (d + 1) * sizeof(float));
  size_t o3 = take(align_up((size_t)na, BN) * sizeof(float)), o4 = take((size_t)na * sizeof(float)), o5 = take((size_t)na * sizeof(float));
  char* b = reinterpret_cast<char*>(p);
  P2PState st;
  st.u = reinterpret_cast<float*>(b + o0); st.bsum = reinterpret_cast<float*>(b + o1); st.absum = reinterpret_cast<float*>(b + o2);
  st.colshift = reinterpret_cast<float*>(b + o3); st.alpha = reinterpret_cast<float*>(b + o4); st.beta = reinterpret_cast<float*>(b + o5);
  st.total = off;
  return st;
}

// workspace layout (one carve-up serves the general and the analytic path)
constexpr int kMaxFinishBlocks = 1024;
struct P2PWs {
  float* stat_partial;     // [2*splits_a][Na][3]
  float4* anchor_stat;     // general: [pad64(Na)]
  float* grad_partial_a;   // [splits_a][Na][d]   (general dA sweep / analytic U)
  float* grad_partial_b;   // [splits_b][M][d]
  float* lab_partial_b;    // analytic: [blocks_b][K][d], cnt [blocks_b][K]
  float* lab_cnt_b;
  float* ab_partial;       // [kMaxFinishBlocks][K][d], cnt [kMaxFinishBlocks][K]
  float* ab_cnt;
  float* bsum;             // [K][d+1]   (forward without state)
  float* stats_scratch;    // [Na][3]    (backward without state)
  float* gself;            // [Na]       (general sweeps with self maps)
  unsigned int* done;      // ticket counter of the forward finish
  double* loss_partial;    // [max(kMaxFinishBlocks, ceil(Na / 8))]
  void* state;             // backward without state: regenerated here
  int blocks_b;
  size_t total;
};

P2PWs carve(void* ws, int64_t na, int64_t m, int d) {
  Sweep sa = plan_sweep(na, m), sb = plan_sweep(m, na);
  size_t off = 0;
  auto take = [&](size_t bytes) { size_t o = off; off += align_up(bytes, 256); return o; };
  P2PWs w;
  w.blocks_b = (int)(ceil_div<int64_t>(m, kLabelRowsPerBlock) + ceil_div<int64_t>(m, BM));      // + one ragged block per batch
  const size_t K = kMaxLabelClasses;
  const size_t ab_blocks = (size_t)std::max<int64_t>(kMaxFinishBlocks, ceil_div<int64_t>(na, BM));
  size_t o[14];
  const size_t spa = (size_t)std::max(sa.splits, max_splits(na)), spb = (size_t)std::max(sb.splits, max_splits(m));      // any batching
  o[0] = take((size_t)2 * spa * na * 3 * sizeof(float));
  o[1] = take((size_t)align_up((size_t)na, BN) * sizeof(float4));
  o[2] = take(spa * na * d * sizeof(float));
  o[3] = take(spb * m * d * sizeof(float));
  o[4] = take((size_t)w.blocks_b * K * d * sizeof(float));
  o[5] = take((size_t)w.blocks_b * K * sizeof(float));
  o[6] = take(ab_blocks * K * d * sizeof(float));
  o[7] = take(ab_blocks * K * sizeof(float));
  o[8] = take(K * (size_t)ceil_div<int64_t>(na, BM) * (d + 1) * sizeof(float));
  o[9] = take((size_t)na * 3 * sizeof(float));
  const int64_t n_loss_partial = ceil_div<int64_t>(na, 8) > kMaxFinishBlocks ? ceil_div<int64_t>(na, 8) : kMaxFinishBlocks;
  o[10] = take((size_t)n_loss_partial * sizeof(double));
  o[11] = take(carve_state(nullptr, na, d).total);
  o[12] = take((size_t)na * sizeof(float));
  o[13] = take(sizeof(unsigned int));
  char* b = reinterpret_cast<char*>(ws);
  w.stat_partial = reinterpret_cast<float*>(b + o[0]);
  w.anchor_stat = reinterpret_cast<float4*>(b + o[1]);
  w.grad_partial_a = reinterpret_cast<float*>(b + o[2]);
  w.grad_partial_b = reinterpret_cast<float*>(b + o[3]);
  w.lab_partial_b = reinterpret_cast<float*>(b + o[4]);
  w.lab_cnt_b = reinterpret_cast<float*>(b + o[5]);
  w.ab_partial = reinterpret_cast<float*>(b + o[6]);
  w.ab_cnt = reinterpret_cast<float*>(b + o[7]);
  w.bsum = reinterpret_cast<float*>(b + o[8]);
  w.stats_scratch = reinterpret_cast<float*>(b + o[9]);
  w.loss_partial = reinterpret_cast<double*>(b + o[10]);
  w.state = b + o[11];
  w.gself = reinterpret_cast<float*>(b + o[12]);
  w.done = reinterpret_cast<unsigned int*>(b + o[13]);
  w.total = off;
  return w;
}

bool p2p_args_ok(const void* a, const void* b, int64_t na, int64_t m, int64_t dp) {
  return a && b && na > 0 && m > 0 && dp >= KCH && dp <= kMaxD && dp % KCH == 0 && na < (int64_t)INT_MAX - BM &&
         m < (int64_t)INT_MAX - BM && aligned16(a) && aligned16(b);
}

// block-diagonal batching: equal batches whose row / column ranges are whole tiles
bool batches_ok(int64_t na, int64_t m, int n_class, int n_batch) {
  if (n_batch == 1) return true;
  (void)n_class;
  return n_batch > 1 && n_batch <= 65535 && na % n_batch == 0 && m % n_batch == 0 && (na / n_batch) % BM == 0 &&
         (m / n_batch) % BM == 0;
}

int finish_blocks(int64_t rows, int lpr) {          // forward finish: lpr lanes per anchor up to kMaxFinishBlocks partials
  const int64_t want = ceil_div<int64_t>(rows, (32 / lpr) * kFinWarps);
  return (int)(want < kMaxFinishBlocks ? want : kMaxFinishBlocks);
}

int big_smem_ok() {          // K = 8, d = 256 needs 64 KB of dynamic shared memory (> the 48 KB default)
  static bool done_dev[64] = {};
  bool& done = done_dev[current_device_slot()];
  if (!done) {
    const int bytes = (int)(8 * kMaxLabelClasses * (kMaxD + 1) * sizeof(float));
    cudaError_t e = cudaFuncSetAttribute(p2p_label_part_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(p2p_label_part_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
    if (e != cudaSuccess) { set_cuda_error(e, "cudaFuncSetAttribute(p2p label tables)"); return SLCL_ERR_CUDA; }
    done = true;
  }
  return SLCL_OK;
}

// Side stream for work that does not depend on the sweep (the per-class sums of the contrast rows): it runs on the
// SMs the sweep leaves idle.  One stream + two events per host thread and device, created on first use; the fork
// and the join are ordinary event dependencies, so they are captured into CUDA graphs like any other edge.
struct Aux { cudaStream_t s = nullptr; cudaEvent_t fork = nullptr, join = nullptr; };
Aux* aux_stream() {
  static thread_local Aux cache[64];
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return nullptr;
  Aux& x = cache[dev];
  if (x.s == nullptr) {
    if (cudaStreamCreateWithFlags(&x.s, cudaStreamNonBlocking) != cudaSuccess ||
        cudaEventCreateWithFlags(&x.fork, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&x.join, cudaEventDisableTiming) != cudaSuccess) {
      x.s = nullptr;
      cudaGetLastError();
      return nullptr;
    }
  }
  return &x;
}

// analytic forward: [side stream: label sums of b -> beta~ and ABsum of the anchors]  ||  sweep  ->  finish (+ loss)
int ana_forward(const void* a, const void* b, int64_t na, int64_t m, int d, const int2* am, const int2* bm,
                const int32_t* a_selfcol, int n_class, const float* shift, const float* weight, float inv_t,
                float* stats, float* loss, const P2PState* state, const P2PWs& w, cudaStream_t stream, int n_batch = 1) {
  const int rpb_a = (int)(na / n_batch), rpb_b = (int)(m / n_batch);          // rows per block-diagonal batch
  const int blocks_b = ceil_div(rpb_b, kLabelRowsPerBlock);
  const __nv_bfloat16* ab = reinterpret_cast<const __nv_bfloat16*>(a);
  const __nv_bfloat16* bb = reinterpret_cast<const __nv_bfloat16*>(b);
  if (int st0 = big_smem_ok()) return st0;
  const bool keep = state != nullptr;
  float* bsum = keep ? state->bsum : w.bsum;
  const size_t table_smem = (size_t)8 * n_class * (d + 1) * sizeof(float);
  const int n_red = ceil_div(n_class * (d + 1), 32);
  Aux* aux = aux_stream();
  cudaStream_t side = stream;
  if (aux != nullptr && cudaEventRecord(aux->fork, stream) == cudaSuccess && cudaStreamWaitEvent(aux->s, aux->fork, 0) == cudaSuccess)
    side = aux->s;
  launch_pdl(p2p_label_part_kernel<false>, dim3(blocks_b, n_batch), dim3(256), table_smem, side, bb, rpb_b, d, bm, n_class,
             w.lab_partial_b, w.lab_cnt_b, (const float*)nullptr, 0.f, (const int32_t*)nullptr, (const int2*)nullptr,
             (const float*)nullptr, (float*)nullptr, w.done);
  launch_pdl(p2p_label_reduce_kernel, dim3(n_red, n_batch), dim3(256), 0, side, (const float*)w.lab_partial_b,
             (const float*)w.lab_cnt_b, blocks_b, n_class, d, bsum);
  if (keep) {
    const int blocks_a = (int)std::max<int64_t>(1, std::min<int64_t>(ceil_div<int64_t>(rpb_a, kLabelRowsPerBlock),
                                                                     (int64_t)kMaxFinishBlocks / n_batch));
    launch_pdl(p2p_label_part_kernel<true>, dim3(blocks_a, n_batch), dim3(256), table_smem, side, ab, rpb_a, d, am, n_class,
               w.ab_partial, w.ab_cnt, weight, inv_t, a_selfcol, bm, (const float*)bsum, state->beta, (unsigned int*)nullptr);
    launch_pdl(p2p_label_reduce_kernel, dim3(n_red, n_batch), dim3(256), 0, side, (const float*)w.ab_partial,
               (const float*)w.ab_cnt, blocks_a, n_class, d, state->absum);
  }
  if (side != stream) cudaEventRecord(aux->join, side);
  Sweep sw = plan_sweep(na / n_batch, m / n_batch, n_batch);
  P2PArgs args{};
  args.row_shift = shift;
  args.stat_partial = w.stat_partial;
  args.grad_partial = keep ? state->u : w.grad_partial_a;
  int st = keep ? launch_sweep<kAnaFwdU>(a, na, b, m, d, inv_t, args, sw, stream, n_batch)
                : launch_sweep<kAnaFwd>(a, na, b, m, d, inv_t, args, sw, stream, n_batch);
  if (side != stream) cudaStreamWaitEvent(stream, aux->join, 0);          // join even when the sweep failed to launch
  if (st != SLCL_OK) return st;
  const int lpr = lanes_per_row(d), nb = finish_blocks(na, lpr);
  auto fin = [&](auto kernel) {
    launch_pdl(kernel, dim3(nb), dim3(32 * kFinWarps), 0, stream, (const float*)w.stat_partial, 2 * sw.splits, (int)na, shift,
               weight, inv_t, ab, bb, d, am, bm, a_selfcol, (const float*)bsum, n_class, rpb_a,
               keep ? state->alpha : (float*)nullptr, keep ? state->colshift : (float*)nullptr, (int)align_up((size_t)na, BN),
               stats, w.loss_partial, w.done, loss);
  };
  if (lpr == 8) fin(p2p_finish_fwd_kernel<8>); else if (lpr == 16) fin(p2p_finish_fwd_kernel<16>); else fin(p2p_finish_fwd_kernel<32>);
  return SLCL_OK;
}

}  // namespace
}  // namespace slcl

using namespace slcl;

extern "C" size_t slcl_p2p_workspace_bytes(int64_t n_anchor, int64_t n_contrast, int64_t dim_padded) {
  if (n_anchor <= 0 || n_contrast <= 0 || dim_padded <= 0 || dim_padded > kMaxD) return 0;
  return carve(nullptr, n_anchor, n_contrast, (int)dim_padded).total;
}

extern "C" size_t slcl_p2p_state_bytes(int64_t n_anchor, int64_t dim_padded) {
  if (n_anchor <= 0 || dim_padded <= 0 || dim_padded > kMaxD) return 0;
  return carve_state(nullptr, n_anchor, (int)dim_padded).total;
}

extern "C" int slcl_p2p_state_layout(int64_t n_anchor, int64_t dim_padded, int64_t* offsets_host) {
  if (n_anchor <= 0 || dim_padded <= 0 || dim_padded > kMaxD || dim_padded % KCH || !offsets_host) return SLCL_ERR_INVALID_ARGUMENT;
  const P2PState s = carve_state(nullptr, n_anchor, (int)dim_padded);
  const float* f[6] = {s.u, s.bsum, s.absum, s.colshift, s.alpha, s.beta};
  for (int i = 0; i < 6; ++i) offsets_host[i] = (int64_t)reinterpret_cast<uintptr_t>(f[i]);
  offsets_host[6] = (int64_t)s.total;
  return SLCL_OK;
}

namespace slcl {
namespace {
// Backward state of the dB sweep over the anchors of all ranks: per-anchor constants as gathered (colshift padded with the
// switch-off shift), ABsum = sum of the ranks' tables in rank order (identical bits on every rank).  n_tab covers the
// tables of every block-diagonal batch ([n_batch][K][d+1], contiguous in the parts and in the state alike).
__global__ void __launch_bounds__(256) p2p_state_assemble_kernel(int n_anchor, int n_padded, int n_tab, const float* alpha,
                                                                 const float* beta, const float* colshift, const float* absum_parts,
                                                                 int n_parts, float* st_alpha, float* st_beta,
                                                                 float* st_colshift, float* st_absum) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n_padded || i < n_tab; i += gridDim.x * blockDim.x) {
    if (i < n_anchor) { st_alpha[i] = alpha[i]; st_beta[i] = beta[i]; }
    if (i < n_padded) st_colshift[i] = i < n_anchor ? colshift[i] : kShiftOff;
    if (i < n_tab) {
      float t = 0.f;
      for (int p = 0; p < n_parts; ++p) t += absum_parts[(size_t)p * n_tab + i];
      st_absum[i] = t;
    }
  }
}
}  // namespace
}  // namespace slcl

extern "C" int slcl_p2p_state_assemble_batched(void* bwd_state, int64_t n_anchor, int64_t dim_padded, int n_class, int n_batch,
                                               const float* alpha, const float* beta, const float* colshift,
                                               const float* absum_parts, int n_parts, slcl_stream_t stream_) {
  if (!bwd_state || !aligned16(bwd_state) || !alpha || !beta || !colshift || !absum_parts || n_anchor <= 0 ||
      n_anchor >= (int64_t)INT_MAX - BM || dim_padded <= 0 || dim_padded > kMaxD || dim_padded % KCH || n_class < 1 ||
      n_class > kMaxLabelClasses || n_parts < 1 || n_batch < 1)
    return SLCL_ERR_INVALID_ARGUMENT;
  // the state holds one table per possible batch of whole 128-row tiles (carve_state)
  if (n_batch > 1 && (n_anchor % n_batch || (n_anchor / n_batch) % BM)) return SLCL_ERR_INVALID_ARGUMENT;
  const int d = (int)dim_padded;
  P2PState s = carve_state(bwd_state, n_anchor, d);
  const int64_t n_padded = (int64_t)align_up((size_t)n_anchor, BN), n_tab = (int64_t)n_batch * n_class * (d + 1);
  const int64_t n = n_padded > n_tab ? n_padded : n_tab;
  if (n >= (int64_t)INT_MAX - 256) return SLCL_ERR_INVALID_ARGUMENT;
  p2p_state_assemble_kernel<<<(unsigned)ceil_div<int64_t>(n, 256), 256, 0, (cudaStream_t)stream_>>>(
      (int)n_anchor, (int)n_padded, (int)n_tab, alpha, beta, colshift, absum_parts, n_parts, s.alpha, s.beta, s.colshift,
      s.absum);
  return check_launch("slcl_p2p_state_assemble");
}

extern "C" int slcl_p2p_state_assemble(void* bwd_state, int64_t n_anchor, int64_t dim_padded, int n_class, const float* alpha,
                                       const float* beta, const float* colshift, const float* absum_parts, int n_parts,
                                       slcl_stream_t stream_) {
  return slcl_p2p_state_assemble_batched(bwd_state, n_anchor, dim_padded, n_class, 1, alpha, beta, colshift, absum_parts,
                                         n_parts, stream_);
}

extern "C" int slcl_p2p_fwd(const void* a_bf16, const void* b_bf16, int64_t n_anchor, int64_t n_contrast, int64_t dim_padded,
                            const int32_t* a_meta, const int32_t* b_meta, const int32_t* a_selfcol, int n_class, int n_batch,
                            const float* shift, const float* weight, float temperature, float* stats, float* loss,
                            void* bwd_state, void* workspace, size_t workspace_bytes, slcl_stream_t stream_) {
  if (!p2p_args_ok(a_bf16, b_bf16, n_anchor, n_contrast, dim_padded) || !a_meta || !b_meta || !shift || !weight || !stats ||
      !loss || !workspace || !(temperature > 0.f) || n_class < 0 || n_class > kMaxLabelClasses)
    return SLCL_ERR_INVALID_ARGUMENT;
  if (n_class == 0 && bwd_state) return SLCL_ERR_INVALID_ARGUMENT;
  if (bwd_state && !aligned16(bwd_state)) return SLCL_ERR_INVALID_ARGUMENT;
  if (!batches_ok(n_anchor, n_contrast, n_class, n_batch)) return SLCL_ERR_INVALID_ARGUMENT;
  const int d = (int)dim_padded;
  if (workspace_bytes < slcl_p2p_workspace_bytes(n_anchor, n_contrast, dim_padded) || !aligned16(workspace))
    return SLCL_ERR_WORKSPACE;
  cudaStream_t stream = (cudaStream_t)stream_;
  P2PWs w = carve(workspace, n_anchor, n_contrast, d);
  const float inv_t = 1.0f / temperature;
  const int na = (int)n_anchor;
  const int2* am = reinterpret_cast<const int2*>(a_meta);
  const int2* bm = reinterpret_cast<const int2*>(b_meta);
  if (n_class > 0) {
    P2PState st_ = carve_state(bwd_state, n_anchor, d);
    int st = ana_forward(a_bf16, b_bf16, n_anchor, n_contrast, d, am, bm, a_selfcol, n_class, shift, weight, inv_t, stats, loss,
                         bwd_state ? &st_ : nullptr, w, stream, n_batch);
    if (st != SLCL_OK) return st;
    return check_launch("slcl_p2p_fwd");
  }
  Sweep sw = plan_sweep(n_anchor / n_batch, n_contrast / n_batch, n_batch, true);
  P2PArgs args{};
  args.row_meta = am; args.col_meta = bm; args.row_shift = shift; args.stat_partial = w.stat_partial;
  args.self_by_id = a_selfcol == nullptr;
  int st = launch_sweep<kGenFwd>(a_bf16, n_anchor, b_bf16, n_contrast, d, inv_t, args, sw, stream, n_batch);
  if (st != SLCL_OK) return st;
  int nb;
  if (a_selfcol == nullptr) {
    nb = ceil_div(na, 256);
    launch_pdl(p2p_reduce_stats_kernel, dim3(nb), dim3(256), 0, stream, w.stat_partial, 2 * sw.splits, na, shift, weight, inv_t,
               stats, w.loss_partial);
  } else {
    nb = ceil_div(na, 8);
    launch_pdl(p2p_reduce_stats_self_kernel, dim3(nb), dim3(256), 0, stream, (const float*)w.stat_partial, 2 * sw.splits, na, shift,
               weight, inv_t, reinterpret_cast<const __nv_bfloat16*>(a_bf16), reinterpret_cast<const __nv_bfloat16*>(b_bf16), d, am,
               bm, a_selfcol, stats, w.loss_partial);
  }
  launch_pdl(p2p_loss_kernel, dim3(1), dim3(256), 0, stream, w.loss_partial, nb, loss);
  return check_launch("slcl_p2p_fwd");
}

extern "C" int slcl_p2p_bwd(const void* a_bf16, const void* b_bf16, int64_t n_anchor, int64_t n_contrast, int64_t dim_padded,
                            int64_t dim, const int32_t* a_meta, const int32_t* b_meta, const int32_t* a_selfcol,
                            const int32_t* b_selfrow, int n_class, int n_batch, const float* shift, const float* weight,
                            float temperature, const float* stats, const void* bwd_state, const float* grad_out, float* d_a,
                            float* d_b, void* workspace, size_t workspace_bytes, slcl_stream_t stream_) {
  if (!p2p_args_ok(a_bf16, b_bf16, n_anchor, n_contrast, dim_padded) || !a_meta || !b_meta || !shift || !weight || !stats ||
      !grad_out || !workspace || !(temperature > 0.f) || dim <= 0 || dim > dim_padded || (!d_a && !d_b) || n_class < 0 ||
      n_class > kMaxLabelClasses)
    return SLCL_ERR_INVALID_ARGUMENT;
  if ((a_selfcol == nullptr) != (b_selfrow == nullptr)) return SLCL_ERR_INVALID_ARGUMENT;
  if (n_class == 0 && bwd_state) return SLCL_ERR_INVALID_ARGUMENT;
  if (!batches_ok(n_anchor, n_contrast, n_class, n_batch)) return SLCL_ERR_INVALID_ARGUMENT;
  if (bwd_state && !aligned16(bwd_state)) return SLCL_ERR_INVALID_ARGUMENT;
  const int d = (int)dim_padded;
  if (workspace_bytes < slcl_p2p_workspace_bytes(n_anchor, n_contrast, dim_padded) || !aligned16(workspace))
    return SLCL_ERR_WORKSPACE;
  cudaStream_t stream = (cudaStream_t)stream_;
  P2PWs w = carve(workspace, n_anchor, n_contrast, d);
  const float inv_t = 1.0f / temperature;
  const int na = (int)n_anchor;
  const int2* am = reinterpret_cast<const int2*>(a_meta);
  const int2* bm = reinterpret_cast<const int2*>(b_meta);
  if (n_class > 0) {
    const __nv_bfloat16* ab = reinterpret_cast<const __nv_bfloat16*>(a_bf16);
    const __nv_bfloat16* bb = reinterpret_cast<const __nv_bfloat16*>(b_bf16);
    P2PState st_ = carve_state(const_cast<void*>(bwd_state ? bwd_state : w.state), n_anchor, d);
    if (bwd_state == nullptr) {
      // the caller did not keep the forward's state: one more forward sweep regenerates it in the workspace
      int st = ana_forward(a_bf16, b_bf16, n_anchor, n_contrast, d, am, bm, a_selfcol, n_class, shift, weight, inv_t,
                           w.stats_scratch, reinterpret_cast<float*>(w.loss_partial) /* scratch */, &st_, w, stream, n_batch);
      if (st != SLCL_OK) return st;
    }
    int n_splits_b = 0, fused_db = 0;
    if (d_b) {
      Sweep sw = plan_sweep(n_contrast / n_batch, n_anchor / n_batch, n_batch);
      P2PArgs args{};
      args.col_shift = st_.colshift;
      args.grad_partial = w.grad_partial_b;
      if (sw.splits == 1 && dim % 4 == 0) {        // one CTA sees all anchors of its rows: the drain writes d_b itself
                                                  // (TMA store: the row pitch must be a multiple of 16 bytes)
        fused_db = 1;
        args.fused_out = d_b; args.ld_out = (int)dim; args.n_class = n_class; args.ab_sums = st_.absum; args.grad_out = grad_out;
        args.row_meta = bm;
      }
      int st = launch_sweep<kAnaCols>(b_bf16, n_contrast, a_bf16, n_anchor, d, inv_t, args, sw, stream, n_batch);
      if (st != SLCL_OK) return st;
      n_splits_b = sw.splits;
    }
    const int64_t rows = ((d_a || fused_db) ? n_anchor : 0) + ((d_b && !fused_db) ? n_contrast : 0);
    const int lpr = lanes_per_row(d);
    auto fin = [&](auto kernel) {
      launch_pdl(kernel, dim3((unsigned)ceil_div<int64_t>(rows, 8 * (32 / lpr))), dim3(256), 0, stream, na, (int)n_contrast, d,
                 (int)dim, ab, bb, am, bm, a_selfcol, b_selfrow, (const float*)st_.bsum, (const float*)st_.absum, n_class,
                 (int)(n_anchor / n_batch), (int)(n_contrast / n_batch),
                 (const float*)st_.alpha, (const float*)st_.beta, (const float*)st_.colshift, shift, inv_t * kLog2e,
                 (const float*)st_.u, plan_sweep(n_anchor / n_batch, n_contrast / n_batch, n_batch).splits,
                 (const float*)w.grad_partial_b, n_splits_b, fused_db, grad_out, d_a, d_b);
    };
    if (lpr == 8) fin(p2p_finish_bwd_kernel<8>); else if (lpr == 16) fin(p2p_finish_bwd_kernel<16>); else fin(p2p_finish_bwd_kernel<32>);
    return check_launch("slcl_p2p_bwd");
  }
  launch_pdl(p2p_anchor_stat_kernel, dim3(ceil_div(na + BN, 256)), dim3(256), 0, stream, stats, shift, weight, grad_out, na,
             (int)align_up((size_t)na, BN), inv_t, w.anchor_stat);
  const __nv_bfloat16* ab = reinterpret_cast<const __nv_bfloat16*>(a_bf16);
  const __nv_bfloat16* bb = reinterpret_cast<const __nv_bfloat16*>(b_bf16);
  const int by_id = a_selfcol == nullptr;
  const float* gself = nullptr;
  if (!by_id) {          // self maps: the sweeps treat the self pair as an ordinary pair, its entry is taken out afterwards
    launch_pdl(p2p_gself_kernel, dim3(ceil_div(na, 8)), dim3(256), 0, stream, (const float4*)w.anchor_stat, inv_t * kLog2e, ab, bb, d,
               am, bm, a_selfcol, na, w.gself);
    gself = w.gself;
  }
  if (d_a) {
    Sweep sw = plan_sweep(n_anchor / n_batch, n_contrast / n_batch, n_batch, true);
    P2PArgs args{};
    args.row_meta = am; args.col_meta = bm; args.row_stat = w.anchor_stat; args.grad_partial = w.grad_partial_a;
    args.self_by_id = by_id;
    int st = launch_sweep<kGenRows>(a_bf16, n_anchor, b_bf16, n_contrast, d, inv_t, args, sw, stream, n_batch);
    if (st != SLCL_OK) return st;
    const int64_t n = n_anchor * dim;
    launch_pdl(p2p_reduce_grad_kernel, dim3((unsigned)ceil_div<int64_t>(n, 256)), dim3(256), 0, stream, (const float*)w.grad_partial_a,
               sw.splits, n, d, (int)dim, d_a, gself, a_selfcol, bb, 1);
  }
  if (d_b) {
    Sweep sw = plan_sweep(n_contrast / n_batch, n_anchor / n_batch, n_batch);
    P2PArgs args{};
    args.row_meta = bm; args.col_meta = am; args.col_stat = w.anchor_stat; args.grad_partial = w.grad_partial_b;
    args.self_by_id = by_id;
    const bool fused = sw.splits == 1 && dim % 4 == 0;        // one CTA sees all anchors of its rows: the drain writes d_b
    if (fused) { args.fused_out = d_b; args.ld_out = (int)dim; }
    int st = launch_sweep<kGenCols>(b_bf16, n_contrast, a_bf16, n_anchor, d, inv_t, args, sw, stream, n_batch);
    if (st != SLCL_OK) return st;
    if (!fused) {
      const int64_t n = n_contrast * dim;
      launch_pdl(p2p_reduce_grad_kernel, dim3((unsigned)ceil_div<int64_t>(n, 256)), dim3(256), 0, stream,
                 (const float*)w.grad_partial_b, sw.splits, n, d, (int)dim, d_b, gself, b_selfrow, ab, 0);
    } else if (!by_id) {
      launch_pdl(p2p_self_fix_kernel, dim3(ceil_div(na, 8)), dim3(256), 0, stream, gself, a_selfcol, ab, d, (int)dim, na, d_b);
    }
  }
  return check_launch("slcl_p2p_bwd");
}
