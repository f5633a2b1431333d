// peer_rows.cu -- bulk all-gather of byte records over NVLink peer memory (the pixel<->pixel losses over the global batch,
// SURVEY.md 8(e)): every rank contributes one record of n bytes (gathered bf16 rows, their {label, id} rows, norms, ...),
// every rank receives all `world` records in rank order, in a private buffer of its own.
//
// Shape: PULL.  Each rank owns a region in memory that all ranks have mapped (torch symmetric memory, or plain device
// memory when ranks are streams of one GPU).  It copies its record into its own send slot, publishes the slot's flag, and
// every peer reads the slot with 16-byte loads straight into the private output.  Pull rather than push: the payload
// crosses NVLink exactly once either way, but with pull a rank writes only its own slot (one local copy at HBM rate), the
// remote traffic is loads issued by the rank that needs the data, and the result lands in a caller-owned tensor that no
// later call can overwrite -- push would need a receive slot per sender plus the same private copy.
//
// Region layout (slcl_peer_rows_region_bytes):
//   word 0, 1   ready[q]  : epoch whose record slot q holds (written by the owner, read by peers)
//   word 2      ticket of the publish kernel, word 3 ticket of the pull kernel (self-resetting)
//   word 8 + p  ack[p]    : last epoch at which rank p finished reading this rank's slots (written remotely by p)
//   byte kHeader + q * slot_bytes : send slot of epoch parity q
// The epoch is the mailbox's (peer.cuh): the call counts as one exchange of the mailbox sequence, so it interleaves with the
// scalar exchanges of the other losses.  A slot of parity q is rewritten only after every peer has acked the epoch it last
// published there (ready[q]).  A call whose status is bad -- a time-out or a size mismatch, here or in an earlier exchange
// of the same loss -- publishes nothing and waits for nobody.  Four launches per call, none of which polls with more than
// one block:
//   wait_free (1 block) -> publish (copy + last-block ticket + system-scope release of the flag)
//   -> wait_ready (1 block) -> pull (copy + key check + last-block acks and epoch).
#include "common.cuh"
#include "peer.cuh"

namespace slcl {
namespace {

constexpr int kRowsHeaderBytes = 512;
constexpr int kRowsAckWord = 8;
constexpr int kKeyBytes = 16;            // leading bytes of a record that must be equal on every rank (sizes, shapes)
constexpr int kCopyThreads = 256;

struct RowsCtx {
  unsigned long long* const* regions;    // device array [world]
  long long slot_bytes;
};

__device__ __forceinline__ unsigned long long* rows_hdr(const RowsCtx& x, int r) { return x.regions[r]; }
__device__ __forceinline__ char* rows_slot(const RowsCtx& x, int r, unsigned q) {
  return reinterpret_cast<char*>(x.regions[r]) + kRowsHeaderBytes + (long long)q * x.slot_bytes;
}

__device__ __forceinline__ bool poll_until(volatile unsigned long long* p, long long want, bool at_least, const PeerCtx& c) {
  unsigned long long t0 = 0ull, now;
  for (unsigned int spin = 0;; ++spin) {
    const long long v = (long long)*p;
    if (at_least ? v >= want : v == want) return true;
    if (c.timeout_ns != 0ull && (spin & 63u) == 63u) {
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
      if (t0 == 0ull) t0 = now;
      else if (now - t0 > c.timeout_ns) { atomicAdd(c.boxes[c.rank] + 1, 1ull); return false; }
    }
  }
}

// Lane p waits until peer p has read what this rank last published in the slot of this parity: the epoch in the own
// header's ready[q] (0 = never published).  Not that of epoch e - 2: the epoch counter is shared with the scalar exchanges
// of the mailbox, so the last row exchange on this parity may lie any number of epochs back.  Skipped when the status is
// already bad: the publish behind this kernel is then skipped too.
__global__ void __launch_bounds__(32) rows_wait_free_kernel(PeerCtx c, RowsCtx x, int* status) {
  const unsigned int e = peer_epoch_begin(c);
  const int p = threadIdx.x;
  unsigned long long* mine = rows_hdr(x, c.rank);
  const long long last = (long long)*reinterpret_cast<volatile unsigned long long*>(mine + (e & 1u));
  const bool skip = *reinterpret_cast<volatile int*>(status) != 0;
  bool ok = true;
  if (!skip && p < c.world && p != c.rank && last > 0)
    ok = poll_until(reinterpret_cast<volatile unsigned long long*>(mine + kRowsAckWord + p), last, true, c);
  if (__any_sync(0xffffffffu, !ok) && p == 0) atomicOr(status, 1);
  __threadfence_system();
}

// Copy the record into this rank's send slot; the last block releases the flag at system scope.  Nothing is written when
// the status is bad (a time-out, here or in an earlier exchange of the same call): a peer still reading the slot's previous
// record can never see it torn, and the peers waiting for this flag time out and return NaN as well -- fail-closed on every
// rank.
__global__ void __launch_bounds__(kCopyThreads) rows_publish_kernel(PeerCtx c, RowsCtx x, const uint4* record, long long n16,
                                                                    const int* status) {
  if (*reinterpret_cast<const volatile int*>(status) != 0) return;          // same value in every block
  const unsigned int e = peer_epoch_begin(c);
  uint4* dst = reinterpret_cast<uint4*>(rows_slot(x, c.rank, e & 1u));
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n16; i += (long long)gridDim.x * blockDim.x)
    dst[i] = __ldg(record + i);
  __syncthreads();
  if (threadIdx.x == 0) {
    unsigned long long* hdr = rows_hdr(x, c.rank);
    __threadfence_system();
    if (atomicAdd(hdr + 2, 1ull) == (unsigned long long)gridDim.x - 1ull) {
      hdr[2] = 0ull;
      __threadfence_system();
      asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(hdr + (e & 1u)), "l"((unsigned long long)e) : "memory");
    }
  }
}

// Lane p waits for peer p's flag of this epoch (skipped when the caller's status is already bad: the result is NaN anyway).
__global__ void __launch_bounds__(32) rows_wait_ready_kernel(PeerCtx c, RowsCtx x, int* status) {
  const unsigned int e = peer_epoch_begin(c);
  const int p = threadIdx.x;
  const bool skip = *reinterpret_cast<volatile int*>(status) != 0;
  bool ok = true;
  if (!skip && p < c.world && p != c.rank)
    ok = poll_until(reinterpret_cast<volatile unsigned long long*>(rows_hdr(x, p) + (e & 1u)), (long long)e, false, c);
  if (__any_sync(0xffffffffu, !ok) && p == 0) atomicOr(status, 1);
  __threadfence_system();          // acquire: the pull kernel behind this one reads what the flags released
}

// out[p] = record of rank p.  Block 0 compares every record's key with this rank's own (status bit 2 and mailbox word 5
// count a mismatch); the last block acks every peer and ends the epoch.
__global__ void __launch_bounds__(kCopyThreads) rows_pull_kernel(PeerCtx c, RowsCtx x, const uint4* record, long long n16,
                                                                 uint4* out, int* status) {
  const unsigned int e = peer_epoch_begin(c);
  const unsigned q = e & 1u;
  const long long total = n16 * c.world;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int p = (int)(i / n16);
    const long long k = i - (long long)p * n16;
    out[i] = p == c.rank ? __ldg(record + k) : __ldcv(reinterpret_cast<const uint4*>(rows_slot(x, p, q)) + k);
  }
  if (blockIdx.x == 0 && threadIdx.x < c.world && threadIdx.x != c.rank) {
    const int p = threadIdx.x;
    const uint4 mine = __ldg(record);
    const uint4 theirs = __ldcv(reinterpret_cast<const uint4*>(rows_slot(x, p, q)));
    static_assert(kKeyBytes == sizeof(uint4), "key = the first 16-byte word");
    if (mine.x != theirs.x || mine.y != theirs.y || mine.z != theirs.z || mine.w != theirs.w) {
      atomicOr(status, 2);
      atomicAdd(c.boxes[c.rank] + 5, 1ull);
    }
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    unsigned long long* hdr = rows_hdr(x, c.rank);
    __threadfence_system();
    if (atomicAdd(hdr + 3, 1ull) == (unsigned long long)gridDim.x - 1ull) {
      hdr[3] = 0ull;
      __threadfence_system();
      for (int p = 0; p < c.world; ++p)
        if (p != c.rank) *reinterpret_cast<volatile unsigned long long*>(rows_hdr(x, p) + kRowsAckWord + c.rank) = e;
      __threadfence_system();
      *reinterpret_cast<volatile unsigned long long*>(c.boxes[c.rank]) = (unsigned long long)e;
    }
  }
}

int copy_blocks(long long n16) {
  const long long want = ceil_div<long long>(n16, kCopyThreads * 4);
  const long long cap = 4ll * sm_count();
  return (int)(want < 1 ? 1 : (want > cap ? cap : want));
}

}  // namespace
}  // namespace slcl

using namespace slcl;

extern "C" size_t slcl_peer_rows_region_bytes(int64_t slot_bytes) {
  if (slot_bytes < kKeyBytes || slot_bytes % 16) return 0;
  return (size_t)kRowsHeaderBytes + 2 * (size_t)slot_bytes;
}

extern "C" int slcl_peer_allgather(const void* record, int64_t n_bytes, void* out, int32_t* status, const slcl_peer_t* peer,
                                   const void* regions_dev, int64_t slot_bytes, slcl_stream_t stream_) {
  if (!record || !out || !status || !regions_dev || !peer_valid(peer) || n_bytes < kKeyBytes || n_bytes % 16 ||
      slot_bytes % 16 || !aligned16(record) || !aligned16(out))
    return SLCL_ERR_INVALID_ARGUMENT;
  if (n_bytes > slot_bytes) return SLCL_ERR_WORKSPACE;
  cudaStream_t stream = (cudaStream_t)stream_;
  const PeerCtx c = peer_ctx(peer);
  const RowsCtx x{reinterpret_cast<unsigned long long* const*>(regions_dev), (long long)slot_bytes};
  const long long n16 = n_bytes / 16;
  const uint4* rec = reinterpret_cast<const uint4*>(record);
  rows_wait_free_kernel<<<1, 32, 0, stream>>>(c, x, status);
  rows_publish_kernel<<<copy_blocks(n16), kCopyThreads, 0, stream>>>(c, x, rec, n16, status);
  rows_wait_ready_kernel<<<1, 32, 0, stream>>>(c, x, status);
  rows_pull_kernel<<<copy_blocks(n16 * c.world), kCopyThreads, 0, stream>>>(c, x, rec, n16, reinterpret_cast<uint4*>(out), status);
  return check_launch("slcl_peer_allgather");
}
