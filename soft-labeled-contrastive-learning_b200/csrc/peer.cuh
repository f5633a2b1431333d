// peer.cuh -- NVLink peer-memory mailboxes: the scalar / small-vector exchanges of the data-parallel path
// (SURVEY.md 8(e)) done INSIDE our own kernels instead of as NCCL collectives.
//
// Every rank owns one mailbox in memory that all ranks of the box have mapped (torch symmetric memory, or plain
// device memory when several "ranks" share one GPU in the tests); `boxes[r]` is rank r's mailbox in THIS process'
// address space.  Layout in 8-byte words:
//   word 0  epoch    : number of exchange calls this rank has completed (only its own kernels write it)
//   word 1  timeouts : number of polls that gave up (diagnostic; a timed-out value is NaN)
//   word 2  ticket   : block counter of a multi-block exchange kernel (self-resetting)
//   word 3  ready    : split-phase exchanges: the epoch whose result this rank has published to its own blocks
//   word 4  pending  : split-phase exchanges: the epoch a sender kernel has put on the wire and a later kernel completes
//   word 5   mismatch: number of bulk all-gathers (peer_rows.cu) whose records disagreed in size between ranks
//   word 6..7        : reserved
//   word 8 + (q * world + r) * capacity + s : payload word s of sender r for epoch parity q
// A payload word is {epoch : 32 | data : 32}: an aligned 8-byte store is single-copy atomic, so flag and data arrive
// together and no fence is needed (the protocol NCCL calls LL).  A call with epoch e writes its words into every
// peer's mailbox (P2P stores over NVLink), then polls its OWN mailbox until all `world` senders show e.  Two
// parities suffice: a sender can reach epoch e+2 only after this rank has SENT its epoch e+1 words, which its
// stream orders after everything it read at epoch e.  All ranks must make the same sequence of exchange calls on
// one stream per mailbox.
#pragma once

#include "common.cuh"

namespace slcl {

constexpr int kMaxPeers = 16;
constexpr int kPeerHeaderWords = 8;
constexpr long long kPeerMinCapacity = 2;

struct PeerCtx {
  unsigned long long* const* boxes;   // device array [world]; null = no exchange
  int rank, world;
  long long capacity;                 // payload words per sender per parity
  unsigned long long timeout_ns;      // 0 = wait for ever
};

inline bool peer_valid(const slcl_peer_t* p) {
  return p && p->mailboxes_dev && p->world >= 1 && p->world <= kMaxPeers && p->rank >= 0 && p->rank < p->world &&
         p->capacity_words >= kPeerMinCapacity && p->timeout_s >= 0.0;
}
inline PeerCtx peer_ctx(const slcl_peer_t* p) {
  PeerCtx c{};
  if (!p) return c;
  c.boxes = reinterpret_cast<unsigned long long* const*>(p->mailboxes_dev);
  c.rank = p->rank; c.world = p->world; c.capacity = p->capacity_words;
  c.timeout_ns = (unsigned long long)(p->timeout_s * 1e9);
  return c;
}

__device__ __forceinline__ unsigned long long* peer_slot(unsigned long long* box, const PeerCtx& c, unsigned q, int sender,
                                                         long long s) {
  return box + kPeerHeaderWords + ((long long)(q * (unsigned)c.world + (unsigned)sender) * c.capacity + s);
}

// Epoch of the call in flight.  Every thread of every block may call it; the counter moves only in peer_epoch_end().
__device__ __forceinline__ unsigned int peer_epoch_begin(const PeerCtx& c) {
  return (unsigned int)(*reinterpret_cast<volatile unsigned long long*>(c.boxes[c.rank])) + 1u;
}

// ONE thread per block, after the block's last poll (and a __syncthreads): the block that arrives last publishes the
// new epoch and resets the ticket.  Returns true for that last block (it may run a grid-wide epilogue).
__device__ __forceinline__ bool peer_epoch_end(const PeerCtx& c, unsigned int e, unsigned int n_blocks) {
  unsigned long long* mine = c.boxes[c.rank];
  __threadfence();
  const unsigned long long t = atomicAdd(mine + 2, 1ull);
  if (t != (unsigned long long)n_blocks - 1ull) return false;
  mine[2] = 0ull;
  __threadfence();
  *reinterpret_cast<volatile unsigned long long*>(mine) = (unsigned long long)e;
  return true;
}

// Split-phase halves of peer_send_recv: a producer kernel only SENDS (and records the epoch in word 4), a later kernel
// on the same stream RECEIVES -- the wire latency then hides behind whatever runs in between (launch, prologue, loads).
__device__ __forceinline__ void peer_send(const PeerCtx& c, unsigned int e, int peer, long long s, unsigned int data) {
  volatile unsigned long long* dst = peer_slot(c.boxes[peer], c, e & 1u, c.rank, s);
  *dst = ((unsigned long long)e << 32) | (unsigned long long)data;
}
__device__ __forceinline__ unsigned int peer_recv(const PeerCtx& c, unsigned int e, int peer, long long s, bool& ok) {
  volatile unsigned long long* src = peer_slot(c.boxes[c.rank], c, e & 1u, peer, s);
  unsigned long long t0 = 0ull, now, got;
  ok = true;
  for (unsigned int spin = 0;; ++spin) {
    got = *src;
    if ((unsigned int)(got >> 32) == e) break;
    if (c.timeout_ns != 0ull && (spin & 63u) == 63u) {
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
      if (t0 == 0ull) t0 = now;
      else if (now - t0 > c.timeout_ns) { atomicAdd(c.boxes[c.rank] + 1, 1ull); ok = false; break; }
    }
  }
  return (unsigned int)got;
}

// Send one 32-bit word to `dst_rank` (payload slot s) and return the word `src_rank` sent to us in slot s.
// ok = false after a time-out (the return value is then undefined).
__device__ __forceinline__ unsigned int peer_send_recv(const PeerCtx& c, unsigned int e, int peer, long long s,
                                                       unsigned int data, bool& ok) {
  const unsigned int q = e & 1u;
  volatile unsigned long long* dst = peer_slot(c.boxes[peer], c, q, c.rank, s);
  *dst = ((unsigned long long)e << 32) | (unsigned long long)data;
  volatile unsigned long long* src = peer_slot(c.boxes[c.rank], c, q, peer, s);
  unsigned long long t0 = 0ull, now, got;
  ok = true;
  for (unsigned int spin = 0;; ++spin) {
    got = *src;
    if ((unsigned int)(got >> 32) == e) break;
    if (c.timeout_ns != 0ull && (spin & 63u) == 63u) {
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
      if (t0 == 0ull) t0 = now;
      else if (now - t0 > c.timeout_ns) {
        atomicAdd(c.boxes[c.rank] + 1, 1ull);
        ok = false;
        break;
      }
    }
  }
  return (unsigned int)got;
}

// Warp-collective all-reduce (sum, in rank order: identical bits on every rank) of one double per warp; payload
// slots 2*idx and 2*idx+1 carry its two 32-bit halves.  Lane 2p+v talks to rank p about half v (world <= 16).
// Returns NaN when any peer timed out.
__device__ __forceinline__ double peer_warp_allreduce(const PeerCtx& c, unsigned int e, long long idx, double t) {
  const int lane = threadIdx.x & 31;
  unsigned int got = 0u;
  bool ok = true;
  if (lane < 2 * c.world) {
    const int p = lane >> 1, v = lane & 1;
    const unsigned long long bits = (unsigned long long)__double_as_longlong(t);
    got = peer_send_recv(c, e, p, 2 * idx + v, v ? (unsigned int)(bits >> 32) : (unsigned int)bits, ok);
  }
  const bool bad = __any_sync(0xffffffffu, !ok);
  double acc = 0.0;
  for (int r = 0; r < c.world; ++r) {
    const unsigned int lo = __shfl_sync(0xffffffffu, got, 2 * r), hi = __shfl_sync(0xffffffffu, got, 2 * r + 1);
    acc += __longlong_as_double((long long)(((unsigned long long)hi << 32) | (unsigned long long)lo));
  }
  return bad ? __longlong_as_double(0x7FF8000000000000ll) : acc;
}

}  // namespace slcl
