"""NVLink peer-memory mailboxes for the small exchanges of the data-parallel path (SURVEY.md 8(e)).

A batch-sharded step needs two kinds of exchange: the pair ``{sum(pixel_sel_loc), sum(sel * row_loss)}`` between the
forward and the backward of the prototype loss (utils/loss.py:558-565 over the global batch), and the per-class sums
``[sets*K, C+1]`` float64 between the class-sum sweep and its finaliser (update_class_center_iter / cal_centroid over the
global batch).  With NCCL each is a collective launch (~20 us of latency plus the Python dispatch) on the critical
path; here they are done INSIDE our own kernels (``slcl_proto_rescale_peer``, the reduce kernel of
``slcl_class_centres_update`` / ``slcl_centroids_fwd``, ``slcl_peer_allreduce_f64``), which store 8-byte
``{epoch | 32-bit payload}`` words straight into every peer's mailbox over NVLink and poll their own.

The mailboxes live in ``torch.distributed._symmetric_memory`` (one process per GPU, one box).  Pass a ``PeerMailbox`` as
the ``group=`` argument of ``mpcl_loss_calc`` / ``mpcl_target_step`` / ``update_class_center_iter`` / ``cal_centroid``.
Rules: every rank makes the same sequence of ``group=mailbox`` calls, all on one CUDA stream per mailbox.  When
symmetric memory cannot be set up, pass ``group=True`` (or a ProcessGroup) and the same calls use NCCL all-reduces.

The pixel <-> pixel losses over the global batch (``SupConLoss`` / ``LocalConLoss`` / ``sampled_supcon_loss`` with
``group=mailbox``) exchange whole row sets (megabytes per rank).  Those go through a second, bulk region per rank
(``rows_bytes`` at construction; ``slcl_peer_allgather``): each rank copies its record into its own send slot and its
peers read it with 16-byte NVLink loads into private tensors, with the mailbox epoch as the flag.
"""
from __future__ import annotations

from typing import List

import torch
import torch.distributed as dist

from . import _lib

DEFAULT_CAPACITY_WORDS = 8192        # 4096 doubles per message: [16, 255+1] class sums
DEFAULT_TIMEOUT_S = 600.0            # a rank that checkpoints / evaluates for minutes must not poison the step


def _slot_bytes(rows_bytes: int) -> int:
    if rows_bytes < 16:
        raise ValueError("rows_bytes must be at least 16")
    return (int(rows_bytes) + 255) // 256 * 256


class PeerMailbox:
    """One mailbox per rank of ``group``.  Construction is a collective call.

    ``capacity_words``: payload words per message (two per float64).  ``timeout_s``: how long a kernel waits for a
    peer before it gives up and returns NaN (0 = for ever, like an NCCL collective); ``timeouts()`` reads the count of
    such events and ``check()`` raises if there were any.  ``rows_bytes``: size of the send slot of the bulk row exchange
    (0 = none; ``slcl.p2p.global_record_bytes`` gives what a pixel <-> pixel loss needs); it must be equal on every rank."""

    def __init__(self, device, group=None, capacity_words: int = DEFAULT_CAPACITY_WORDS, timeout_s: float = DEFAULT_TIMEOUT_S,
                 rows_bytes: int = 0):
        import torch.distributed._symmetric_memory as symm
        if not dist.is_initialized():
            raise RuntimeError("PeerMailbox needs an initialised torch.distributed process group")
        self.lib = _lib.load()
        self.dev = torch.device(device)
        pg = dist.group.WORLD if group is None or group is True else group
        self.group = pg
        self.world = dist.get_world_size(pg)
        self.rank = dist.get_rank(pg)
        self.capacity_words = int(capacity_words)
        self.timeout_s = float(timeout_s)
        n_bytes = self.lib.slcl_peer_mailbox_bytes(self.world, self.capacity_words)
        if n_bytes == 0:
            raise ValueError(f"peer exchange supports 1..16 ranks and capacity >= 2 words, got world={self.world}")
        self.buf = symm.empty(n_bytes // 8, dtype=torch.int64, device=self.dev)
        self.buf.zero_()
        torch.cuda.synchronize(self.dev)
        self.handle = symm.rendezvous(self.buf, pg)
        self.ptrs_dev = int(self.handle.buffer_ptrs_dev)
        self.rows_slot_bytes, self.rows_ptrs_dev, self.rows_buf = 0, 0, None
        if rows_bytes:
            slot = _slot_bytes(rows_bytes)
            agree = torch.tensor([slot, -slot], dtype=torch.int64, device=self.dev)
            dist.all_reduce(agree, op=dist.ReduceOp.MAX, group=pg)
            if int(agree[0]) != -int(agree[1]):
                raise ValueError(f"rows_bytes must be equal on every rank (rank {self.rank}: {rows_bytes})")
            self.rows_buf = symm.empty(self.lib.slcl_peer_rows_region_bytes(slot), dtype=torch.uint8, device=self.dev)
            self.rows_buf.zero_()
            torch.cuda.synchronize(self.dev)
            self.rows_handle = symm.rendezvous(self.rows_buf, pg)
            self.rows_ptrs_dev = int(self.rows_handle.buffer_ptrs_dev)
            self.rows_slot_bytes = slot
        dist.barrier(pg)                      # every mailbox is zeroed and mapped before the first store can arrive
        torch.cuda.synchronize(self.dev)

    def struct(self) -> "_lib.PeerT":
        return _lib.PeerT(self.ptrs_dev, self.rank, self.world, self.capacity_words, self.timeout_s)

    def args(self):
        """(ptrs_dev, rank, world, capacity_words, timeout_s): the flat form the torch custom ops take."""
        return self.ptrs_dev, self.rank, self.world, self.capacity_words, self.timeout_s

    def rows_args(self):
        """(regions_ptr, slot_bytes) of the bulk row exchange (0, 0 without ``rows_bytes``)."""
        return self.rows_ptrs_dev, self.rows_slot_bytes

    def epoch(self) -> int:
        return int(self.buf[0].item())

    def timeouts(self) -> int:
        return int(self.buf[1].item())

    def mismatches(self) -> int:
        """Bulk row exchanges whose records differed in size between ranks (the affected results are NaN)."""
        return int(self.buf[5].item())

    def check(self) -> None:
        """Host-side check (synchronises): raise if any exchange kernel gave up waiting for a peer, or if ranks exchanged
        row sets of different sizes."""
        n = self.timeouts()
        if n:
            raise RuntimeError(f"slcl peer exchange: {n} poll(s) timed out after {self.timeout_s} s on rank {self.rank}; "
                               "the affected results are NaN")
        n = self.mismatches()
        if n:
            raise RuntimeError(f"slcl peer exchange: {n} row exchange(s) on rank {self.rank} got records of another size "
                               "from a peer (ranks with different shapes); the affected results are NaN")


class _LoopbackBox(PeerMailbox):
    def __init__(self, owner, rank):        # noqa: D401 - built by LoopbackMailboxes only
        self._owner = owner                 # keeps the pointer table (and every peer's mailbox) alive
        self.lib = owner.lib
        self.dev = owner.dev
        self.group = None
        self.world = owner.world
        self.rank = rank
        self.capacity_words = owner.capacity_words
        self.timeout_s = owner.timeout_s
        self.buf = owner.bufs[rank]
        self.ptrs_dev = owner.table.data_ptr()
        self.rows_slot_bytes = owner.rows_slot_bytes
        self.rows_ptrs_dev = owner.rows_table.data_ptr() if owner.rows_table is not None else 0


class LoopbackMailboxes:
    """``world`` mailboxes in ordinary memory of ONE device (no process group): ``boxes[r]`` is what rank r would hold.
    Several "ranks" can then run on different CUDA streams of one GPU and really exchange through the protocol --
    how the single-GPU test box exercises the multi-rank kernels."""

    def __init__(self, world: int, device, capacity_words: int = DEFAULT_CAPACITY_WORDS, timeout_s: float = 20.0,
                 rows_bytes: int = 0):
        self.lib = _lib.load()
        self.dev = torch.device(device)
        self.world = int(world)
        self.capacity_words = int(capacity_words)
        self.timeout_s = float(timeout_s)
        n_bytes = self.lib.slcl_peer_mailbox_bytes(self.world, self.capacity_words)
        if n_bytes == 0:
            raise ValueError("peer exchange supports 1..16 ranks and capacity >= 2 words")
        self.bufs: List[torch.Tensor] = [torch.zeros(n_bytes // 8, dtype=torch.int64, device=self.dev) for _ in range(world)]
        self.table = torch.tensor([b.data_ptr() for b in self.bufs], dtype=torch.int64, device=self.dev)
        self.rows_slot_bytes, self.rows_table = 0, None
        if rows_bytes:                        # the bulk row regions, in plain device memory
            self.rows_slot_bytes = _slot_bytes(rows_bytes)
            n = self.lib.slcl_peer_rows_region_bytes(self.rows_slot_bytes)
            self.rows_bufs = [torch.zeros(n, dtype=torch.uint8, device=self.dev) for _ in range(world)]
            self.rows_table = torch.tensor([b.data_ptr() for b in self.rows_bufs], dtype=torch.int64, device=self.dev)
        torch.cuda.synchronize(self.dev)
        self.boxes = [_LoopbackBox(self, r) for r in range(world)]
