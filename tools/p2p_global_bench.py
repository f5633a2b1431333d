"""Pixel <-> pixel loss over the global batch of N GPUs (``sampled_supcon_loss(group=)``, ``BlockConLoss(group=)``):
check, then time.

    torchrun --nproc_per_node N tools/p2p_global_bench.py [--loss sampled|blockcon] [--out FILE]

Check first, on both routes (NVLink peer memory: ``PeerMailbox(rows_bytes=...)``; NCCL: ``group=True``): every rank's
sharded loss and gradient equal the global problem evaluated on that rank's own GPU (loss rtol 1e-5, gradient rtol 1e-4
with an absolute floor of 1e-4 max|grad|: the bf16 rounding of the G tiles next to a column shift summed in another
fp32 order, see tests/test_p2p_global.py:grad_close), the loss has identical bits on every rank, and no exchange timed out.  The
script exits non-zero otherwise.

Then times fwd+bwd as ONE CUDA graph per step on the peer route at the per-rank shape of cfg3 (a [16, 256, 64, 64] map,
4096 anchors and 16384 contrast rows drawn per rank, K = 5, T = 0.7; the draw itself is outside the timed graph), the row
exchange on its own, and the replicas-only loss (each rank alone, no group) at the same per-rank shape.  Rank 0 prints one
JSON line (and appends it to --out) with the card name and power limit read in the same run.

``--loss blockcon``: the same check and timings for ``BlockConLoss(group=)`` at the reference's per-rank shape
(1, 2, 32, 224, 224) with block_size 32 (49 tiles of 2048 rows) and labels in [0, 4); the global problem evaluated on each
rank's GPU is ``BlockConLoss`` of the ranks' batches concatenated.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "soft-labeled-contrastive-learning_b200")]

from slcl import ops  # noqa: E402
from slcl.p2p import BlockConLoss, _Exchange, _pack, global_record_bytes, sample_class_balanced, sampled_supcon_loss  # noqa: E402
from slcl.peer import PeerMailbox  # noqa: E402

B, C, H, W, K, TEMP = 16, 256, 64, 64, 5, 0.7
N_ANCHOR, N_CONTRAST = 4096, 16384
BF16_PEAK_TFLOPS = 1643.3          # the measured bf16 peak DESIGN.md quotes fractions against
BC_SHAPE, BC_BLOCK, BC_K = (1, 2, 32, 224, 224), 32, 4          # --loss blockcon, per rank


def shard_inputs(q, dev):
    g = torch.Generator().manual_seed(7000 + q)
    feat = torch.randn(B, C, H, W, generator=g).to(dev)
    lab = torch.randint(0, K, (B, H, W), generator=g).to(dev)
    a, c = sample_class_balanced(lab, N_ANCHOR, N_CONTRAST, K, torch.Generator(dev).manual_seed(8000 + q))
    return feat, lab, a, c


def grad_ok(a, b, rtol=1e-4, floor=1.0):
    b = b.double()
    atol = rtol * floor * float(b.abs().max())
    return bool(((a.double() - b).abs() <= atol + rtol * b.abs()).all())


def fwd_bwd(feat, lab, a, c, group):
    f = feat.clone().requires_grad_(True)
    loss = sampled_supcon_loss(f, lab, N_ANCHOR, N_CONTRAST, K, TEMP, anchor_idx=a, contrast_idx=c, group=group)
    loss.backward()
    return loss.detach(), f.grad


class Sampled:
    """cfg3: 4096 anchors x 16384 contrast rows drawn per rank from a [16, 256, 64, 64] map."""
    what = "sampled_supcon_loss(group=PeerMailbox) fwd+bwd, one CUDA graph per step"
    shape = {"map": [B, C, H, W], "n_anchor": N_ANCHOR, "n_contrast": N_CONTRAST, "K": K, "T": TEMP}
    channels = C
    rows_bytes = global_record_bytes(N_ANCHOR, N_CONTRAST, C)

    def __init__(self, rank, world, dev):
        shards = [shard_inputs(q, dev) for q in range(world)]
        n_pix = B * H * W
        self.feat_g = torch.cat([s[0] for s in shards])
        self.lab_g = torch.cat([s[1] for s in shards])
        self.a_g = torch.cat([s[2] + q * n_pix for q, s in enumerate(shards)])
        self.c_g = torch.cat([s[3] + q * n_pix for q, s in enumerate(shards)])
        self.feat, self.lab, self.a, self.c = shards[rank]
        self.batch = B
        self.flop = 8.0 * N_ANCHOR * (N_CONTRAST * world) * C

    def global_here(self):
        return fwd_bwd(self.feat_g, self.lab_g, self.a_g, self.c_g, None)

    def run(self, f, group):
        return sampled_supcon_loss(f, self.lab, N_ANCHOR, N_CONTRAST, K, TEMP, anchor_idx=self.a, contrast_idx=self.c,
                                   group=group)

    def rows_record_parts(self, dp, dev):
        parts = []
        for n in (N_CONTRAST, N_ANCHOR):
            parts += [torch.zeros(n, dp, dtype=torch.bfloat16, device=dev), torch.zeros(n, 2, dtype=torch.int32, device=dev),
                      torch.zeros(n, dtype=torch.float32, device=dev)]
        return parts


class BlockCon:
    """BlockConLoss at the reference's per-rank shape: every tile's problem holds that tile's rows of all ranks."""
    what = "BlockConLoss(group=PeerMailbox) fwd+bwd, one CUDA graph per step"
    b, v, c, h, w = BC_SHAPE
    tiles = (w // BC_BLOCK) ** 2
    rows = b * v * tiles * BC_BLOCK * BC_BLOCK          # per rank: anchors = contrast rows
    shape = {"features": list(BC_SHAPE), "block_size": BC_BLOCK, "tiles": tiles, "rows_per_rank": rows, "K": BC_K, "T": TEMP}
    channels = c
    rows_bytes = global_record_bytes(rows, rows, c, same_rows=True, n_batch=tiles)

    def __init__(self, rank, world, dev):
        ins = []
        for q in range(world):
            g = torch.Generator().manual_seed(9000 + q)
            f = torch.nn.functional.normalize(torch.randn(*BC_SHAPE, generator=g), dim=2)
            ins.append((f.to(dev), torch.randint(0, BC_K, (self.b, self.v, self.h, self.w), generator=g).to(dev)))
        self.feat_g = torch.cat([x[0] for x in ins])
        self.lab_g = torch.cat([x[1] for x in ins])
        self.feat, self.lab = ins[rank]
        self.batch = self.b
        self.mod = {}
        # 8 A_l M_g d per tile problem: this rank's rows of the tile against every rank's rows of it
        r_tile = self.rows // self.tiles
        self.flop = 8.0 * self.tiles * r_tile * (r_tile * world) * self.c

    def global_here(self):
        f = self.feat_g.clone().requires_grad_(True)
        loss = BlockConLoss(TEMP, BC_BLOCK)(f, self.lab_g)
        loss.backward()
        return loss.detach(), f.grad

    def run(self, f, group):
        key = id(group)
        if key not in self.mod:          # one module per route, as a trainer would hold it
            self.mod[key] = BlockConLoss(TEMP, BC_BLOCK, group=group)
        return self.mod[key](f, self.lab)

    def rows_record_parts(self, dp, dev):
        return [torch.zeros(self.rows, dp, dtype=torch.bfloat16, device=dev),
                torch.zeros(self.rows, 2, dtype=torch.int32, device=dev), torch.zeros(self.rows, dtype=torch.float32, device=dev)]


def graph_time(step, n_iter=50):
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(3):
            step()
    torch.cuda.current_stream().wait_stream(side)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        step()
    for _ in range(5):
        g.replay()
    torch.cuda.synchronize()
    dist.barrier()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(n_iter):
        g.replay()
    t1.record()
    torch.cuda.synchronize()
    return t0.elapsed_time(t1) / n_iter


def max_over_ranks(x, dev):
    t = torch.tensor([x], dtype=torch.float64, device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--loss", choices=("sampled", "blockcon"), default="sampled")
    args = ap.parse_args()
    dist.init_process_group("nccl")
    rank, world = dist.get_rank(), dist.get_world_size()
    local = int(os.environ.get("LOCAL_RANK", rank))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    work = (BlockCon if args.loss == "blockcon" else Sampled)(rank, world, dev)
    box = PeerMailbox(dev, rows_bytes=work.rows_bytes)

    # -- check: sharded == the global problem on this GPU, both routes ---------------------------------------------------
    ref_loss, ref_grad = work.global_here()
    ref_grad = ref_grad[rank * work.batch:(rank + 1) * work.batch]
    feat = work.feat
    checks = {}
    for route, group in (("peer", box), ("nccl", True)):
        fr = feat.clone().requires_grad_(True)
        loss = work.run(fr, group)
        loss.backward()
        loss, grad = loss.detach(), fr.grad
        torch.cuda.synchronize()
        every = [torch.zeros_like(loss) for _ in range(world)]
        dist.all_gather(every, loss)
        same_bits = all(torch.equal(e, every[0]) for e in every)
        ok = (same_bits and bool(torch.isfinite(loss)) and abs(float(loss) - float(ref_loss)) <= 1e-5 * abs(float(ref_loss))
              and grad_ok(grad, ref_grad))
        checks[route] = {"ok": ok, "loss": float(loss), "global_loss_here": float(ref_loss), "same_bits": same_bits}
    checks["timeouts"] = box.timeouts()
    checks["mismatches"] = box.mismatches()
    flags = torch.tensor([int(checks["peer"]["ok"] and checks["nccl"]["ok"] and checks["timeouts"] == 0
                              and checks["mismatches"] == 0)], device=dev)
    dist.all_reduce(flags, op=dist.ReduceOp.MIN)
    if not int(flags):
        print(json.dumps({"rank": rank, "check": checks}), flush=True)
        dist.destroy_process_group()
        sys.exit(1)
    del ref_grad
    work.feat_g = work.lab_g = None
    torch.cuda.reset_peak_memory_stats(dev)          # the peak below is the timed steps', not the global check's

    # -- timing ---------------------------------------------------------------------------------------------------------
    f = feat.clone().requires_grad_(True)

    def step_group():
        f.grad = None
        work.run(f, box).backward()

    def step_alone():
        f.grad = None
        work.run(f, None).backward()

    ms_group = max_over_ranks(graph_time(step_group, args.iters), dev)
    ms_alone = max_over_ranks(graph_time(step_alone, args.iters), dev)
    # the row exchange alone: the forward's first all-gather, at its real record size
    x = _Exchange(box)
    dp = (work.channels + 63) // 64 * 64
    rec, _ = _pack([torch.zeros(4, dtype=torch.int32, device=dev), torch.zeros(1, dtype=torch.int32, device=dev)]
                   + work.rows_record_parts(dp, dev))
    status = torch.zeros(1, dtype=torch.int32, device=dev)
    ms_xchg = max_over_ranks(graph_time(lambda: x.allgather(rec, status), args.iters), dev)
    box.check()

    flop = work.flop
    peak_mib = torch.cuda.max_memory_allocated(dev) / 2 ** 20
    if rank == 0:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", str(local)],
                           capture_output=True, text=True).stdout.strip()
        line = {
            "what": work.what, "world": world,
            "per_rank_shape": work.shape,
            "check": {"peer": checks["peer"]["ok"], "nccl": checks["nccl"]["ok"], "timeouts": 0},
            "ms_per_step_max_over_ranks": round(ms_group, 4),
            "exchange_ms_rows_record": round(ms_xchg, 4), "rows_record_bytes": rec.numel(),
            "per_rank_tflop": round(flop / 1e12, 4),
            "tflops_per_rank": round(flop / (ms_group * 1e-3) / 1e12, 1),
            "frac_of_measured_bf16_peak": round(flop / (ms_group * 1e-3) / 1e12 / BF16_PEAK_TFLOPS, 3),
            "replicas_only_ms_same_shape": round(ms_alone, 4),
            "peak_allocated_mib_rank0": round(peak_mib, 1),
            "gpu": q or torch.cuda.get_device_name(dev),
        }
        print(json.dumps(line), flush=True)
        if args.out:
            with open(args.out, "a") as fh:
                fh.write(json.dumps(line) + "\n")
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
