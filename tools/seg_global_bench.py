"""Segmentation losses over the global batch of N GPUs (``seg_losses(group=)``): check, then time.

    torchrun --nproc_per_node N tools/seg_global_bench.py [--iters 50] [--out FILE]

Check first, on both routes (NVLink peer memory: ``PeerMailbox``; NCCL: ``group=True``): every rank's losses
{cross entropy, dice, jaccard} and its shard of dlogits equal the global batch evaluated on that rank's own GPU (losses
rtol 1e-5, gradients rtol 1e-5 with an absolute floor of 1e-5 max|grad|), the losses have identical bits on every rank,
and no exchange timed out.  The ranks hold different batch sizes (``shard_range`` of 64 N - 1 images when N > 1), as a
data loader's last batch would.  The script exits non-zero otherwise.

Then times fwd+bwd (upstream weights 1 / 0.5 / 2 on the three losses) as ONE CUDA graph per step at the logits size of
cfg5 per rank ([64, 4, 224, 224] fp32, labels in [0, 4)): the peer route, the NCCL route, and the local call (each rank
alone, no group).  Each time is the max over ranks.  Rank 0 prints one JSON line (and appends it to --out) with the card
name and power limit read in the same run.  With one process the group= calls are the single-rank call and only the
local timing means anything.
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

from slcl.distributed import shard_range  # noqa: E402
from slcl.peer import PeerMailbox  # noqa: E402
from slcl.seg import seg_losses  # noqa: E402

B, K, H, W = 64, 4, 224, 224          # cfg5 logits per rank
WEIGHTS = (1.0, 0.5, 2.0)


def make_inputs(n_images, dev):
    g = torch.Generator().manual_seed(5150)
    z = 1.5 * torch.randn(n_images, K, H, W, generator=g)
    lab = torch.randint(0, K, (n_images, H, W), generator=g)
    lab[:, :8] = -100                                  # a band of ignored pixels, as padded crops carry
    return z.to(dev), lab.to(dev)


def fwd_bwd(z, lab, group, w):
    zz = z.clone().requires_grad_(True)
    out = seg_losses(zz, lab, group=group)
    (out * w).sum().backward()
    return out.detach(), zz.grad


def grad_ok(a, b, rtol=1e-5, floor=1.0):
    b = b.double()
    atol = rtol * floor * float(b.abs().max())
    return bool(((a.double() - b).abs() <= atol + rtol * b.abs()).all())


def graph_time(step, n_iter):
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
    args = ap.parse_args()
    dist.init_process_group("nccl")
    rank, world = dist.get_rank(), dist.get_world_size()
    local = int(os.environ.get("LOCAL_RANK", rank))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    box = PeerMailbox(dev)
    w = torch.tensor(WEIGHTS, device=dev)

    # -- check: sharded == the global batch on this GPU, both routes (unequal shards) ------------------------------------
    n_global = B * world - (1 if world > 1 else 0)
    lo, hi = shard_range(n_global, rank, world)
    z_g, lab_g = make_inputs(n_global, dev)
    ref_l, ref_dz = fwd_bwd(z_g, lab_g, None, w)
    ref_dz = ref_dz[lo:hi]
    z_r, lab_r = z_g[lo:hi].contiguous(), lab_g[lo:hi].contiguous()
    checks = {}
    for route, group in (("peer", box), ("nccl", True)):
        out, dz = fwd_bwd(z_r, lab_r, group, w)
        torch.cuda.synchronize()
        every = [torch.zeros_like(out) for _ in range(world)]
        dist.all_gather(every, out)
        same_bits = all(torch.equal(e, every[0]) for e in every)
        loss_ok = bool(((out.double() - ref_l.double()).abs() <= 1e-5 * ref_l.double().abs()).all())
        ok = same_bits and bool(torch.isfinite(out).all()) and loss_ok and grad_ok(dz, ref_dz)
        checks[route] = {"ok": ok, "losses": out.tolist(), "global_losses_here": ref_l.tolist(), "same_bits": same_bits}
    checks["timeouts"] = box.timeouts()
    flags = torch.tensor([int(checks["peer"]["ok"] and checks["nccl"]["ok"] and checks["timeouts"] == 0)], device=dev)
    dist.all_reduce(flags, op=dist.ReduceOp.MIN)
    if not int(flags):
        print(json.dumps({"rank": rank, "check": checks}), flush=True)
        dist.destroy_process_group()
        sys.exit(1)
    del z_g, lab_g, ref_dz, z_r, lab_r

    # -- timing at the cfg5 logits size per rank -------------------------------------------------------------------------
    z, lab = make_inputs(B, dev)
    f = z.clone().requires_grad_(True)

    def step(group):
        def run():
            f.grad = None
            (seg_losses(f, lab, group=group) * w).sum().backward()
        return run

    ms = {name: max_over_ranks(graph_time(step(group), args.iters), dev)
          for name, group in (("peer", box), ("nccl", True), ("local", None))}
    box.check()
    if rank == 0:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", str(local)],
                           capture_output=True, text=True).stdout.strip()
        line = {
            "what": "seg_losses(group=) fwd+bwd, one CUDA graph per step, max over ranks",
            "world": world,
            "per_rank_logits": [B, K, H, W],
            "check_global_images": n_global,
            "check": {"peer": checks["peer"]["ok"], "nccl": checks["nccl"]["ok"], "timeouts": 0},
            "ms_peer": round(ms["peer"], 4), "ms_nccl": round(ms["nccl"], 4), "ms_local": round(ms["local"], 4),
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
