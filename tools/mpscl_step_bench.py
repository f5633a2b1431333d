"""mpscl_step against the composition it replaces (mpcl_source_step + mpcl_target_step: the EMA class centres, the
source loss, the fused pseudo-label + target loss), forward + backward with both losses weighted as the trainer weights
them (w_s loss_s + w_t loss_t), single GPU.

    python tools/mpscl_step_bench.py [--iters 30] [--out FILE] [--profile FILE]
    torchrun --nproc_per_node N tools/mpscl_step_bench.py [--iters 30] [--out FILE]

Shapes (per map, K classes): the cfg4 8-GPU shard 16 x 32 x 224^2 K 4, 64 x 32 x 224^2 K 4, cfg2 32 x 128 x 256^2 K 5.
At each shape the script first checks that mpscl_step equals the composition bit for bit (losses, centres, pseudo labels,
mask, both gradients) and exits non-zero otherwise.  It then times four arms alternately in one process -- the
composition and mpscl_step, each eager and as one CUDA graph -- with CUDA events around each step, and reports the median
and the spread (min, max) over --iters runs.  It also records the peak memory of one eager step of each form and, with
--profile, the per-kernel times and launch counts of one eager step of each form from torch.profiler (a separate pass).
The JSON line carries the GPU name and power limit read in the same run.

Under torchrun (N ranks, one GPU each) every rank holds a shard of one global batch: unequal shards (``shard_range`` of
16 N - 1 source and 16 N + 1 target images of 32 x 224^2, K 4).  On both routes (NVLink peer memory: a ``PeerMailbox``;
NCCL: ``group=True``) each rank's losses, centres, pseudo labels, mask and gradients are checked against the global batch
evaluated on that rank's GPU, with identical loss bits on every rank; the script exits non-zero otherwise.  Then every
rank takes its own cfg4 8-GPU shard (16 images per map) and the arms are timed alternately, behind a barrier each: the
composition and mpscl_step over the mailbox, eager and as a CUDA graph, and mpscl_step over NCCL eager; the line reports
the median of each arm, the max over ranks."""
from __future__ import annotations

import argparse
import json
import os
import re
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "soft-labeled-contrastive-learning_b200")]

W_S, W_T, M, TH = 1.0, 0.1, 0.9, 0.25
SHAPES = [("cfg4_shard", 16, 32, 224, 4), ("b64_c32_224", 64, 32, 224, 4), ("cfg2", 32, 128, 256, 5)]


def gpu_info(dev):
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", str(dev.index or 0)],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power = [s.strip() for s in out.split(",")]
    except Exception:
        name, power = torch.cuda.get_device_name(dev), "unknown"
    return name, power


def inputs(b, c, h, k, dev, seed=1):
    g = torch.Generator(device=dev).manual_seed(seed)
    return dict(ft_s=torch.randn(b, c, h, h, device=dev, generator=g),
                labels_s=torch.randint(0, k, (b, h, h), device=dev, generator=g),
                ft_t=torch.randn(b, c, h, h, device=dev, generator=g),
                centres=torch.randn(k, c, device=dev, generator=g))


def modules(k, dev):
    from slcl.loss import MPCL
    return (MPCL(dev, num_class=k, temperature=1.0, m=0.4, base_temperature=1.0),
            MPCL(dev, num_class=k, temperature=1.0, m=0.2, base_temperature=1.0))


def composition(x, mods, k):
    from slcl.loss import mpcl_source_step, mpcl_target_step
    centres, loss_s = mpcl_source_step(x["ft_s"], x["labels_s"], x["centres"], mods[0], m=M, num_class=k)
    loss_t, hard, mask = mpcl_target_step(x["ft_t"], centres.detach(), mods[1], pixel_sel_th=TH)
    return loss_s, loss_t, centres, hard, mask


def fused(x, mods, k):
    from slcl.loss import mpscl_step
    return mpscl_step(x["ft_s"], x["labels_s"], x["ft_t"], x["centres"], mods[0], mods[1], m=M, num_class=k, pixel_sel_th=TH)


def stepper(fn, d, mods, k):
    x = dict(d, ft_s=d["ft_s"].clone().requires_grad_(True), ft_t=d["ft_t"].clone().requires_grad_(True))

    def step():
        x["ft_s"].grad = x["ft_t"].grad = None
        loss_s, loss_t, centres, hard, mask = fn(x, mods, k)
        (W_S * loss_s + W_T * loss_t).backward()
        return [loss_s.detach(), loss_t.detach(), centres.detach(), hard, mask, x["ft_s"].grad, x["ft_t"].grad]
    return step


def graphed(step):
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        step()
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        step()
    return g.replay


def time_arms(arms, iters, barrier=None):
    ev = {name: [] for name in arms}
    for fn in arms.values():
        fn()
    torch.cuda.synchronize()
    for _ in range(iters):
        for name, fn in arms.items():
            if barrier is not None:
                torch.cuda.synchronize()
                barrier()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            b.synchronize()
            ev[name].append(a.elapsed_time(b))
    return {name: dict(median_ms=round(statistics.median(t), 4), min_ms=round(min(t), 4), max_ms=round(max(t), 4))
            for name, t in ev.items()}


def peak_mem(step):
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    step()
    torch.cuda.synchronize()
    return round((torch.cuda.max_memory_allocated() - base) / 2 ** 20, 1)


def profile_step(step):
    from torch.profiler import ProfilerActivity, profile
    step()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        step()
        torch.cuda.synchronize()
    out = {}
    for e in prof.events():
        if e.device_type != torch.autograd.DeviceType.CUDA:
            continue
        m = re.search(r"(\w+)(<[^()]*>)?\(", e.name)           # kernel name and template arguments, without the parameters
        name = (m.group(1) + (m.group(2) or "")) if m else e.name[:80]
        row = out.setdefault(name, dict(count=0, total_us=0.0))
        row["count"] += 1
        row["total_us"] = round(row["total_us"] + e.device_time, 1)
    return dict(launches=sum(v["count"] for v in out.values()), kernels=out)


def composition_group(x, mods, k, group):
    from slcl.loss import mpcl_source_step, mpcl_target_step
    centres, loss_s = mpcl_source_step(x["ft_s"], x["labels_s"], x["centres"], mods[0], m=M, num_class=k, group=group)
    loss_t, hard, mask = mpcl_target_step(x["ft_t"], centres.detach(), mods[1], pixel_sel_th=TH, group=group)
    return loss_s, loss_t, centres, hard, mask


def fused_group(x, mods, k, group):
    from slcl.loss import mpscl_step
    return mpscl_step(x["ft_s"], x["labels_s"], x["ft_t"], x["centres"], mods[0], mods[1], m=M, num_class=k, pixel_sel_th=TH,
                      group=group)


def distributed(args):
    import torch.distributed as dist
    from slcl.distributed import shard_range
    from slcl.peer import PeerMailbox
    dist.init_process_group("nccl")
    rank, world = dist.get_rank(), dist.get_world_size()
    local = int(os.environ.get("LOCAL_RANK", rank))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    box = PeerMailbox(dev)
    b, c, h, k = 16, 32, 224, 4
    mods = modules(k, dev)

    # -- check: sharded == the global batch on this GPU, both routes, unequal shards ------------------------------------
    n_s, n_t = b * world - 1, b * world + 1
    (lo_s, hi_s), (lo_t, hi_t) = shard_range(n_s, rank, world), shard_range(n_t, rank, world)
    g = torch.Generator(device=dev).manual_seed(7)
    d_g = dict(ft_s=torch.randn(n_s, c, h, h, device=dev, generator=g),
               labels_s=torch.randint(0, k, (n_s, h, h), device=dev, generator=g),
               ft_t=torch.randn(n_t, c, h, h, device=dev, generator=g), centres=torch.randn(k, c, device=dev, generator=g))
    ref = stepper(fused, d_g, mods, k)()
    px = h * h
    ref_r = ref[:3] + [ref[3][lo_t * px:hi_t * px], ref[4][lo_t * px:hi_t * px], ref[5][lo_s:hi_s], ref[6][lo_t:hi_t]]
    d_r = dict(d_g, ft_s=d_g["ft_s"][lo_s:hi_s], labels_s=d_g["labels_s"][lo_s:hi_s], ft_t=d_g["ft_t"][lo_t:hi_t])
    checks = {}
    for route, group in (("peer", box), ("nccl", True)):
        got = stepper(lambda x, m_, k_: fused_group(x, m_, k_, group), d_r, mods, k)()
        torch.cuda.synchronize()
        losses = torch.stack([got[0], got[1]])
        every = [torch.zeros_like(losses) for _ in range(world)]
        dist.all_gather(every, losses)
        same_bits = all(torch.equal(e, every[0]) for e in every)
        close = lambda a, r, rtol, atol: bool(torch.allclose(a, r, rtol=rtol, atol=atol))
        ok = (same_bits and bool(torch.isfinite(losses).all()) and close(got[0], ref_r[0], 1e-5, 0)
              and close(got[1], ref_r[1], 1e-5, 0) and close(got[2], ref_r[2], 1e-5, 1e-6)
              and torch.equal(got[3], ref_r[3]) and torch.equal(got[4], ref_r[4])
              and close(got[5], ref_r[5], 1e-5, 1e-9) and close(got[6], ref_r[6], 1e-5, 1e-9))
        checks[route] = {"ok": bool(ok), "same_bits": same_bits, "losses": [float(v) for v in losses],
                         "global_losses_here": [float(ref_r[0]), float(ref_r[1])]}
    checks["timeouts"] = box.timeouts()
    flag = torch.tensor([int(checks["peer"]["ok"] and checks["nccl"]["ok"] and checks["timeouts"] == 0)], device=dev)
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    if not int(flag):
        print(json.dumps({"rank": rank, "check": checks}), flush=True)
        dist.destroy_process_group()
        sys.exit(1)
    del d_g, d_r, ref, ref_r

    # -- timing: each rank its own cfg4 8-GPU shard ------------------------------------------------------------------
    d = inputs(b, c, h, k, dev, seed=100 + rank)
    on = lambda fn, group: (lambda x, m_, k_: fn(x, m_, k_, group))
    comp, step = stepper(on(composition_group, box), d, mods, k), stepper(on(fused_group, box), d, mods, k)
    arms = dict(composition_eager=comp, mpscl_step_eager=step, composition_graph=graphed(comp),
                mpscl_step_graph=graphed(step), mpscl_step_nccl_eager=stepper(on(fused_group, True), d, mods, k))
    m = time_arms(arms, args.iters, barrier=dist.barrier)
    worst = {}
    for a, t in m.items():
        v = torch.tensor([t["median_ms"]], dtype=torch.float64, device=dev)
        dist.all_reduce(v, op=dist.ReduceOp.MAX)
        worst[a] = round(float(v), 4)
    box.check()
    if rank == 0:
        name, power = gpu_info(dev)
        rec = dict(tool="mpscl_step_bench", world=world, gpu=name, power_limit=power, shape_per_rank=[b, c, h * h], n_class=k,
                   check_global_images={"source": n_s, "target": n_t}, check={"peer": True, "nccl": True, "timeouts": 0},
                   iters=args.iters, median_ms_max_over_ranks=worst)
        line = json.dumps(rec)
        print(line, flush=True)
        if args.out:
            with open(args.out, "w") as fh:
                fh.write(line + "\n")
    dist.barrier()
    dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=30)
    ap.add_argument("--out", default=None)
    ap.add_argument("--profile", default=None)
    ap.add_argument("--shapes", default=",".join(s[0] for s in SHAPES))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("mpscl_step_bench needs a CUDA GPU")
    if "WORLD_SIZE" in os.environ:          # under torchrun (with one process the group= calls are single-rank calls)
        return distributed(args)
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    name, power = gpu_info(dev)
    result = dict(tool="mpscl_step_bench", gpu=name, power_limit=power, iters=args.iters, w_s=W_S, w_t=W_T, shapes={})
    prof = dict(gpu=name, power_limit=power, shapes={})
    for tag, b, c, h, k in SHAPES:
        if tag not in args.shapes.split(","):
            continue
        d = inputs(b, c, h, k, dev)
        mods = modules(k, dev)
        comp, step = stepper(composition, d, mods, k), stepper(fused, d, mods, k)
        ref, got = comp(), step()
        names = ("loss_s", "loss_t", "centres", "hard", "mask", "grad_s", "grad_t")
        bad = [n for n, a, r in zip(names, got, ref) if not torch.equal(a, r)]
        if bad:
            raise SystemExit(f"{tag}: mpscl_step differs from mpcl_source_step + mpcl_target_step in {bad}")
        map_mib = b * c * h * h * 4 / 2 ** 20
        row = dict(batch=b, channels=c, hw=h * h, n_class=k, map_mib=round(map_mib, 1), bit_equal=True)
        row["peak_mib"] = dict(composition=peak_mem(comp), mpscl_step=peak_mem(step))
        arms = dict(composition_eager=comp, mpscl_step_eager=step, composition_graph=graphed(comp),
                    mpscl_step_graph=graphed(step))
        row["time"] = time_arms(arms, args.iters)
        result["shapes"][tag] = row
        if args.profile:
            prof["shapes"][tag] = dict(composition=profile_step(comp), mpscl_step=profile_step(step))
        del arms, comp, step, d
        torch.cuda.empty_cache()
        print(json.dumps({tag: row}), flush=True)
    line = json.dumps(result)
    print(line)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(line + "\n")
    if args.profile:
        with open(args.profile, "w") as fh:
            json.dump(prof, fh, indent=1)


if __name__ == "__main__":
    main()
