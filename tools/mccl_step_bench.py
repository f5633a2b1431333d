"""mccl_step against the composition it replaces (cal_centroid x 3 + mccl_centroid_losses), forward + backward, at the
cfg5 geometry per GPU (configs[4]: 64 x 32 x 224 x 224 maps, K = 4, P = 2), from logits, aug view included.

    python tools/mccl_step_bench.py [--iters 15] [--out profiles/mccl_step_bench.json]
    torchrun --nproc_per_node N tools/mccl_step_bench.py [--iters 15] [--out FILE]

Arms: (a) the composition eager, (b) the composition as one CUDA graph, (c) mccl_step eager, (d) mccl_step as one CUDA
graph.  The four arms are first checked to give the same loss and the same gradients into the four differentiable
inputs, then timed alternately in one process with CUDA events around each step (median over --iters runs of each
arm).  Eager steps include the host time of every call, which is what a trainer without graphs pays.  The JSON line
records the GPU name and its power limit.

Under torchrun (N > 1) every rank holds its own cfg5 batch, and the script first checks, on both routes (NVLink peer
memory: ``PeerMailbox``; NCCL: ``group=True``), that each rank's loss, terms and centroids equal the global batch
evaluated on that rank's GPU and that its gradients are its shard of the global gradients, with unequal shards
(``shard_range`` of 64 N - 1 images) and identical loss bits on every rank; it exits non-zero otherwise.  Then it times
the four arms with the peer mailbox as the group, plus mccl_step over NCCL, each time the max over ranks."""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "soft-labeled-contrastive-learning_b200")]

C, H, K, P, THR = 32, 224, 4, 2, 0.5
LEAVES = ("ft_t", "ft_a", "pred_t", "pred_a")


def gpu_info(dev):
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", str(dev.index or 0)],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power = [s.strip() for s in out.split(",")]
    except Exception:
        name, power = torch.cuda.get_device_name(dev), "unknown"
    return name, power


def inputs(b, dev, seed=1):
    g = torch.Generator(device=dev).manual_seed(seed)
    d = dict(ft_s=torch.randn(b, C, H, H, device=dev, generator=g),
             labels_s=torch.randint(0, K, (b, H, H), device=dev, generator=g),
             ft_t=torch.randn(b, C, H, H, device=dev, generator=g),
             pred_t=3 * torch.randn(b, K, H, H, device=dev, generator=g),
             ft_a=torch.randn(b, C, H, H, device=dev, generator=g),
             pred_a=3 * torch.randn(b, K, H, H, device=dev, generator=g),
             part_id=(torch.randperm(b * H * H, device=dev, generator=g) % P).to(torch.int32),
             prev=torch.randn(K, C, device=dev, generator=g))
    return d


def shard(d, lo, hi):
    s = {key: (v[lo:hi].contiguous() if key not in ("part_id", "prev") else v) for key, v in d.items()}
    s["part_id"] = d["part_id"].reshape(-1, H * H)[lo:hi].reshape(-1).contiguous()
    return s


def leaves(d):
    x = dict(d)
    for key in LEAVES:
        x[key] = d[key].detach().clone().requires_grad_(True)
    return x


def composition(d, group=None):
    from slcl.loss import mccl_centroid_losses
    from slcl.utils_ import cal_centroid
    cs, _, _ = cal_centroid(d["ft_s"], d["labels_s"], previous_centroid=d["prev"], momentum=0.95, n_class=K, group=group)
    ct, _, _ = cal_centroid(d["ft_t"], d["pred_t"], pseudo_label=True, partition=P, threshold=THR, weighted_ave=True,
                            n_class=K, part_id=d["part_id"], from_logits=True, group=group)
    ca, _, _ = cal_centroid(d["ft_a"], d["pred_a"], pseudo_label=True, threshold=THR, weighted_ave=True, n_class=K,
                            from_logits=True, group=group)
    total, terms = mccl_centroid_losses(cs.detach(), ct, ca)
    return total, terms, torch.cat([cs.detach(), torch.cat(ct).detach(), ca.detach()])


def fused(d, group=None):
    from slcl.loss import mccl_step
    total, terms, cs, ct, ca = mccl_step(d["ft_s"], d["labels_s"], d["ft_t"], d["pred_t"], d["ft_a"], d["pred_a"], n_class=K,
                                         partition=P, part_id=d["part_id"], threshold=THR, previous_centroid_s=d["prev"],
                                         momentum=0.95, group=group)
    return total, terms, torch.cat([cs, torch.cat(ct), ca])


def fwd_bwd(fn, d, group=None):
    x = leaves(d)
    total, terms, cen = fn(x, group)
    total.backward()
    return total.detach(), terms.detach(), cen, [x[key].grad for key in LEAVES]


def grads_close(got, ref, rtol=1e-5):
    return all(torch.allclose(a, r, rtol=rtol, atol=rtol * 0.1 * float(r.abs().max())) for a, r in zip(got, ref))


def check_arms(d, dev):
    """-> the four timed callables after checking that they give the same loss and gradients."""
    x = leaves(d)
    grads = [x[key] for key in LEAVES]

    def step(fn):
        def run():
            for t in grads:
                t.grad = None
            total = fn(x)[0]
            total.backward()
            return total.detach()
        return run
    ref_total, _, _, ref_g = fwd_bwd(composition, d)
    for name, fn in (("composition", composition), ("mccl_step", fused)):
        got = step(fn)()
        if not (torch.allclose(got, ref_total, rtol=1e-6, atol=0) and grads_close([t.grad for t in grads], ref_g)):
            raise SystemExit(f"eager {name} differs from the composition")
    graphs = {}
    for name, fn in (("composition", composition), ("mccl_step", fused)):
        side = torch.cuda.Stream(dev)
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            step(fn)()
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        for t in grads:
            t.grad = None
        gr = torch.cuda.CUDAGraph()
        with torch.cuda.graph(gr):
            static = fn(x)[0]
            static.backward()
        gr.replay()
        torch.cuda.synchronize()
        if not (torch.allclose(static.detach(), ref_total, rtol=1e-6, atol=0) and grads_close([t.grad for t in grads], ref_g)):
            raise SystemExit(f"{name} as a CUDA graph differs from the composition")
        graphs[name] = gr
    return {"a_composition_eager": step(composition), "b_composition_graph": graphs["composition"].replay,
            "c_mccl_step_eager": step(fused), "d_mccl_step_graph": graphs["mccl_step"].replay}


def time_arms(arms, iters, barrier=None):
    for fn in arms.values():             # warm-up
        for _ in range(3):
            fn()
    torch.cuda.synchronize()
    times = {name: [] for name in arms}
    for _ in range(iters):
        for name, fn in arms.items():
            if barrier is not None:
                barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            e0.record()
            fn()
            e1.record()
            e1.synchronize()
            times[name].append(e0.elapsed_time(e1))
    return {a: statistics.median(t) for a, t in times.items()}


def speedups(m):
    return {"eager_speedup": round(m["a_composition_eager"] / m["c_mccl_step_eager"], 3),
            "graph_speedup": round(m["b_composition_graph"] / m["d_mccl_step_graph"], 3),
            "mccl_step_eager_over_graph": round(m["c_mccl_step_eager"] / m["d_mccl_step_graph"], 3)}


def write(line, out):
    print(line, flush=True)
    if out:
        os.makedirs(os.path.dirname(os.path.abspath(out)), exist_ok=True)
        with open(out, "w") as fh:
            fh.write(line + "\n")


def single(args):
    dev = torch.device("cuda")
    d = inputs(args.batch, dev)
    arms = check_arms(d, dev)
    m = time_arms(arms, args.iters)
    name, power = gpu_info(dev)
    rec = {"tool": "mccl_step_bench", "gpu": name, "power_limit": power, "geometry": [args.batch, C, H, H], "n_class": K,
           "partition": P, "from_logits": True, "aug": True, "iters": args.iters,
           "median_ms": {a: round(t, 4) for a, t in m.items()}}
    rec.update(speedups(m))
    write(json.dumps(rec), args.out)


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

    # -- check: sharded == the global batch on this GPU, both routes, unequal shards ------------------------------------
    n_global = args.batch * world - 1
    lo, hi = shard_range(n_global, rank, world)
    d_g = inputs(n_global, dev, seed=7)
    ref_total, ref_terms, ref_cen, ref_g = fwd_bwd(fused, d_g)
    ref_g = [t[lo:hi] for t in ref_g]
    d_r = shard(d_g, lo, hi)
    checks = {}
    for route, group in (("peer", box), ("nccl", True)):
        total, terms, cen, g = fwd_bwd(fused, d_r, group)
        torch.cuda.synchronize()
        every = [torch.zeros_like(total) for _ in range(world)]
        dist.all_gather(every, total)
        same_bits = all(torch.equal(e, every[0]) for e in every)
        ok = (same_bits and bool(torch.isfinite(total)) and torch.allclose(total, ref_total, rtol=1e-5, atol=0)
              and torch.allclose(terms, ref_terms, rtol=1e-5, atol=1e-7) and torch.allclose(cen, ref_cen, rtol=1e-5, atol=1e-6)
              and grads_close(g, ref_g))
        checks[route] = {"ok": bool(ok), "same_bits": same_bits, "total": float(total), "global_total_here": float(ref_total)}
    checks["timeouts"] = box.timeouts()
    flag = torch.tensor([int(checks["peer"]["ok"] and checks["nccl"]["ok"] and checks["timeouts"] == 0)], device=dev)
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    if not int(flag):
        print(json.dumps({"rank": rank, "check": checks}), flush=True)
        dist.destroy_process_group()
        sys.exit(1)
    del d_g, d_r, ref_g

    # -- timing: each rank its own cfg5 batch; the four arms over the mailbox, mccl_step over NCCL -----------------------
    d = inputs(args.batch, dev, seed=100 + rank)
    x = leaves(d)
    grads = [x[key] for key in LEAVES]
    arms = {}
    for name, fn, group in (("a_composition_eager", composition, box), ("c_mccl_step_eager", fused, box),
                            ("e_mccl_step_nccl_eager", fused, True)):
        def run(fn=fn, group=group):
            for t in grads:
                t.grad = None
            fn(x, group)[0].backward()
        arms[name] = run
    for name, fn in (("b_composition_graph", composition), ("d_mccl_step_graph", fused)):
        side = torch.cuda.Stream(dev)
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            fn(x, box)[0].backward()
        torch.cuda.current_stream().wait_stream(side)
        torch.cuda.synchronize()
        for t in grads:
            t.grad = None
        gr = torch.cuda.CUDAGraph()
        with torch.cuda.graph(gr):
            fn(x, box)[0].backward()
        arms[name] = gr.replay
    m = time_arms(dict(sorted(arms.items())), args.iters, barrier=dist.barrier)
    worst = {}
    for a, t in m.items():
        v = torch.tensor([t], dtype=torch.float64, device=dev)
        dist.all_reduce(v, op=dist.ReduceOp.MAX)
        worst[a] = float(v)
    box.check()
    if rank == 0:
        name, power = gpu_info(dev)
        rec = {"tool": "mccl_step_bench", "world": world, "gpu": name, "power_limit": power,
               "geometry_per_rank": [args.batch, C, H, H], "n_class": K, "partition": P, "from_logits": True, "aug": True,
               "check_global_images": n_global, "check": {"peer": True, "nccl": True, "timeouts": 0}, "iters": args.iters,
               "median_ms_max_over_ranks": {a: round(t, 4) for a, t in worst.items()}}
        rec.update(speedups(worst))
        write(json.dumps(rec), args.out)
    dist.barrier()
    dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=15)
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--out", default=None, help="default: profiles/mccl_step_bench.json without torchrun")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("mccl_step_bench needs a CUDA device")
    if "WORLD_SIZE" in os.environ:          # under torchrun (with one process the group= calls are single-rank calls)
        distributed(args)
    else:
        if args.out is None:
            args.out = os.path.join(ROOT, "profiles", "mccl_step_bench.json")
        single(args)


if __name__ == "__main__":
    main()
