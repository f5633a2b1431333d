"""AdvEnt entropy maps from logits: torch.softmax + prob_2_entropy against prob_2_entropy(from_logits=True), one GPU.

    python tools/entropy_logits_bench.py [--rounds 15] [--reps 10]

Trainer_MPSCL's adversarial branch makes entropy maps of the segmentor's logits two ways: the generator step feeds
d_main(prob_2_entropy(F.softmax(pred_trg))) and back-propagates through it into the logits (Trainer_MPSCL.py:171-191),
and the discriminator updates take prob_2_entropy(F.softmax(pred.detach())), forward only (:202-278).  One "step" here is
one of each, on logits [B, 4, 224, 224]:

  (a) chain: e = prob_2_entropy(torch.softmax(z, 1)), backward of e with a fixed upstream gradient into z, plus
      prob_2_entropy(torch.softmax(z_src, 1)) under no_grad;
  (b) fused: the same with prob_2_entropy(z, from_logits=True).

B = 16 is the cfg4 per-GPU shard, B = 64 the cfg5 geometry.  The script first checks that (b) equals (a) at each size
with the tolerances of tests/test_entropy_logits.py (map rtol 1e-5 / atol 1e-6; gradient rtol 1e-5 with an absolute
floor of 1e-5 * max|grad|) and exits with status 1 on a mismatch.  Then it captures each step in one CUDA graph and times
the two alternately (--rounds rounds of --reps replays each, CUDA events), profiles one eager step of each with
torch.profiler for the per-kernel times, and records the peak memory one eager step allocates beyond its inputs.  One
JSON line on stdout, with the card name and power limit read in the same run.

At B = 16 a step's working set (five or six 12.8 MB maps) fits in the 126 MB L2, so those times are partly L2 times; at
B = 64 every map is 51 MB and the step's maps do not fit.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for _p in (ROOT, os.path.join(ROOT, "soft-labeled-contrastive-learning_b200")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import torch  # noqa: E402

K, H = 4, 224
BATCHES = (16, 64)
COPY_TBPS = 6.52            # measured device-to-device copy bandwidth of a B200 (DESIGN.md), for the prediction only
BYTES_PER_PX = {"chain": 56 * K, "fused": 28 * K}   # fwd+bwd map 40K vs 20K, forward-only map 16K vs 8K


def make_step(z, z_src, w, fused):
    from slcl.seg import prob_2_entropy

    def step():
        e = prob_2_entropy(z, from_logits=True) if fused else prob_2_entropy(torch.softmax(z, 1))
        torch.autograd.backward(e, w)
        with torch.no_grad():
            e_src = prob_2_entropy(z_src, from_logits=True) if fused else prob_2_entropy(torch.softmax(z_src, 1))
        z.grad = None
        return e.detach(), e_src
    return step


def check(z0, z_src, w):
    """(b) against (a): the map with gradient, its dL/dz, and the forward-only map."""
    from slcl.seg import prob_2_entropy
    out = []
    for fused in (False, True):
        z = z0.detach().clone().requires_grad_(True)
        e = prob_2_entropy(z, from_logits=True) if fused else prob_2_entropy(torch.softmax(z, 1))
        torch.autograd.backward(e, w)
        with torch.no_grad():
            e_src = prob_2_entropy(z_src, from_logits=True) if fused else prob_2_entropy(torch.softmax(z_src, 1))
        out.append([e.detach(), z.grad, e_src])
    bad = []
    for name, a, b in zip(("map", "dlogits", "map_no_grad"), *out):
        a, b = a.double(), b.double()
        atol = 1e-5 * float(a.abs().max()) if name == "dlogits" else 1e-6
        if not torch.allclose(b, a, rtol=1e-5, atol=atol):
            bad.append({"tensor": name, "max_abs_diff": float((b - a).abs().max()), "max_abs": float(a.abs().max())})
    return bad


def capture(step, dev):
    side = torch.cuda.Stream(dev)
    side.wait_stream(torch.cuda.current_stream(dev))
    with torch.cuda.stream(side):
        step()
    torch.cuda.current_stream(dev).wait_stream(side)
    torch.cuda.synchronize(dev)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        step()
    return graph


def kernel_times(step, dev, iters=3):
    """Per-call device time (us) of every kernel of one eager step."""
    from torch.profiler import ProfilerActivity, profile
    step()
    torch.cuda.synchronize(dev)
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(iters):
            step()
        torch.cuda.synchronize(dev)
    acc = {}
    for e in prof.key_averages():
        if e.device_type != torch.autograd.DeviceType.CUDA:
            continue
        t = getattr(e, "self_device_time_total", getattr(e, "self_cuda_time_total", 0.0))
        name = e.key.replace("(anonymous namespace)::", "").replace("void ", "").split("(")[0][:120]
        tot, cnt = acc.get(name, (0.0, 0))
        acc[name] = (tot + t, cnt + e.count)
    out = {name: {"calls_per_step": cnt / iters, "us_per_call": tot / cnt if cnt else 0.0} for name, (tot, cnt) in acc.items()}
    out["all_kernels_us_per_step"] = sum(tot for tot, _ in acc.values()) / iters
    return out


def peak_bytes(step, dev):
    """Memory one eager step allocates beyond what is live before it (its outputs included)."""
    torch.cuda.synchronize(dev)
    base = torch.cuda.memory_allocated(dev)
    torch.cuda.reset_peak_memory_stats(dev)
    res = step()
    torch.cuda.synchronize(dev)
    peak = torch.cuda.max_memory_allocated(dev) - base
    del res
    return peak


def card():
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        info["nvidia_smi"] = q.stdout.strip()
    except (OSError, subprocess.SubprocessError) as exc:
        info["nvidia_smi"] = f"unavailable: {exc!r}"
    return info


def summary(v):
    s = sorted(v)
    return {"median_ms": statistics.median(s), "min_ms": s[0], "max_ms": s[-1], "iqr_ms": s[(3 * len(s)) // 4] - s[len(s) // 4]}


def run_shape(b, args, dev):
    gen = torch.Generator(device=dev).manual_seed(2024 + b)
    z = 3 * torch.randn(b, K, H, H, device=dev, generator=gen)
    z_src = 3 * torch.randn(b, K, H, H, device=dev, generator=gen)
    w = torch.randn(b, K, H, H, device=dev, generator=gen)
    n_px = b * H * H
    mismatch = check(z, z_src, w)
    if mismatch:
        return {"batch": b, "equal": False, "mismatch": mismatch}

    # each graph reads its leaf and writes its gradient at fixed addresses: keep the step (and through it the leaf)
    # alive next to its graph
    graphs, keep = {}, []
    for name in ("chain", "fused"):
        step = make_step(z.clone().requires_grad_(True), z_src, w, name == "fused")
        keep.append(step)
        graphs[name] = capture(step, dev)
    times = {"chain": [], "fused": []}
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    for name in times:                              # warm-up replays
        for _ in range(3):
            graphs[name].replay()
    torch.cuda.synchronize(dev)
    for _ in range(args.rounds):
        for name in ("chain", "fused"):
            ev[0].record()
            for _ in range(args.reps):
                graphs[name].replay()
            ev[1].record()
            torch.cuda.synchronize(dev)
            times[name].append(ev[0].elapsed_time(ev[1]) / args.reps)
    del graphs, keep
    torch.cuda.synchronize(dev)

    kern, peak = {}, {}
    for name in ("chain", "fused"):
        step = make_step(z.clone().requires_grad_(True), z_src, w, name == "fused")
        kern[name] = kernel_times(step, dev)
        peak[name] = peak_bytes(step, dev)
    med = {name: statistics.median(v) for name, v in times.items()}
    return {
        "batch": b, "equal": True, "logits": [b, K, H, H],
        "chain_ms": summary(times["chain"]), "fused_ms": summary(times["fused"]),
        "saved_ms_median": med["chain"] - med["fused"],
        "kernels": kern,
        "peak_step_bytes": peak,
        "bytes": {"pixels": n_px, "bytes_per_px": BYTES_PER_PX,
                  "step_bytes": {k: v * n_px for k, v in BYTES_PER_PX.items()},
                  "floor_ms_at_copy_bw": {k: v * n_px / (COPY_TBPS * 1e12) * 1e3 for k, v in BYTES_PER_PX.items()},
                  "achieved_tbps": {k: BYTES_PER_PX[k] * n_px / (med[k] * 1e-3) / 1e12 for k in med}},
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=15)
    ap.add_argument("--reps", type=int, default=10)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        print(json.dumps({"error": "needs a CUDA device"}))
        return 2
    dev = torch.device("cuda:0")
    shapes = [run_shape(b, args, dev) for b in BATCHES]
    equal = all(s["equal"] for s in shapes)
    print(json.dumps({
        "equal": equal,
        "workload": "AdvEnt entropy maps from logits [B, 4, 224, 224]: one map forward + backward into the logits plus one "
                    "forward-only map; torch.softmax + prob_2_entropy vs prob_2_entropy(from_logits=True); each variant "
                    "one CUDA graph, timed alternately",
        "shapes": shapes,
        "rounds": args.rounds, "reps_per_round": args.reps,
        "card": card(),
    }))
    return 0 if equal else 1


if __name__ == "__main__":
    sys.exit(main())
