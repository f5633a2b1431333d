"""MCCL loss section from logits: torch.softmax + cal_centroid against cal_centroid(from_logits=True), one GPU.

    python tools/mccl_logits_bench.py [--rounds 15] [--reps 10]

The section is bench.py's MCCL loss section at the cfg5 geometry (64 x 32 x 224 x 224 per map, K = 4, P = 2
reversed-Monte-Carlo partitions, centroid terms through mccl_centroid_losses), except that both target views start
from segmentor logits [64, 4, 224, 224], as Trainer_MCCL's do (pseudo_label_t = softmax(pred_t)):

  (a) softmax: p = torch.softmax(z, 1), then cal_centroid(ft, p, pseudo_label=True, ...)
  (b) logits:  cal_centroid(ft, z, pseudo_label=True, ..., from_logits=True)

Both run forward and autograd backward to dL/dfeatures and dL/dlogits.  The script first checks that (b) equals (a) at
this size with the tolerances of tests/test_centroid_logits.py (rtol 1e-4; gradients with an absolute floor of
1e-5 * max|grad|) and exits with status 1 on a mismatch.  Then it captures each section in one CUDA graph and times them
alternately (--rounds rounds of --reps replays each, CUDA events), and separately profiles one eager step of each with
torch.profiler for the per-call kernel times of the class-sum sweep and the centroid backward.  One JSON line on stdout,
with the card name and power limit read in the same run.

The logits are 3 * randn with every pixel away from a decision edge (largest probability within 1e-4 of the 0.5
threshold, or top-two logits within 1e-3, redrawn): our softmax and torch's differ in the last bits, and one flipped
certainty moves a centroid by more than the tolerance.
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

B, C, H, K, PARTS, THR = 64, 32, 224, 4, 2, 0.5
COPY_TBPS = 6.52            # measured device-to-device copy bandwidth of a B200 (DESIGN.md), for the prediction only


def edge_free_logits(gen, dev, scale=3.0):
    z = scale * torch.randn(B, K, H, H, device=dev, generator=gen)
    for _ in range(100):
        p = torch.softmax(z, 1)
        top = torch.topk(z, 2, dim=1).values
        bad = ((p.amax(1) - THR).abs() < 1e-4) | ((top[:, 0] - top[:, 1]) < 1e-3)
        n_bad = int(bad.sum())
        if n_bad == 0:
            return z
        zp = z.permute(0, 2, 3, 1)
        zp[bad] = scale * torch.randn(n_bad, K, device=dev, generator=gen)
        z = zp.permute(0, 3, 1, 2).contiguous()
    raise RuntimeError("could not draw logits away from the decision edges")


def make_step(ft, zs, lab_s, part, from_logits):
    from slcl.loss import mccl_centroid_losses
    from slcl.utils_ import cal_centroid

    def step():
        cs, _, _ = cal_centroid(ft[0], lab_s, n_class=K)
        loss = 0
        for i in range(2):
            lab = zs[i] if from_logits else torch.softmax(zs[i], 1)
            ct, _, _ = cal_centroid(ft[1 + i], lab, pseudo_label=True, weighted_ave=True, partition=PARTS, n_class=K,
                                    threshold=THR, part_id=part[i], from_logits=from_logits)
            total, _ = mccl_centroid_losses(cs, ct, None, inter_w=float(PARTS), intra_w=0.0, cnr_w=4e-5)
            loss = loss + total
        loss.backward()
        for t in ft + zs:
            t.grad = None
        return loss.detach()
    return step


def leaves(ft, zs):
    return [t.detach().clone().requires_grad_(True) for t in ft], [t.detach().clone().requires_grad_(True) for t in zs]


def check(ft, zs, lab_s, part):
    """(b) against (a): loss, the three feature-map gradients and the two logit gradients."""
    from slcl.loss import mccl_centroid_losses
    from slcl.utils_ import cal_centroid
    out = []
    for from_logits in (False, True):
        f, z = leaves(ft, zs)
        cs, _, _ = cal_centroid(f[0], lab_s, n_class=K)
        loss = 0
        for i in range(2):
            lab = z[i] if from_logits else torch.softmax(z[i], 1)
            ct, _, _ = cal_centroid(f[1 + i], lab, pseudo_label=True, weighted_ave=True, partition=PARTS, n_class=K,
                                    threshold=THR, part_id=part[i], from_logits=from_logits)
            loss = loss + mccl_centroid_losses(cs, ct, None, inter_w=float(PARTS), intra_w=0.0, cnr_w=4e-5)[0]
        loss.backward()
        out.append([loss.detach()] + [t.grad for t in f + z])
    bad = []
    for i, (a, b) in enumerate(zip(*out)):
        a, b = a.double(), b.double()
        atol = 1e-6 if i == 0 else 1e-5 * float(a.abs().max())
        if not torch.allclose(b, a, rtol=1e-4, atol=atol):
            bad.append({"tensor": ["loss", "dF_s", "dF_t", "dF_t2", "dz_t", "dz_t2"][i],
                        "max_abs_diff": float((b - a).abs().max()), "max_abs": float(a.abs().max())})
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
    """Per-call device time (us) of the kernels of one eager step, by kernel family."""
    from torch.profiler import ProfilerActivity, profile
    step()
    torch.cuda.synchronize(dev)
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(iters):
            step()
        torch.cuda.synchronize(dev)
    fam = {"class_sums_sweep": "class_sums_v3_kernel", "centroid_bwd": "centroid_bwd4_kernel", "softmax": "softmax"}
    out = {}
    for name, key in fam.items():
        evs = [e for e in prof.key_averages() if key in e.key.lower() or key in e.key]
        tot = sum(getattr(e, "device_time_total", getattr(e, "cuda_time_total", 0.0)) for e in evs)
        cnt = sum(e.count for e in evs)
        out[name] = {"calls_per_step": cnt / iters, "us_per_call": (tot / cnt) if cnt else 0.0, "us_per_step": tot / iters}
    evs = [e for e in prof.key_averages() if e.device_type == torch.autograd.DeviceType.CUDA]
    out["all_kernels_us_per_step"] = sum(getattr(e, "self_device_time_total", getattr(e, "self_cuda_time_total", 0.0))
                                         for e in evs) / iters
    return out


def card():
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        info["nvidia_smi"] = q.stdout.strip()
    except (OSError, subprocess.SubprocessError) as exc:
        info["nvidia_smi"] = f"unavailable: {exc!r}"
    return info


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=15)
    ap.add_argument("--reps", type=int, default=10)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        print(json.dumps({"error": "needs a CUDA device"}))
        return 2
    dev = torch.device("cuda:0")
    torch.backends.cuda.matmul.allow_tf32 = False
    gen = torch.Generator(device=dev).manual_seed(4321)
    ft = [torch.randn(B, C, H, H, device=dev, generator=gen) for _ in range(3)]
    lab_s = torch.randint(0, K, (B, H, H), device=dev, generator=gen)
    zs = [edge_free_logits(gen, dev) for _ in range(2)]
    n_px = B * H * H
    part = [(torch.randperm(n_px, device=dev, generator=gen) % PARTS).to(torch.int32) for _ in range(2)]

    mismatch = check(ft, zs, lab_s, part)
    if mismatch:
        print(json.dumps({"equal": False, "mismatch": mismatch}))
        return 1

    # each graph reads its leaves and writes their gradients at fixed addresses: keep the step (and through it the leaves)
    # alive next to its graph, or the next capture's empty_cache() releases that memory under the graph
    graphs, keep = {}, []
    for name, from_logits in (("softmax", False), ("logits", True)):
        f, z = leaves(ft, zs)
        step = make_step(f, z, lab_s, part, from_logits)
        keep.append(step)
        graphs[name] = capture(step, dev)
    times = {"softmax": [], "logits": []}
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    for name in times:                              # warm-up replays
        for _ in range(3):
            graphs[name].replay()
    torch.cuda.synchronize(dev)
    for _ in range(args.rounds):
        for name in ("softmax", "logits"):
            ev[0].record()
            for _ in range(args.reps):
                graphs[name].replay()
            ev[1].record()
            torch.cuda.synchronize(dev)
            times[name].append(ev[0].elapsed_time(ev[1]) / args.reps)

    kern = {}
    for name, from_logits in (("softmax", False), ("logits", True)):
        f, z = leaves(ft, zs)
        kern[name] = kernel_times(make_step(f, z, lab_s, part, from_logits), dev)

    def summary(v):
        s = sorted(v)
        return {"median_ms": statistics.median(s), "min_ms": s[0], "max_ms": s[-1],
                "iqr_ms": s[(3 * len(s)) // 4] - s[len(s) // 4]}
    med_a, med_b = statistics.median(times["softmax"]), statistics.median(times["logits"])
    bytes_saved = 2 * 20 * K * n_px                  # per view: softmax fwd 8K B/px (read z, write p) + bwd 12K (p, dp -> dz)
    print(json.dumps({
        "equal": True,
        "workload": "cfg5 MCCL loss section from logits, one GPU: hard source centroids + 2 target views "
                    f"[{B}, {C}, {H}, {H}], K={K}, P={PARTS}, threshold {THR}, weighted, mccl_centroid_losses; "
                    "forward + backward to dF and dlogits, each variant one CUDA graph, timed alternately",
        "softmax_then_cal_centroid": summary(times["softmax"]),
        "cal_centroid_from_logits": summary(times["logits"]),
        "saved_ms_median": med_a - med_b,
        "kernels": kern,
        "bytes": {"pixels_per_view": n_px, "softmax_fwd_bwd_bytes_per_px_per_view": 20 * K,
                  "removed_bytes_two_views": bytes_saved,
                  "predicted_saving_ms_at_copy_bw": bytes_saved / (COPY_TBPS * 1e12) * 1e3},
        "rounds": args.rounds, "reps_per_round": args.reps,
        "card": card(),
    }))
    return 0


if __name__ == "__main__":
    sys.exit(main())
