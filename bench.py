#!/usr/bin/env python
"""bench.py -- SLCL loss fwd+bwd pixels/sec on B200 (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W          # product arm (CUDA kernels)
    python bench.py --impl reference --gpus N --steps K --warmup W   # CPU reference arm
    python bench.py ... --dump-outputs DIR     # also write the last timed step's outputs as DIR/*.npy (either arm)

Workload at every N (weak scaling, one process per GPU): BASELINE.json configs[1] --
"SLCL prototype path at 256x256 full-res 128-d embeddings, batch 32, 5 classes" (cfg2 of
SURVEY.md 8): per GPU a [32,128,256,256] fp32 NCHW feature map (1.07 GB), int64 labels,
fp32 pixel-selection mask, [5,128] class centres, T=0.1, base_T=1, m=0.2.

A step = one forward + backward of the prototype loss (reference mpcl_loss_calc + MPCL.forward,
utils/loss.py:576-605,484-573 and its autograd backward): 3 forward launches (centre prep, fused
loss, finalise) + 1 backward launch; with N>1 the loss is the mean over the GLOBAL batch, so one
8-byte exchange sits between forward and backward -- done inside the forward's own finaliser kernel over NVLink peer
memory (slcl_proto_fwd_peer), or by an NCCL all-reduce + rescale launch when symmetric memory is unavailable.

Prints ONE JSON line (rank 0).  Timing: CUDA events on the launching stream, barrier +
synchronize on both sides, max over ranks.  No L2 flush is needed: every step streams
1.07 GB (> 126 MB L2) of input.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG_DIR = os.path.join(ROOT, "soft-labeled-contrastive-learning_b200")
for _p in (ROOT, PKG_DIR):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import torch  # noqa: E402

METRIC = "SLCL loss fwd+bwd pixels/sec"
UNIT = "pixels/s"
E2E_CHUNK = int(os.environ.get("SLCL_E2E_CHUNK", "2"))      # images per pipeline chunk of the host-buffer path
CFG = dict(B=32, C=128, H=256, W=256, K=5, temperature=0.1, base_temperature=1.0, margin=0.2, seed=1234)
WORKLOAD = ("cfg2: SLCL prototype path (mpcl_loss_calc+MPCL fwd+bwd, target variant with pixel_sel_loc), "
            "B32 C128 256x256 K5 fp32 NCHW per GPU")
FALLBACK_HBM_GBS = 6650.0        # B200_PROFILING.md fallback when MEASURED_PEAKS.json is absent
DUMP_SAMPLE = 1 << 21            # dL/dF elements --dump-outputs writes (8 MB of the 1.07 GB map, + 16 MB of positions)


def base_config(world: int):
    """`config` of the JSON line: identical for the product arm and the reference arm (same workload, same batch)."""
    B, C, H, W, K = CFG["B"], CFG["C"], CFG["H"], CFG["W"], CFG["K"]
    return {"workload": WORKLOAD, "B_per_gpu": B, "C": C, "H": H, "W": W, "K": K, "pixels_per_gpu": B * H * W,
            "temperature": CFG["temperature"], "base_temperature": CFG["base_temperature"], "margin": CFG["margin"],
            "parallelism": f"dp{world} (batch sharded, one process per GPU)" if world > 1 else "single GPU",
            "l2": "no flush: each step streams a 1.07 GB feature map (> 126 MB L2)"}


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="slcl", choices=["slcl", "reference"])
    ap.add_argument("--cpu-sample-images", type=int, default=CFG["B"],
                    help="images of the cfg2 shape per CPU step (default: the full batch of 32, the product arm's config)")
    ap.add_argument("--no-extras", action="store_true", help="skip the per-kernel table of the other path kernels")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step returned as DIR/<name>.npy (rank 0; "
                         "either arm, same names): loss.npy and a fixed, seeded sample of dL/dF (see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


def hbm_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as fh:
            return float(json.load(fh)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return FALLBACK_HBM_GBS, "fallback (B200_PROFILING.md)"


def ncu_traffic(kernel: str):
    """Per-launch DRAM bytes of `kernel` from the committed ncu --set full summary, if any."""
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_summary.json")) as fh:
            return json.load(fh)["kernels"][kernel]["dram_bytes_per_launch"]
    except Exception:
        return None


# ----------------------------------------------------------------------------
# synthetic inputs (SURVEY.md 8(d)): CPU generator -> identical bits for oracle and GPU
# ----------------------------------------------------------------------------
def make_inputs(n_images: int, seed: int, pin: bool):
    gen = torch.Generator().manual_seed(seed)
    c, h, w, k = CFG["C"], CFG["H"], CFG["W"], CFG["K"]
    feats = torch.empty((n_images, c, h, w), dtype=torch.float32, pin_memory=pin)
    feats.normal_(generator=gen)
    labels = torch.empty((n_images * h * w,), dtype=torch.int64, pin_memory=pin)
    labels.random_(0, k, generator=gen)
    sel = torch.empty((n_images * h * w,), dtype=torch.float32, pin_memory=pin)
    sel.copy_((torch.rand(n_images * h * w, generator=gen) > 0.5).float())
    centres = torch.randn(k, c, generator=gen)
    return feats, labels, sel, centres


def dump_outputs(out_dir: str, dfeat: torch.Tensor, **arrays: torch.Tensor):
    """--dump-outputs: what one step hands its caller, so that two builds -- or the two arms, whose inputs are the same
    with the default --cpu-sample-images -- can be compared output for output on the same seeded inputs.  Each of
    `arrays` goes to <name>.npy as fp32 (both arms write loss.npy; the product arm adds scal.npy, the forward's four
    scalars: loss, coefficient, weight sum, weighted row-loss sum); dfeat_sample.npy: dL/dF at DUMP_SAMPLE flat NCHW
    positions drawn with a fixed seed, which dfeat_sample_index.npy lists (float64, exact below 2**53)."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    flat = dfeat.detach().reshape(-1)
    idx = torch.randint(0, flat.numel(), (min(DUMP_SAMPLE, flat.numel()),),
                        generator=torch.Generator().manual_seed(CFG["seed"])).sort().values
    for name, value in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), value.detach().float().cpu().numpy())
    np.save(os.path.join(out_dir, "dfeat_sample.npy"), flat[idx.to(flat.device)].float().cpu().numpy())
    np.save(os.path.join(out_dir, "dfeat_sample_index.npy"), idx.double().numpy())


# ----------------------------------------------------------------------------
# clocks sampler (NVML, same fields as the nvidia-smi line of B200_PROFILING.md)
# ----------------------------------------------------------------------------
class ClockSampler:
    def __init__(self, index: int, period_s: float = 0.005):
        self.samples = []
        self.period = period_s
        self.stop_flag = threading.Event()
        self.ok = False
        try:
            import pynvml
            self.nv = pynvml
            pynvml.nvmlInit()
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception as e:                                   # pragma: no cover
            self.err = repr(e)
        self.thread = threading.Thread(target=self._run, daemon=True)

    def _run(self):
        nv = self.nv
        while not self.stop_flag.is_set():
            try:
                mhz = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
                try:
                    reasons = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    reasons = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                util = nv.nvmlDeviceGetUtilizationRates(self.h).gpu
                self.samples.append((time.perf_counter(), mhz, reasons, util))
            except Exception:
                pass
            time.sleep(self.period)

    def start(self):
        if self.ok:
            self.thread.start()
            self.started = True

    def stop(self):
        self.stop_flag.set()
        if self.ok and getattr(self, "started", False):
            self.thread.join(timeout=2)

    def summary(self, t0: float, t1: float):
        if not self.ok:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvml unavailable"]}
        nv = self.nv
        inside = [s for s in self.samples if t0 <= s[0] <= t1]
        where = "timed region"
        if len(inside) < 3:          # timed region shorter than the sampling period: use every sample under load
            inside = [s for s in self.samples if s[3] > 0] or self.samples
            where = "whole run under load (timed region too short to sample)"
        names = {
            getattr(nv, "nvmlClocksEventReasonGpuIdle", 0x1): "gpu_idle",
            getattr(nv, "nvmlClocksEventReasonApplicationsClocksSetting", 0x2): "applications_clocks_setting",
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
            getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksEventReasonSyncBoost", 0x10): "sync_boost",
            getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksThrottleReasonHwPowerBrakeSlowdown", 0x80): "hw_power_brake_slowdown",
        }
        mask = 0
        for s in inside:
            mask |= int(s[2])
        reasons = sorted(n for bit, n in names.items() if mask & bit and n != "gpu_idle")
        return {"sm_mhz": statistics.median(s[1] for s in inside) if inside else None, "sm_max_mhz": self.max_mhz,
                "reasons": reasons, "samples": len(inside), "sampled_over": where}


# ----------------------------------------------------------------------------
# CPU baseline: the oracle port of the reference's own call sequence
# ----------------------------------------------------------------------------
def cpu_step_fn(n_images: int):
    from oracle import slcl_oracle as O
    feats, labels, sel, centres = make_inputs(n_images, CFG["seed"], pin=False)
    spec = O.MarginSpec(num_class=CFG["K"], temperature=CFG["temperature"], m=CFG["margin"],
                        base_temperature=CFG["base_temperature"])
    feats.requires_grad_(True)

    def step():
        feats.grad = None
        loss = O.mpcl_loss_calc(feats, labels, centres, spec, pixel_sel_loc=sel, tag="target")
        loss.backward()
        return loss.detach(), feats.grad
    return step, n_images * CFG["H"] * CFG["W"]


def time_cpu(n_images: int, warmup: int, steps: int):
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    step, pixels = cpu_step_fn(n_images)
    for _ in range(warmup):
        step()
    times = []
    for _ in range(steps):
        t0 = time.perf_counter()
        out = step()
        times.append(time.perf_counter() - t0)
    return pixels, times, cores, out           # out: (loss, dL/dF) of the last timed step


def time_torch_eager_gpu(dev, feats, labels, sel, centres, iters: int = 5):
    """SURVEY 8(d) second comparator: the reference's own op sequence (oracle port: same ATen calls, same order) run as
    plain eager PyTorch on the SAME GPU and the SAME resident cfg2 batch.  Reported beside the CPU arm; never on the
    product path.  Also a full-size loss check of the CUDA path against eager fp32."""
    from oracle import slcl_oracle as O
    spec = O.MarginSpec(num_class=CFG["K"], temperature=CFG["temperature"], m=CFG["margin"],
                        base_temperature=CFG["base_temperature"])
    x = feats.detach().clone().requires_grad_(True)

    def step():
        x.grad = None
        loss = O.mpcl_loss_calc(x, labels, centres, spec, pixel_sel_loc=sel, tag="target")
        loss.backward()
        return loss.detach()
    for _ in range(2):
        step()
    torch.cuda.synchronize(dev)
    times = []
    for _ in range(iters):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        loss = step()
        e1.record()
        torch.cuda.synchronize(dev)
        times.append(e0.elapsed_time(e1))
    grad = x.grad
    x.grad = None
    return min(times), float(loss), grad


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    n_img = args.cpu_sample_images
    pixels, times, cores, (loss, dfeat) = time_cpu(n_img, max(args.warmup, 1), args.steps)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, dfeat, loss=loss.reshape(1))
    total = sum(times)
    value = pixels * len(times) / total
    sample = (("the full cfg2 batch per step" if n_img == CFG["B"] else f"{n_img} of the 32 images of the cfg2 batch per step")
              + f" ({pixels} px, same shapes/hyper-parameters); oracle port of mpcl_loss_calc+MPCL.forward fwd+bwd "
                f"(torch CPU ops, fp32, {cores} threads)")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * total / len(times), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": base_config(args.gpus),
        "note": "CPU arm: the reference's op sequence (oracle port: the original project is a script collection, not an "
                "installable package) on the box's host cores, rank 0 only",
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------
# product arm
# ----------------------------------------------------------------------------
def run_slcl(args):
    import torch.distributed as dist
    from slcl import ops  # noqa: F401
    from slcl.loss import MPCL, mpcl_loss_calc
    from slcl.plan import ProtoPlan

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py (product arm) needs a CUDA device; there is no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    # one slice of the host cores per rank, set BEFORE the pinned buffers are first touched (NUMA placement follows the
    # touching thread); SLCL_BENCH_AFFINITY=0 leaves the scheduler alone
    affinity = "unchanged"
    if world > 1 and os.environ.get("SLCL_BENCH_AFFINITY", "1") != "0" and hasattr(os, "sched_setaffinity"):
        try:
            cpus = sorted(os.sched_getaffinity(0))
            per = max(1, len(cpus) // world)
            mine = cpus[local_rank * per:(local_rank + 1) * per] or cpus
            os.sched_setaffinity(0, mine)
            affinity = f"rank pinned to {len(mine)} of {len(cpus)} host cpus ({mine[0]}..{mine[-1]})"
        except Exception as exc:  # noqa: BLE001
            affinity = f"unchanged ({exc!r})"
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    B, C, H, W, K = CFG["B"], CFG["C"], CFG["H"], CFG["W"], CFG["K"]
    n_px = B * H * W
    feats_h, labels_h, sel_h, centres_h = make_inputs(B, CFG["seed"] + rank, pin=True)
    feats = feats_h.to(dev, non_blocking=True)
    labels = labels_h.to(dev, non_blocking=True)
    sel = sel_h.to(dev, non_blocking=True)
    centres = centres_h.to(dev)
    # Timed loop: raw C-ABI launches on pre-allocated buffers (slcl.plan.ProtoPlan) so the host
    # never gates the GPU; the torch custom-op / autograd route is what `e2e` measures.
    plan = ProtoPlan(feats, labels, sel, centres, K, CFG["temperature"], CFG["base_temperature"], CFG["margin"])

    ev = lambda: torch.cuda.Event(enable_timing=True)
    marks = []

    # N > 1: the 8-byte exchange between forward and backward goes through NVLink peer memory inside our own rescale kernel
    # (slcl_proto_rescale_peer); NCCL all-reduce + rescale when symmetric memory cannot be set up on this box
    mailbox, exchange_how = None, "none"
    if world > 1:
        ok = torch.zeros(1, device=dev)
        why = ""
        if os.environ.get("SLCL_BENCH_EXCHANGE", "peer") == "peer":
            try:
                from slcl.peer import PeerMailbox
                mailbox = PeerMailbox(dev)
                ok.fill_(1.0)
            except Exception as exc:  # noqa: BLE001
                why = repr(exc)[:160]
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)          # all ranks or none
        if float(ok) < 1.0:
            mailbox = None
        exchange_how = ("split-phase exchange over NVLink peer memory: the forward's finaliser kernel stores this rank's 8-byte "
                        "{epoch|fp32} words into every peer's mailbox, the backward kernel receives them (block 0) -- no launch "
                        "between forward and backward, latency hidden behind the backward's launch") if mailbox is not None \
            else f"NCCL all-reduce of 8 bytes + rescale kernel ({why})"

    def step(record: bool):
        e0, e1, e2, e3 = (ev(), ev(), ev(), ev()) if record else (None,) * 4
        if record:
            e0.record()
        # N > 1 with mailboxes: split-phase exchange -- the forward's finaliser sends this rank's {weight sum, loss sum},
        # the backward kernel receives (block 0) while its other blocks already stream: no launch, no exposed latency
        scal = plan.forward(mailbox, split_phase=True)
        if record:
            e1.record()
        if mailbox is None and world > 1:
            dist.all_reduce(scal[2:4], op=dist.ReduceOp.SUM)
            plan.rescale()
        if record:
            e2.record()
        dfeat = plan.backward(mailbox)
        if record:
            e3.record()
            marks.append((e0, e1, e2, e3))
        return scal, dfeat

    exchange_check = None
    if mailbox is not None:
        # before anything is timed: the peer exchange must give what the NCCL all-reduce gives, on every rank -- else NCCL
        scal_p, d_p = step(False)
        loss_p, d_p = float(scal_p[0]), d_p.clone()
        scal_n = plan.forward()
        dist.all_reduce(scal_n[2:4], op=dist.ReduceOp.SUM)
        plan.rescale()
        d_n = plan.backward()
        torch.cuda.synchronize(dev)
        rel = abs(float(scal_n[0]) - loss_p) / max(abs(float(scal_n[0])), 1e-30)
        gdiff = float((d_p - d_n).abs().max()) / max(float(d_n.abs().max()), 1e-30)
        exchange_check = {"loss_rel_diff_vs_nccl": rel, "grad_max_abs_diff_over_max_abs": gdiff, "timeouts": mailbox.timeouts()}
        good = torch.tensor([1.0 if (rel < 1e-6 and gdiff < 1e-6 and exchange_check["timeouts"] == 0) else 0.0], device=dev)
        dist.all_reduce(good, op=dist.ReduceOp.MIN)
        del d_p, d_n
        if float(good) < 1.0:
            print(f"[bench] rank {rank}: peer exchange disagrees with NCCL ({exchange_check}); using NCCL", file=sys.stderr)
            mailbox = None
            exchange_how = f"NCCL all-reduce of 8 bytes + rescale kernel (peer exchange failed its check: {exchange_check})"

    sharded_check = None
    if world > 1:
        sharded_check = sharded_vs_global_check(dev, world, rank, mailbox)
        if not sharded_check["ok_on_every_rank"]:
            print(f"[bench] rank {rank}: SHARDED RESULT DIFFERS FROM THE GLOBAL ONE: {sharded_check}", file=sys.stderr)

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    for _ in range(max(args.warmup, 3)):
        step(False)
    barrier()
    start, end = ev(), ev()
    t_wall0 = time.perf_counter()
    start.record()
    for _ in range(args.steps):
        scal, dfeat = step(True)
    end.record()
    barrier()
    t_wall1 = time.perf_counter()
    elapsed_ms = start.elapsed_time(end)
    if world > 1:
        t = torch.tensor([elapsed_ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        elapsed_ms = float(t.item())
    ms_per_step = elapsed_ms / args.steps
    value = world * n_px * args.steps / (elapsed_ms * 1e-3)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, dfeat, loss=scal[:1], scal=scal)   # the last timed step's, before e2e frees the plan
    fwd_ms = statistics.mean(m[0].elapsed_time(m[1]) for m in marks)
    xch_ms = statistics.mean(m[1].elapsed_time(m[2]) for m in marks)
    bwd_ms = statistics.mean(m[2].elapsed_time(m[3]) for m in marks)
    loss_value = float(scal[0])
    launches_per_step = 4 + (1 if (world > 1 and mailbox is None) else 0)

    # ---- end to end through the public API with HOST buffers --------------------------------
    e2e = None
    if not args.no_e2e:
        mp = MPCL(dev, num_class=K, temperature=CFG["temperature"], m=CFG["margin"],
                  base_temperature=CFG["base_temperature"])
        grad_h = torch.empty_like(feats_h, pin_memory=True)
        loss_h = torch.empty((), dtype=torch.float32, pin_memory=True)
        group = True if world > 1 else None
        del dfeat, plan

        from slcl.host import mpcl_loss_and_grad_host

        def e2e_step():
            # public host-buffer API: chunked H2D -> fwd -> bwd -> D2H pipeline over 3 streams
            loss, _ = mpcl_loss_and_grad_host(feats_h, labels_h, centres, mp, pixel_sel_loc_h=sel_h, grad_out_h=grad_h,
                                              device=dev, chunk_images=E2E_CHUNK, group=group)
            loss_h.copy_(loss, non_blocking=True)

        n_e2e = max(1, min(args.steps, 20))
        for _ in range(2):
            e2e_step()
        barrier()
        s2, e2 = ev(), ev()
        s2.record()
        for _ in range(n_e2e):
            e2e_step()
        e2.record()
        barrier()
        ms = s2.elapsed_time(e2)
        if world > 1:
            t = torch.tensor([ms], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        # the same host-buffer step through the DROP-IN signature itself (no pipelining: copy in, mpcl_loss_calc(...)
        # .backward(), copy out) -- what a trainer that keeps its batch on the host would see without slcl.host
        def dropin_step():
            f = feats_h.to(dev, non_blocking=True).requires_grad_(True)
            lab_d = labels_h.to(dev, non_blocking=True)
            sel_d = sel_h.to(dev, non_blocking=True)
            loss = mpcl_loss_calc(f, lab_d, centres, mp, pixel_sel_loc=sel_d, tag="target", group=group)
            loss.backward()
            grad_h.copy_(f.grad, non_blocking=True)
            loss_h.copy_(loss.detach(), non_blocking=True)
        dropin_step()
        barrier()
        s3, e3 = ev(), ev()
        s3.record()
        for _ in range(5):
            dropin_step()
        e3.record()
        barrier()
        ms_dropin = s3.elapsed_time(e3) / 5
        if world > 1:
            t = torch.tensor([ms_dropin], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms_dropin = float(t.item())
        h2d = feats_h.numel() * 4 + labels_h.numel() * 8 + sel_h.numel() * 4
        d2h = grad_h.numel() * 4 + 4
        # what the box's IO fabric gives at this N: plain pinned cudaMemcpyAsync of the same buffers, all ranks at once --
        # H2D alone, D2H alone, both directions together (the e2e step needs both)
        dbuf = torch.empty_like(feats_h, device=dev)
        s_in, s_out = torch.cuda.Stream(dev), torch.cuda.Stream(dev)

        def copy_ceiling(do_in, do_out):
            barrier()
            c0, c1 = ev(), ev()
            c0.record()
            s_in.wait_event(c0); s_out.wait_event(c0)
            for _ in range(3):
                if do_in:
                    with torch.cuda.stream(s_in):
                        dbuf.copy_(feats_h, non_blocking=True)
                if do_out:
                    with torch.cuda.stream(s_out):
                        grad_h.copy_(dbuf, non_blocking=True)
            torch.cuda.current_stream(dev).wait_stream(s_in); torch.cuda.current_stream(dev).wait_stream(s_out)
            c1.record()
            barrier()
            t_ms = c0.elapsed_time(c1)
            if world > 1:
                tt = torch.tensor([t_ms], device=dev, dtype=torch.float64)
                dist.all_reduce(tt, op=dist.ReduceOp.MAX)
                t_ms = float(tt.item())
            return 3 * feats_h.numel() * 4 / (t_ms * 1e-3) / 1e9
        pcie = {"h2d_alone_GBps_per_gpu": copy_ceiling(True, False), "d2h_alone_GBps_per_gpu": copy_ceiling(False, True),
                "duplex_GBps_per_gpu_each_way": copy_ceiling(True, True)}
        del dbuf
        e2e = {"value": world * n_px * n_e2e / (ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": h2d,
               "d2h_bytes_per_step": d2h, "steps": n_e2e, "ms_per_step": ms / n_e2e,
               "api": f"slcl.host.mpcl_loss_and_grad_host(pinned feats/labels/sel -> loss, pinned dF): {E2E_CHUNK}-image chunks, "
                      "H2D / kernels / D2H overlapped on 3 streams",
               "loss": float(loss_h),
               "drop_in_signature": {"value": world * n_px / (ms_dropin * 1e-3), "ms_per_step": ms_dropin,
                                     "api": "feats.to(device) -> slcl.loss.mpcl_loss_calc(...).backward() -> grad.cpu(), unpipelined "
                                            "(H2D, kernels and D2H one after the other)"},
               "achieved_h2d_GBps_per_gpu": h2d * n_e2e / (ms * 1e-3) / 1e9, "achieved_d2h_GBps_per_gpu": d2h * n_e2e / (ms * 1e-3) / 1e9,
               "memcpy_ceiling_same_n": pcie, "cpu_affinity": affinity,
               "bound": "host<->device copies: the step moves %.2f GB in and %.2f GB out per GPU; compare achieved_*_GBps with "
                        "memcpy_ceiling_same_n.duplex (plain pinned cudaMemcpyAsync, all ranks at once) -- when they agree the "
                        "number is set by the box's PCIe / host-memory fabric, not by the kernels" % (h2d / 1e9, d2h / 1e9)}
        del grad_h
    sampler.stop()

    # configs[3]/[4]: the MCCL loss section of one adaptation step at the cfg5 geometry, through the Python API inside
    # autograd, with the centroid all-reduce over NCCL when N > 1 (every rank runs it; rank 0 reports the max)
    mccl = None
    cfg4 = None
    if not args.no_extras:
        mccl = mccl_loss_section(dev, world, mailbox)
        cfg4 = cfg4_strong_scaling(dev, world, rank, mailbox)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peak, peak_src = hbm_peak()
    bwd_bytes = 8 * C * n_px                     # read F + write dF (SURVEY.md 8(d)); the 4(K+1) B/px stash is overhead
    fwd_bytes = (4 * C + 12) * n_px              # read F + labels + sel
    step_bytes = (12 * C + 24) * n_px
    bwd_gbs = bwd_bytes / (bwd_ms * 1e-3) / 1e9
    roofline = {
        "bound": "hbm", "kernel": "proto_bwd_kernel<5,4>", "achieved": bwd_gbs, "peak": peak, "unit": "GB/s",
        "frac": bwd_gbs / peak, "traffic": ncu_traffic("proto_bwd_kernel"), "peak_source": peak_src,
        "algorithmic_bytes_per_launch": bwd_bytes, "avg_launch_ms": bwd_ms,
        "forward": {"kernel": "proto_fwd_kernel<5,4> (+prep, finalise)", "achieved": fwd_bytes / (fwd_ms * 1e-3) / 1e9,
                    "frac": fwd_bytes / (fwd_ms * 1e-3) / 1e9 / peak, "algorithmic_bytes_per_launch": fwd_bytes,
                    "avg_ms": fwd_ms, "traffic": ncu_traffic("proto_fwd_kernel")},
        "step": {"achieved": step_bytes / (ms_per_step * 1e-3) / 1e9, "frac": step_bytes / (ms_per_step * 1e-3) / 1e9 / peak,
                 "algorithmic_bytes": step_bytes, "exchange_ms": xch_ms},
    }

    out = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": base_config(world), "exchange": exchange_how,
        "roofline": roofline, "e2e": e2e, "gpu_launches": launches_per_step * args.steps,
        "clocks": sampler.summary(t_wall0, t_wall1), "loss": loss_value,
    }
    if exchange_check is not None:
        out["exchange_check"] = exchange_check
    if sharded_check is not None:
        out["sharded_vs_global_check"] = sharded_check
    if cfg4 is not None:
        cfg4["frac_of_hbm_peak"] = cfg4["achieved_GBps_aggregate"] / (world * peak)
        out["cfg4_strong_scaling"] = cfg4
    if mccl is not None:
        mccl["frac_of_hbm_peak"] = mccl["achieved_GBps_per_gpu"] / peak
        if mccl.get("fused_centroid_losses"):
            mccl["fused_centroid_losses"]["frac_of_hbm_peak"] = mccl["fused_centroid_losses"]["achieved_GBps_per_gpu"] / peak
        out["mccl_loss_section"] = mccl
    if not args.no_extras and world == 1:
        out["kernels"] = extra_kernels(dev, feats, labels, centres, peak)
    if not args.no_cpu and world == 1:
        try:
            ms_eager, loss_eager, grad_eager = time_torch_eager_gpu(dev, feats, labels, sel, centres)
            gmax = float(grad_eager.abs().max())
            xq = feats.detach().clone().requires_grad_(True)
            mpq = MPCL(dev, num_class=K, temperature=CFG["temperature"], m=CFG["margin"], base_temperature=CFG["base_temperature"])
            mpcl_loss_calc(xq, labels, centres, mpq, pixel_sel_loc=sel, tag="target").backward()
            dfeat = xq.grad
            out["torch_eager_gpu"] = {
                "value": n_px / (ms_eager * 1e-3), "unit": UNIT, "ms_per_step": ms_eager, "kind": "port",
                "what": "oracle port of mpcl_loss_calc+MPCL.forward fwd+bwd as eager PyTorch fp32 on the same B200, same resident "
                        "cfg2 batch, min of 5 after 2 warm-ups (the reference's GPU path; reported comparator, not the product)",
                "loss": loss_eager, "loss_rel_diff_vs_cuda_path": abs(loss_eager - loss_value) / max(abs(loss_eager), 1e-30),
                "grad_max_abs_diff_over_max_abs": float((grad_eager - dfeat).abs().max()) / max(gmax, 1e-30)}
            del grad_eager, dfeat, xq
            torch.cuda.empty_cache()
        except Exception as exc:  # noqa: BLE001 - a comparator must never take the bench line down
            out["torch_eager_gpu"] = {"unavailable": repr(exc)[:200]}
        n_img = args.cpu_sample_images
        pixels, times, cores, _ = time_cpu(n_img, 1, 3)
        out["cpu_baseline"] = {
            "value": pixels / min(times), "unit": UNIT, "cores": cores, "kind": "port",
            "sample": f"{n_img} of the 32 cfg2 images per step ({pixels} px), oracle port of the reference call sequence, "
                      f"fwd+bwd, min of 3 after 1 warm-up, torch CPU fp32 with {cores} threads"}
        del times
    else:
        out["cpu_baseline"] = None
    print(json.dumps(out), flush=True)
    if world > 1:
        dist.destroy_process_group()
    if sharded_check is not None and not sharded_check["ok_on_every_rank"]:
        raise SystemExit("bench.py: sharded multi-GPU result differs from the single-GPU global result (see the JSON line)")


def sharded_vs_global_check(dev, world, rank, mailbox):
    """SURVEY 8(e) on the hardware that has N GPUs: before anything is timed, every rank ALSO evaluates the global batch
    (small shape, identical bits on every rank) on its own GPU and compares its sharded result -- through the Python API,
    with the NCCL route (group=True) and the peer-mailbox route (group=PeerMailbox) -- against it: prototype loss (source,
    target, fused target step) loss rtol 1e-6 / gradients rtol 1e-5; update_class_center_iter and cal_centroid(soft, P=2)
    centres rtol 1e-5 with class counts torch.equal; the host-buffer pipeline's loss.  A mismatch fails the run."""
    import torch.distributed as dist
    from slcl.loss import MPCL, mpcl_loss_calc, mpcl_target_step
    from slcl.utils_ import cal_centroid, update_class_center_iter
    from slcl.host import mpcl_loss_and_grad_host
    op = torch.ops.slcl
    b, c, h, w, k, parts = 2 * world, 32, 48, 40, 4, 2
    g = torch.Generator().manual_seed(2024)
    feat = torch.randn(b, c, h, w, generator=g).to(dev)
    lab = torch.randint(0, k, (b, h, w), generator=g)
    lab[lab == 3] = 1                     # an empty class: the empty-class rule must act on GLOBAL counts
    lab = lab.to(dev)
    sel = (torch.rand(b * h * w, generator=g) > 0.4).float().to(dev)
    probs = torch.softmax(3 * torch.randn(b, k, h, w, generator=g), 1).to(dev)
    part = (torch.randperm(b * h * w, generator=g) % parts).to(torch.int32).to(dev)
    cen = torch.randn(k, c, generator=g).to(dev)
    gcen = torch.randn(parts * k, c, generator=g).to(dev)
    mp = MPCL(dev, num_class=k, temperature=0.1, m=0.4, base_temperature=1.0)
    lo, hi = 2 * rank, 2 * rank + 2
    px = lambda t: t.reshape(b, -1)[lo:hi].reshape(-1)

    def rel(a, ref):
        a, ref = a.detach().double(), ref.detach().double()
        return float((a - ref).abs().max() / ref.abs().max().clamp_min(1e-30))

    def proto(f, labels, selv, group):
        l1 = mpcl_loss_calc(f, labels, cen, mp, tag="source", group=group)
        l2 = mpcl_loss_calc(f, labels.reshape(-1), cen, mp, pixel_sel_loc=selv, tag="target", group=group)
        l3, _, _ = mpcl_target_step(f, cen, mp, 0.05, group=group)
        return l1, l2, l3

    def centres(f, labels, p, pid, group):
        new = update_class_center_iter(f, labels, cen, m=0.9, num_class=k, group=group)
        soft, _, _ = cal_centroid(f, p, pseudo_label=True, weighted_ave=True, partition=parts, n_class=k, part_id=pid,
                                  group=group)
        return new, torch.cat(soft)

    # global references on this rank's GPU
    fg, pg = feat.clone().requires_grad_(True), probs.clone().requires_grad_(True)
    want_l = proto(fg, lab, sel, None)
    want_new, want_soft = centres(fg, lab, pg, part, None)
    (want_l[0] + 2 * want_l[1] + 3 * want_l[2] + (want_soft * gcen).sum()).backward()
    counts_g = op.class_sums(feat, lab.reshape(-1), None, False, 0.0, None, 1, k)[:, -1]

    out, worst = {}, 0.0
    routes = [("nccl", True)] + ([("peer", mailbox)] if mailbox is not None else [])
    for name, group in routes:
        f, p = feat[lo:hi].clone().requires_grad_(True), probs[lo:hi].clone().requires_grad_(True)
        got_l = proto(f, lab[lo:hi], px(sel), group)
        got_new, got_soft = centres(f, lab[lo:hi], p, px(part), group)
        (got_l[0] + 2 * got_l[1] + 3 * got_l[2] + (got_soft * gcen).sum()).backward()
        if name == "peer":
            _, sums = op.class_centres_update(feat[lo:hi].contiguous(), lab[lo:hi].reshape(-1), cen, 0.9, *mailbox.args())
        else:
            sums = op.class_sums(feat[lo:hi].contiguous(), lab[lo:hi].reshape(-1), None, False, 0.0, None, 1, k)
            dist.all_reduce(sums)
        r = {"loss_rel": max(rel(a, b_) for a, b_ in zip(got_l, want_l)),
             "dfeat_rel": rel(f.grad, fg.grad[lo:hi]), "dprobs_rel": rel(p.grad, pg.grad[lo:hi]),
             "ema_centres_rel": rel(got_new, want_new), "soft_centroids_rel": rel(got_soft, want_soft),
             "class_counts_equal": bool(torch.equal(sums[:, -1], counts_g))}
        r["ok"] = (r["loss_rel"] < 1e-6 and r["dfeat_rel"] < 1e-5 and r["dprobs_rel"] < 1e-5 and r["ema_centres_rel"] < 1e-5
                   and r["soft_centroids_rel"] < 1e-5 and r["class_counts_equal"])
        out[name] = r
    # host-buffer pipeline (slcl.host): the returned loss must be the GLOBAL loss, the gradient the global gradient's shard
    grad_h = torch.empty((2, c, h, w), pin_memory=True)
    loss_h, _ = mpcl_loss_and_grad_host(feat[lo:hi].cpu().pin_memory(), lab[lo:hi].cpu(), cen, mp,
                                        pixel_sel_loc_h=px(sel).cpu(), grad_out_h=grad_h, device=dev, chunk_images=1, group=True)
    torch.cuda.synchronize(dev)
    fh = feat.clone().requires_grad_(True)
    want_h = mpcl_loss_calc(fh, lab.reshape(-1), cen, mp, pixel_sel_loc=sel, tag="target")
    want_h.backward()
    r = {"loss_rel": rel(loss_h, want_h), "dfeat_rel": rel(grad_h.to(dev), fh.grad[lo:hi])}
    r["ok"] = r["loss_rel"] < 1e-6 and r["dfeat_rel"] < 1e-5
    out["host_pipeline"] = r
    if mailbox is not None:
        out["peer_timeouts"] = mailbox.timeouts()
    ok = all(v["ok"] for v in out.values() if isinstance(v, dict)) and out.get("peer_timeouts", 0) == 0
    flag = torch.tensor([1.0 if ok else 0.0], device=dev)
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    out["ok_on_every_rank"] = bool(float(flag) == 1.0)
    out["shape"] = f"global batch {b} x {c} x {h} x {w}, K={k}, P={parts}; 2 images per rank; rank-0 numbers"
    return out


def cfg4_strong_scaling(dev, world, rank, mailbox=None):
    """configs[3] (SURVEY.md 8(e)): the MS-CMRSeg bSSFP->LGE shape, a FIXED global batch of 128 images (C = 32, 224 x 224,
    K = 4) sharded over the ranks (128 / N images per GPU: STRONG scaling), prototype loss forward + backward with the
    8-byte {weight sum, weighted row-loss sum} all-reduce + rescale between them, and the EMA class-centre update
    (class sums all-reduced as [K, C+1] fp64) on the same shard.  Aggregate pixels/s = 6 422 528 px / max-over-ranks time."""
    import torch.distributed as dist
    from slcl.plan import ProtoPlan
    from slcl.utils_ import update_class_center_iter
    from slcl.distributed import shard_range
    B, c, h, k = 128, 32, 224, 4
    lo, hi = shard_range(B, rank, world)
    b = hi - lo
    gen = torch.Generator(device=dev).manual_seed(99 + rank)
    f = torch.randn(b, c, h, h, device=dev, generator=gen)
    lab = torch.randint(0, k, (b, h, h), device=dev, generator=gen)
    sel = (torch.rand(b * h * h, device=dev, generator=gen) > 0.3).float()
    cen = torch.randn(k, c, device=dev, generator=gen)
    if world > 1:
        dist.broadcast(cen, 0)
    plan = ProtoPlan(f, lab.reshape(-1), sel, cen, k, CFG["temperature"], CFG["base_temperature"], CFG["margin"])
    group = (mailbox if mailbox is not None else True) if world > 1 else None

    def proto_step():
        scal = plan.forward(mailbox, split_phase=True)
        if mailbox is None and world > 1:
            dist.all_reduce(scal[2:4], op=dist.ReduceOp.SUM)
            plan.rescale()
        plan.backward(mailbox)
        return scal

    def ema_step():
        return update_class_center_iter(f, lab, cen, m=0.9, num_class=k, group=group)

    def timed(fn, iters=20):
        for _ in range(3):
            fn()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        for _ in range(iters):
            out = fn()
        e.record()
        torch.cuda.synchronize(dev)
        t = torch.tensor([s.elapsed_time(e) / iters], device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t), out

    ms_proto, scal = timed(proto_step)
    ms_ema, new_cen = timed(ema_step)
    # the same two steps as CUDA-graph replays (no NCCL on either path when the peer mailboxes are in use): device time
    # without the Python dispatch of the eager API
    ms_proto_graph = ms_ema_graph = None
    if world == 1 or mailbox is not None:
        try:
            side = torch.cuda.Stream(dev)
            side.wait_stream(torch.cuda.current_stream(dev))
            with torch.cuda.stream(side):
                proto_step(); ema_step()
            torch.cuda.current_stream(dev).wait_stream(side)
            torch.cuda.synchronize(dev)
            if world > 1:
                dist.barrier()
            g_proto, g_ema = torch.cuda.CUDAGraph(), torch.cuda.CUDAGraph()
            with torch.cuda.graph(g_proto):
                proto_step()
            with torch.cuda.graph(g_ema):
                keep_ema = ema_step()          # noqa: F841
            ms_proto_graph, _ = timed(g_proto.replay)
            ms_ema_graph, _ = timed(g_ema.replay)
        except Exception as exc:  # noqa: BLE001
            print(f"[bench] cfg4: graph capture unavailable ({exc!r})", file=sys.stderr)
    n_global = B * h * h
    bytes_proto = (12 * c + 24) * n_global
    return {"workload": f"cfg4: global batch 128 x 32 x 224 x 224, K=4, {b} images on this GPU ({world} GPUs, strong scaling): "
                        "prototype loss fwd+bwd (raw C-ABI plan) and the EMA class-centre update (Python API)",
            "scaling": "strong", "n_gpus": world, "global_pixels": n_global,
            "proto_fwd_bwd_ms": ms_proto, "proto_pixels_per_s": n_global / (ms_proto * 1e-3),
            "algorithmic_bytes_global": bytes_proto, "achieved_GBps_aggregate": bytes_proto / (ms_proto * 1e-3) / 1e9,
            "proto_fwd_bwd_graph_ms": ms_proto_graph, "ema_class_centres_graph_ms": ms_ema_graph,
            "ema_class_centres_ms": ms_ema, "ema_pixels_per_s": n_global / (ms_ema * 1e-3),
            "ema_achieved_GBps_aggregate": (4 * c + 8) * n_global / (ms_ema * 1e-3) / 1e9, "loss": float(scal[0]),
            "exchange": "none" if world == 1 else
                        ("loss pair: " + ("fused peer-memory exchange + rescale kernel" if mailbox is not None else "NCCL all-reduce")
                         + "; EMA: " + ("class sums exchanged inside the reduce kernel over NVLink peer mailboxes"
                                        if mailbox is not None else "NCCL all-reduce of the [K, C+1] fp64 class sums"))}


def mccl_loss_section(dev, world, mailbox=None):
    import torch.distributed as dist
    """Trainer_MCCL.py:275-332 between "the decoder produced feature maps" and "the loss has gradients": source centroids
    (hard labels), target and augmented-target centroids (soft labels x certainty, 2 reversed-Monte-Carlo partitions),
    ContrastiveLoss per partition + centroid-norm regulariser, backward to the three feature maps and both soft-label
    maps.  cfg5 geometry per GPU: 64 images of 224x224, C = 32, K = 4 (weak scaling); the per-class sums are all-reduced
    with NCCL when N > 1.  Bytes: source 8C+8, each target 12C+12K+8 per pixel (SURVEY.md 8(d))."""
    from slcl.loss import ContrastiveLoss, cnr_loss
    from slcl.utils_ import cal_centroid
    b, c, h, k, parts = 64, 32, 224, 4, 2
    n_px = b * h * h
    gen = torch.Generator(device=dev).manual_seed(4321 + int(os.environ.get("RANK", "0")))
    ft = [torch.randn(b, c, h, h, device=dev, generator=gen).requires_grad_(True) for _ in range(3)]
    lab_s = torch.randint(0, k, (b, h, h), device=dev, generator=gen)
    pr = [torch.softmax(3 * torch.randn(b, k, h, h, device=dev, generator=gen), 1).requires_grad_(True) for _ in range(2)]
    part = [(torch.randperm(n_px, device=dev, generator=gen) % parts).to(torch.int32) for _ in range(2)]
    crit = ContrastiveLoss()
    # N > 1: the [sets*K, C+1] fp64 class sums are exchanged inside the reduce kernels over the NVLink peer mailboxes (no
    # collective launch, so the section is graph-capturable at every N); NCCL all-reduce when there is no mailbox
    group = (mailbox if mailbox is not None else True) if world > 1 else None

    def make_step(ft, pr):
        def step():
            cs, _, _ = cal_centroid(ft[0], lab_s, n_class=k, group=group)
            loss = 0
            for i in range(2):
                ct, _, _ = cal_centroid(ft[1 + i], pr[i], pseudo_label=True, weighted_ave=True, partition=parts, n_class=k,
                                        part_id=part[i], group=group)
                for c_p in ct:
                    loss = loss + crit(cs, c_p)
                loss = loss + 4e-5 * cnr_loss(cs, ct)
            loss.backward()
            for t in ft + pr:
                t.grad = None
            return loss.detach()
        return step

    step = make_step(ft, pr)

    def make_fused_step(ft, pr):
        """the same section with the centroid<->centroid terms as ONE op per target map (slcl.loss.mccl_centroid_losses)"""
        from slcl.loss import mccl_centroid_losses

        def step():
            cs, _, _ = cal_centroid(ft[0], lab_s, n_class=k, group=group)
            loss = 0
            for i in range(2):
                ct, _, _ = cal_centroid(ft[1 + i], pr[i], pseudo_label=True, weighted_ave=True, partition=parts, n_class=k,
                                        part_id=part[i], group=group)
                total, _ = mccl_centroid_losses(cs, ct, None, inter_w=float(parts), intra_w=0.0, cnr_w=4e-5)
                loss = loss + total
            loss.backward()
            for t in ft + pr:
                t.grad = None
            return loss.detach()
        return step

    def timed(fn, iters=10):
        for _ in range(3):
            fn()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        for _ in range(iters):
            out = fn()
        e.record()
        torch.cuda.synchronize(dev)
        t = torch.tensor([s.elapsed_time(e) / iters], device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t), out

    ms_eager, loss = timed(step)          # what a plain eager trainer sees: ~30 custom-op calls, host-launch-bound
    ms, how = ms_eager, "eager"
    if world == 1 or mailbox is not None:
        # the same step captured once in a CUDA graph (forward + autograd backward): the device time of the section
        try:
            # fresh leaves: their AccumulateGrad nodes must be born on the capture side stream, not the default one
            gstep = make_step([t.detach().requires_grad_(True) for t in ft], [t.detach().requires_grad_(True) for t in pr])
            side = torch.cuda.Stream(dev)
            side.wait_stream(torch.cuda.current_stream(dev))
            with torch.cuda.stream(side):
                gstep()
            torch.cuda.current_stream(dev).wait_stream(side)
            torch.cuda.synchronize(dev)
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                static_loss = gstep()
            ms, _ = timed(graph.replay)
            loss, how = static_loss, "one CUDA graph (forward + autograd backward captured)"
        except Exception as exc:          # capture is an optimisation of the measurement, not of the product
            print(f"[bench] MCCL section: graph capture unavailable ({exc!r}); reporting the eager time", file=sys.stderr)
    fused = None
    if world == 1 or mailbox is not None:
        try:
            fstep = make_fused_step([t.detach().requires_grad_(True) for t in ft], [t.detach().requires_grad_(True) for t in pr])
            side = torch.cuda.Stream(dev)
            side.wait_stream(torch.cuda.current_stream(dev))
            with torch.cuda.stream(side):
                fstep()
            torch.cuda.current_stream(dev).wait_stream(side)
            torch.cuda.synchronize(dev)
            fgraph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(fgraph):
                f_loss = fstep()
            ms_f, _ = timed(fgraph.replay)
            fused = {"ms_per_step": ms_f, "loss": float(f_loss),
                     "what": "same section, centroid<->centroid terms through slcl.loss.mccl_centroid_losses (one op per target "
                             "map: 2 launches forward, 3 scalings backward), one CUDA graph"}
        except Exception as exc:  # noqa: BLE001
            print(f"[bench] MCCL section (fused losses): unavailable ({exc!r})", file=sys.stderr)
    bytes_ = ((8 * c + 8) + 2 * (12 * c + 12 * k + 8)) * n_px
    if fused is not None:
        fused["achieved_GBps_per_gpu"] = bytes_ / (fused["ms_per_step"] * 1e-3) / 1e9
    return {"fused_centroid_losses": fused, "workload": "cfg5 geometry: MCCL loss section (3 x cal_centroid + 4 x ContrastiveLoss + CNR, fwd+bwd) through the "
                        "Python API inside autograd, per GPU 64 x 32 x 224 x 224, K=4, P=2",
            "ms_per_step": ms, "timed_as": how, "ms_per_step_eager": ms_eager,
            "pixels_per_s": world * 3 * n_px / (ms * 1e-3), "algorithmic_bytes_per_gpu": bytes_,
            "achieved_GBps_per_gpu": bytes_ / (ms * 1e-3) / 1e9, "n_gpus": world, "loss": float(loss),
            "exchange": "none" if world == 1 else
                        ("[sets*K, C+1] fp64 class sums exchanged inside the reduce kernel of each cal_centroid over NVLink peer "
                         "mailboxes (no collective launch)" if mailbox is not None else
                         "all-reduce of [sets*K, C+1] fp64 class sums per cal_centroid (NCCL)")}


def extra_kernels(dev, feats, labels, centres, peak):
    """Device-time and roofline fraction of the other kernels of the path on the same map
    (not part of `value`): pseudo labels, EMA class centres, soft centroid fwd/bwd."""
    op = torch.ops.slcl
    B, C, H, W = feats.shape
    K = centres.shape[0]
    n_px = B * H * W
    gen = torch.Generator(device=dev).manual_seed(7)
    probs = torch.softmax(3 * torch.randn(B, K, H, W, device=dev, generator=gen), 1)
    part = (torch.randperm(n_px, device=dev, generator=gen) % 2).to(torch.int32)
    gcen = torch.randn(2 * K, C, device=dev, generator=gen)

    def timed(fn, iters=10):
        for _ in range(2):
            fn()
        torch.cuda.synchronize(dev)
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        for _ in range(iters):
            fn()
        e.record()
        torch.cuda.synchronize(dev)
        return s.elapsed_time(e) / iters

    res = {}

    def add(name, ms, bytes_):
        gbs = bytes_ / (ms * 1e-3) / 1e9
        res[name] = {"ms": ms, "algorithmic_bytes": bytes_, "achieved_GBps": gbs, "frac_of_hbm_peak": gbs / peak}

    add("pseudo_label (generate_pseudo_label)", timed(lambda: op.pseudo_label(feats, centres, 0.25)), (4 * C + 12) * n_px)
    # f-1: generate_pseudo_label + target MPCL forward fused into one read of the map (vs the two separate passes)
    add("fused target step: pseudo labels + target prototype-loss forward, one read of F_t",
        timed(lambda: op.proto_fwd_target(feats, centres, 0.25, K, CFG["temperature"], CFG["base_temperature"], CFG["margin"],
                                          False)), (4 * C + 12) * n_px)
    # f-1 completed: the same fused target step ALSO producing the hard target centroids (class sums under the pseudo labels
    # it has just generated) from the same single read of F_t -- vs fused target step + a second pass for the centroids
    add("fused target step + hard target centroids, ONE read of F_t (slcl_target_step)",
        timed(lambda: op.target_step(feats, centres, 0.25, False, K, CFG["temperature"], CFG["base_temperature"], CFG["margin"],
                                     False, None, 0.9)), (4 * C + 12) * n_px)

    def target_two_pass():
        o = op.proto_fwd_target(feats, centres, 0.25, K, CFG["temperature"], CFG["base_temperature"], CFG["margin"], False)
        op.centroids_fwd(feats, o[3], None, False, 0.0, None, 1, K, None, 0.9)
    add("the same results from two passes (proto_fwd_target, then centroids_fwd over the pseudo labels): bytes = 2 reads of F_t",
        timed(target_two_pass), (8 * C + 20) * n_px)
    add("class_sums hard + ema_finalize (update_class_center_iter)",
        timed(lambda: op.ema_finalize(op.class_sums(feats, labels, None, False, 0.0, None, 1, K), centres, 0.9)),
        (4 * C + 8) * n_px)
    sums = op.class_sums(feats, None, probs, True, 0.0, part, 2, K)
    add("class_sums soft P=2 (cal_centroid fwd)", timed(lambda: op.class_sums(feats, None, probs, True, 0.0, part, 2, K)),
        (4 * C + 4 * K + 4) * n_px)
    add("centroid_bwd soft P=2 (cal_centroid bwd: dF + dP)",
        timed(lambda: op.centroid_bwd(feats, None, probs, True, 0.0, part, 2, K, gcen, sums, 1.0, True)),
        (8 * C + 8 * K + 4) * n_px)
    # north_star (1): the sampler -- stable per-class compaction of the label map (bit-exact with torch.nonzero) and the
    # gather of the sampled rows (L2-normalised, bf16, padded to 64 columns) for the cfg3 problem.  These are short
    # kernels: timed as CUDA-graph replays so that the host-side launch cost of the Python op is not what is measured.
    def timed_graph(fn, iters=20):
        side = torch.cuda.Stream(dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):
            fn()
        torch.cuda.current_stream(dev).wait_stream(side)
        torch.cuda.synchronize(dev)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            keep = fn()                                   # noqa: F841  (outputs stay alive with the graph)
        return timed(g.replay, iters=iters)

    add("sampler: compact_by_class over the cfg2 label map (int64 in, int64 indices out)",
        timed_graph(lambda: op.compact_by_class(labels, K)), (8 + 8) * n_px)
    fmap3 = torch.randn(16, 256, 64, 64, device=dev, generator=gen)
    rows3 = torch.randperm(16 * 64 * 64, device=dev, generator=gen)[:16384 + 4096]
    add("sampler: gather_unit_rows, 20480 rows x 256 channels from a [16,256,64,64] map -> unit bf16 rows",
        timed_graph(lambda: op.gather_unit_rows(fmap3, rows3, True, True, False)), 20480 * 256 * 32)   # 32 B sector per element
    del fmap3, rows3
    # cfg5 geometry (DRUNet decoder map, C=32, K=4, P=2; 64 images of 224x224 per GPU)
    del probs, part, gcen, sums
    b5, c5, h5, k5 = 64, 32, 224, 4
    n_px = b5 * h5 * h5
    f5 = torch.randn(b5, c5, h5, h5, device=dev, generator=gen)
    p5 = torch.softmax(3 * torch.randn(b5, k5, h5, h5, device=dev, generator=gen), 1)
    part5 = (torch.randperm(n_px, device=dev, generator=gen) % 2).to(torch.int32)
    lab5 = torch.randint(0, k5, (n_px,), device=dev, generator=gen)
    g5 = torch.randn(2 * k5, c5, device=dev, generator=gen)
    s5 = op.class_sums(f5, None, p5, True, 0.0, part5, 2, k5)
    add("cfg5 shape: class_sums hard (EMA centres) C32 K4", timed(lambda: op.class_sums(f5, lab5, None, False, 0.0, None, 1, k5)),
        (4 * c5 + 8) * n_px)
    add("cfg5 shape: class_sums soft P=2 C32 K4 (cal_centroid fwd)",
        timed(lambda: op.class_sums(f5, None, p5, True, 0.0, part5, 2, k5)), (4 * c5 + 4 * k5 + 4) * n_px)
    add("cfg5 shape: centroid_bwd soft P=2 C32 K4 (dF + dP)",
        timed(lambda: op.centroid_bwd(f5, None, p5, True, 0.0, part5, 2, k5, g5, s5, 1.0, True)), (8 * c5 + 8 * k5 + 4) * n_px)
    # the trainer-default call: cal_centroid(..., partition=2) draws the reversed-Monte-Carlo partition itself -- one
    # torch.randperm(N) on the map's device (3.2 M elements) inside the timed call, forward only
    from slcl.utils_ import cal_centroid as _cal_centroid
    add("cfg5 shape: cal_centroid(soft, partition=2) through the Python API INCLUDING the rMC draw (forward)",
        timed(lambda: _cal_centroid(f5, p5, pseudo_label=True, weighted_ave=True, partition=2, n_class=k5)),
        (4 * c5 + 4 * k5 + 4) * n_px)
    # cfg4 geometry per GPU (MS-CMRSeg: 16 of the 128 images per GPU, C = 32, K = 4, 224 x 224): prototype loss fwd+bwd
    from slcl.plan import ProtoPlan
    f4 = f5[:16].contiguous()
    lab4 = torch.randint(0, k5, (16 * h5 * h5,), device=dev, generator=gen)
    sel4 = (torch.rand(16 * h5 * h5, device=dev, generator=gen) > 0.3).float()
    cen4 = torch.randn(k5, c5, device=dev, generator=gen)
    plan4 = ProtoPlan(f4, lab4, sel4, cen4, k5, CFG["temperature"], CFG["base_temperature"], CFG["margin"])

    def proto4():
        plan4.forward()
        plan4.backward()
    add("cfg4 shape per GPU: prototype loss fwd+bwd, 16 x 32 x 224 x 224, K4", timed(proto4, iters=20),
        (12 * c5 + 24) * 16 * h5 * h5)
    # f-1 source side at the same shape: update_class_center_iter + source loss forward + backward as ONE call
    # (slcl.loss.mpcl_source_step), replayed as a CUDA graph; three walks over a 98 MiB map that fits in L2 (zig-zag walk
    # order + evict_last forward: ncu counts 194 MB of DRAM reads for the step instead of 3.4 maps, profiles/README.md)
    try:
        from slcl.loss import MPCL as _MPCL, mpcl_source_step as _src_step
        f4g = f4.clone().requires_grad_(True)
        lab4m = lab4.view(16, h5, h5)
        mp4 = _MPCL(dev, num_class=k5, temperature=CFG["temperature"], m=0.4, base_temperature=CFG["base_temperature"])

        def src_step():
            _, l4 = _src_step(f4g, lab4m, cen4, mp4, m=0.9, num_class=k5)
            l4.backward()
            f4g.grad = None
        add("cfg4 shape per GPU: source step (EMA class centres + source loss fwd+bwd, one call), one CUDA graph",
            timed_graph(src_step, iters=30), (16 * c5 + 32) * 16 * h5 * h5)
        del f4g
    except Exception as exc:  # noqa: BLE001
        print(f"[bench] source step: unavailable ({exc!r})", file=sys.stderr)
    del f4, lab4, sel4, cen4, plan4
    res["cfg1: prototype loss fwd+bwd, source variant, B8 C128 33x33 K5 (configs[0], the reference's CPU-runnable case)"] = \
        cfg1_line(dev, timed)
    # cfg3: sampled pixel<->pixel loss, 4096 anchors x 16384 contrast rows, d = 256, bf16 tensor cores
    del f5, p5, part5, lab5, g5, s5
    res.update(p2p_kernels(dev, gen))
    return res


def cfg1_line(dev, timed):
    """BASELINE configs[0] at FULL size on both sides (no sampling): 8 x 128 x 33 x 33 features (the 2048->128 projection
    is outside the path), labels 8 x 256 x 256 downsampled inside mpcl_loss_calc (utils/loss.py:585-590), K = 5, m = 0.4.
    8 712 pixels: launch-latency-bound on the GPU.  HW = 1089 is odd -> the scalar (VEC = 1) kernels."""
    from slcl.loss import MPCL, mpcl_loss_calc
    from slcl.plan import ProtoPlan
    from oracle import slcl_oracle as O
    g = torch.Generator().manual_seed(CFG["seed"] + 11)
    f_h = torch.randn(8, 128, 33, 33, generator=g)
    lab_h = torch.randint(0, 5, (8, 256, 256), generator=g)
    cen_h = torch.randn(5, 128, generator=g)
    f1, lab1, cen1 = f_h.to(dev).requires_grad_(True), lab_h.to(dev), cen_h.to(dev)
    mp = MPCL(dev, num_class=5, temperature=CFG["temperature"], m=0.4, base_temperature=CFG["base_temperature"])

    def api_step():
        f1.grad = None
        loss = mpcl_loss_calc(f1, lab1, cen1, mp, tag="source")
        loss.backward()
        return loss
    ms_api = timed(api_step, iters=20)
    loss_gpu = float(api_step().detach())
    lab_ds = O.nearest_label_resize(lab_h, 33, 33).reshape(-1).long().to(dev)        # label resize outside the graph
    plan = ProtoPlan(f1.detach(), lab_ds, None, cen1, 5, CFG["temperature"], CFG["base_temperature"], 0.4)
    graph = plan.capture_graph()
    ms_graph = timed(graph.replay, iters=50)
    # CPU port on the same full config, all host threads
    spec = O.MarginSpec(num_class=5, temperature=CFG["temperature"], m=0.4, base_temperature=CFG["base_temperature"])
    fc = f_h.clone().requires_grad_(True)
    torch.set_num_threads(os.cpu_count() or 1)

    def cpu_step():
        fc.grad = None
        loss = O.mpcl_loss_calc(fc, lab_h, cen_h, spec, tag="source")
        loss.backward()
        return float(loss.detach())
    for _ in range(2):
        loss_cpu = cpu_step()
    cpu_times = []
    for _ in range(5):
        t0 = time.perf_counter()
        cpu_step()
        cpu_times.append(time.perf_counter() - t0)
    n_px = 8 * 33 * 33
    return {"ms_api_eager": ms_api, "ms_one_cuda_graph": ms_graph, "pixels_per_s_graph": n_px / (ms_graph * 1e-3),
            "pixels_per_s_api_eager": n_px / (ms_api * 1e-3), "cpu_port_ms": 1e3 * min(cpu_times),
            "cpu_port_pixels_per_s": n_px / min(cpu_times), "cpu_cores": os.cpu_count(),
            "loss_gpu": loss_gpu, "loss_cpu_port": loss_cpu, "loss_rel_diff": abs(loss_gpu - loss_cpu) / abs(loss_cpu),
            "bound": "launch latency (8 712 pixels, 4.5 MB): API = label resize + custom ops, graph = prep/forward/finalise/backward only"}


def p2p_kernels(dev, gen):
    from slcl import ops as slcl_ops
    from slcl.plan import P2PPlan
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
            tf_peak = float(json.load(fh)["bf16_tflops"])
    except Exception:
        tf_peak = 1590.0
    A, M, d, T = 4096, 16384, 256, 0.7
    b = torch.nn.functional.normalize(torch.randn(M, d, device=dev, generator=gen), dim=1).to(torch.bfloat16)
    lb = torch.randint(0, 5, (M,), device=dev, generator=gen, dtype=torch.int32)
    ib = torch.arange(M, device=dev, dtype=torch.int32)
    pick = torch.randperm(M, device=dev, generator=gen)[:A]
    a, la, ia = b[pick].contiguous(), lb[pick].contiguous(), ib[pick].contiguous()
    fg = (la != 0).float()
    shift, weight = torch.full((A,), 1.0 / T, device=dev), fg / fg.sum()
    meta_a, meta_b = slcl_ops.pad_meta(la, ia), slcl_ops.pad_meta(lb, ib)
    selfcol, selfrow = slcl_ops.self_maps(ia, ib)
    # headline: the analytic sweeps (class-index labels; forward keeps U, backward = one dB sweep)
    plan = P2PPlan(a, b, d, meta_a, meta_b, shift, weight, T, n_class=5, a_selfcol=selfcol, b_selfrow=selfrow)
    graph = plan.capture_graph()
    # general-label sweeps (per-element {label, id} tests; what unlabelled SupCon / ISCL use)
    gplan = P2PPlan(a, b, d, meta_a, meta_b, shift, weight, T)
    ggraph = gplan.capture_graph()
    # the same general sweeps the way slcl.p2p drives them for one-row-set problems: contrast rows sorted by label
    # (label-uniform column tiles take the fast path) and self maps instead of per-element id tests
    order = torch.argsort(lb.long(), stable=True)
    inv = torch.empty_like(order)
    inv[order] = torch.arange(M, device=dev)
    b_s, lb_s = b[order].contiguous(), lb[order].contiguous()
    a_order = torch.argsort(la.long(), stable=True)
    a_s, la_s, w_s = a[a_order].contiguous(), la[a_order].contiguous(), weight[a_order].contiguous()
    sc_s = inv[pick[a_order]].to(torch.int32).contiguous()
    sr_s = torch.full((M,), -1, dtype=torch.int32, device=dev)
    sr_s[sc_s.long()] = torch.arange(A, device=dev, dtype=torch.int32)
    splan = P2PPlan(a_s, b_s, d, slcl_ops.pad_meta(la_s, ia), slcl_ops.pad_meta(lb_s, ib), shift, w_s, T, n_class=0,
                    a_selfcol=sc_s, b_selfrow=sr_s)
    sgraph = splan.capture_graph()

    def timed(fn, iters=20):
        for _ in range(3):
            fn()
        torch.cuda.synchronize(dev)
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        for _ in range(iters):
            fn()
        e.record()
        torch.cuda.synchronize(dev)
        return s.elapsed_time(e) / iters

    out = {}
    # cfg3 through the PUBLIC API: class-balanced draw (one randperm on the device) + per-class compaction + gather of the
    # 4096 + 16384 unit rows + tensor-core sweeps + scatter of the row gradients back into the NCHW map; no host sync
    from slcl.p2p import sampled_supcon_loss
    fmap = torch.randn(16, 256, 64, 64, device=dev, generator=gen).requires_grad_(True)
    lmap = torch.randint(0, 5, (16, 64, 64), device=dev, generator=gen)

    def api_step():
        loss_s = sampled_supcon_loss(fmap, lmap, A, M, 5, temperature=T)
        loss_s.backward()
        fmap.grad = None
    ms = timed(api_step, iters=10)
    out["cfg3 through the public API: sampled_supcon_loss (draw + compaction + gather + sweeps + scatter), fwd+bwd, eager"] = {
        "ms": ms, "algorithmic_flop": 8.0 * A * M * d, "achieved_TFLOPs": 8.0 * A * M * d / (ms * 1e-3) / 1e12,
        "frac_of_bf16_peak": 8.0 * A * M * d / (ms * 1e-3) / 1e12 / tf_peak, "rows_per_s": (A + M) / (ms * 1e-3)}
    try:        # nothing in that call synchronises, so the whole public-API step can be replayed as ONE CUDA graph
        fmap_g = fmap.detach().clone().requires_grad_(True)
        gen_g = torch.Generator(device=dev).manual_seed(77)

        def api_step_g():
            loss_s = sampled_supcon_loss(fmap_g, lmap, A, M, 5, temperature=T, generator=gen_g)
            loss_s.backward()
            fmap_g.grad = None
            return loss_s.detach()
        side = torch.cuda.Stream(dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):
            api_step_g()
        torch.cuda.current_stream(dev).wait_stream(side)
        torch.cuda.synchronize(dev)
        g_api = torch.cuda.CUDAGraph()
        g_api.register_generator_state(gen_g)
        with torch.cuda.graph(g_api):
            keep_api = api_step_g()          # noqa: F841
        ms = timed(g_api.replay, iters=10)
        out["cfg3 through the public API: the same sampled_supcon_loss step (incl. the draw) replayed as one CUDA graph"] = {
            "ms": ms, "algorithmic_flop": 8.0 * A * M * d, "achieved_TFLOPs": 8.0 * A * M * d / (ms * 1e-3) / 1e12,
            "frac_of_bf16_peak": 8.0 * A * M * d / (ms * 1e-3) / 1e12 / tf_peak, "rows_per_s": (A + M) / (ms * 1e-3)}
        del g_api, keep_api, fmap_g
    except Exception as exc:  # noqa: BLE001
        print(f"[bench] sampled_supcon_loss: graph capture unavailable ({exc!r})", file=sys.stderr)
    del fmap, lmap
    # BlockConLoss at the reference's documented shape (1, 2, 32, 224, 224), 32 x 32 tiles: 49 tiles of 2048 rows as ONE
    # block-diagonal problem (the reference and the per-tile loop launch 49 separate SupCon problems)
    from slcl.loss import BlockConLoss
    fb = torch.nn.functional.normalize(torch.randn(1, 2, 32, 224, 224, device=dev, generator=gen), dim=2).requires_grad_(True)
    lbk = torch.randint(0, 4, (1, 2, 224, 224), device=dev, generator=gen)
    crit = BlockConLoss(0.7, 32)

    def block_step():
        loss_b = crit(fb, lbk)
        loss_b.backward()
        fb.grad = None
    ms = timed(block_step, iters=10)
    m_t, n_t = 2048, 49
    fl = 8.0 * n_t * m_t * m_t * 64          # 32 channels padded to 64 bf16 columns
    out["BlockConLoss (1,2,32,224,224) fwd+bwd through the Python API, 49 tiles batched"] = {
        "ms": ms, "algorithmic_flop": fl, "achieved_TFLOPs": fl / (ms * 1e-3) / 1e12, "frac_of_bf16_peak": fl / (ms * 1e-3) / 1e12 / tf_peak,
        "rows_per_s": n_t * m_t / (ms * 1e-3)}
    try:        # the same call replayed as one CUDA graph: the device time behind the host-dispatch-bound eager number
        fbg = fb.detach().clone().requires_grad_(True)

        def block_step_g():
            loss_b = crit(fbg, lbk)
            loss_b.backward()
            fbg.grad = None
        side = torch.cuda.Stream(dev)
        side.wait_stream(torch.cuda.current_stream(dev))
        with torch.cuda.stream(side):
            block_step_g()
        torch.cuda.current_stream(dev).wait_stream(side)
        torch.cuda.synchronize(dev)
        g_blk = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g_blk):
            block_step_g()
        ms_g = timed(g_blk.replay, iters=20)
        out["BlockConLoss (1,2,32,224,224) fwd+bwd, the same Python-API step replayed as one CUDA graph"] = {
            "ms": ms_g, "algorithmic_flop": fl, "achieved_TFLOPs": fl / (ms_g * 1e-3) / 1e12,
            "frac_of_bf16_peak": fl / (ms_g * 1e-3) / 1e12 / tf_peak, "rows_per_s": n_t * m_t / (ms_g * 1e-3)}
        del g_blk, fbg
    except Exception as exc:  # noqa: BLE001
        print(f"[bench] BlockConLoss: graph capture unavailable ({exc!r})", file=sys.stderr)
    crit.batched = False
    ms_loop = timed(block_step, iters=3)
    out["BlockConLoss (1,2,32,224,224) fwd+bwd, per-tile loop (49 SupCon calls, the reference's structure)"] = {
        "ms": ms_loop, "algorithmic_flop": fl, "achieved_TFLOPs": fl / (ms_loop * 1e-3) / 1e12,
        "frac_of_bf16_peak": fl / (ms_loop * 1e-3) / 1e12 / tf_peak, "rows_per_s": n_t * m_t / (ms_loop * 1e-3)}
    del fb, lbk
    for name, fn, flops in (("cfg3 p2p forward only (A4096 x M16384 x d256, bf16 tcgen05)", plan.forward_only, 2.0 * A * M * d),
                            ("cfg3 p2p forward keeping U for the backward (S + E.B)", plan.forward, 4.0 * A * M * d),
                            ("cfg3 p2p backward (dB sweep: S recomputed + G^T.A; dA from U)", plan.backward, 4.0 * A * M * d),
                            ("cfg3 p2p fwd+bwd, one CUDA graph", graph.replay, 8.0 * A * M * d),
                            ("cfg3 p2p fwd+bwd, general labels, one CUDA graph", ggraph.replay, 8.0 * A * M * d),
                            ("cfg3 p2p fwd+bwd, general labels sorted by label + self maps, one CUDA graph", sgraph.replay,
                             8.0 * A * M * d)):
        ms = timed(fn)
        tf = flops / (ms * 1e-3) / 1e12
        out[name] = {"ms": ms, "algorithmic_flop": flops, "achieved_TFLOPs": tf, "frac_of_bf16_peak": tf / tf_peak,
                     "rows_per_s": (A + M) / (ms * 1e-3)}
    return out


def main():
    args = parse_args()
    # Keep stdout for the ONE JSON line: libraries (NCCL prints its version banner to stdout) write to
    # stderr while the benchmark runs; the real stdout is restored just for the final print.
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    lines = []
    import builtins
    orig_print = builtins.print

    def capture(*a, **k):
        if k.get("file") in (None, sys.stdout):
            lines.append(" ".join(str(x) for x in a))
        else:
            orig_print(*a, **k)
    builtins.print = capture
    failed = None
    try:
        if args.impl == "reference":
            run_reference(args)
        else:
            run_slcl(args)
    except SystemExit as exc:          # the JSON line (if any) is still printed before the run fails
        failed = exc
    finally:
        builtins.print = orig_print
        sys.stdout.flush()
        os.dup2(real_stdout, 1)
        os.close(real_stdout)
    for ln in lines:
        print(ln, flush=True)
    if failed is not None:
        raise failed


if __name__ == "__main__":
    main()
