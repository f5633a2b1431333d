"""slcl.loss.mpscl_step: the MPSCL loss section (Trainer_MPSCL.py:133-147) in one forward and one backward call, against
the composition of drop-in calls it is defined as (update_class_center_iter + generate_pseudo_label + two
mpcl_loss_calc), the oracle, the sharded global batch over loopback mailboxes and the NCCL route's kernels, the launch
count, host synchronisation and a CUDA-graph replay.

The step runs the same sweeps, reductions and per-pixel arithmetic as the separate calls, so the centres, the pseudo
labels and mask, both losses and both gradients are compared bit for bit."""
import pytest
import torch

from oracle import slcl_oracle as O

pytestmark = pytest.mark.gpu

W_S, W_T = 1.0, 0.1            # the trainer's weighting of the two losses


def dev():
    return torch.device("cuda:0")


def case(b_s, b_t, c, h, w, k, seed, absent=False):
    gen = torch.Generator(device=dev()).manual_seed(seed)
    d = dict(ft_s=torch.randn(b_s, c, h, w, device=dev(), generator=gen),
             labels_s=torch.randint(0, k, (b_s, h, w), device=dev(), generator=gen),
             ft_t=torch.randn(b_t, c, h, w, device=dev(), generator=gen),
             centres=torch.randn(k, c, device=dev(), generator=gen))
    if absent:
        d["labels_s"] = d["labels_s"].clamp(max=k - 2)
    return d


def modules(k, m_s=0.4, m_t=0.2, easy_s=False, easy_t=False, t_s=1.0, t_t=1.0, bt_s=1.0, bt_t=1.0):
    from slcl.loss import MPCL
    return (MPCL(dev(), num_class=k, temperature=t_s, m=m_s, base_temperature=bt_s, easy_margin=easy_s),
            MPCL(dev(), num_class=k, temperature=t_t, m=m_t, base_temperature=bt_t, easy_margin=easy_t))


def composition(x, mods, k, th, m=0.9, group=None):
    """The definition of mpscl_step (Trainer_MPSCL.py:133-147) through the drop-in calls."""
    from slcl.loss import mpcl_loss_calc
    from slcl.utils_ import generate_pseudo_label, update_class_center_iter
    centres = update_class_center_iter(x["ft_s"], x["labels_s"], x["centres"], m=m, num_class=k, group=group)
    hard, mask = generate_pseudo_label(x["ft_t"], centres, th)
    loss_s = mpcl_loss_calc(x["ft_s"], x["labels_s"], centres.detach(), mods[0], tag='source', group=group)
    loss_t = mpcl_loss_calc(x["ft_t"], hard, centres.detach(), mods[1], pixel_sel_loc=mask, tag='target', group=group)
    return loss_s, loss_t, centres, hard, mask


def fused(x, mods, k, th, m=0.9, group=None):
    from slcl.loss import mpscl_step
    return mpscl_step(x["ft_s"], x["labels_s"], x["ft_t"], x["centres"], mods[0], mods[1], m=m, num_class=k,
                      pixel_sel_th=th, group=group)


def run(fn, d, *args, which="both", **kw):
    x = dict(d)
    x["ft_s"] = d["ft_s"].clone().requires_grad_(True)
    x["ft_t"] = d["ft_t"].clone().requires_grad_(True)
    loss_s, loss_t, centres, hard, mask = fn(x, *args, **kw)
    if which == "both":
        (W_S * loss_s + W_T * loss_t).backward()
    elif which == "source":
        (W_S * loss_s).backward()
    else:
        (W_T * loss_t).backward()
    return dict(loss_s=loss_s.detach(), loss_t=loss_t.detach(), centres=centres.detach(), hard=hard, mask=mask,
                g_s=x["ft_s"].grad, g_t=x["ft_t"].grad)


def assert_same(a, b):
    for key in a:
        if b[key] is None:
            assert a[key] is None, key
        else:
            assert a[key] is not None and torch.equal(a[key], b[key]), key


MATRIX = [
    # (b_s, b_t, c, h, w, k, margins/constants, threshold)
    (2, 2, 32, 32, 32, 2, {}, 0.25),
    (2, 3, 32, 24, 24, 4, {}, 0.25),
    (3, 2, 20, 32, 32, 4, dict(easy_s=True), 0.1),
    (2, 2, 128, 16, 16, 5, dict(m_s=0.5, m_t=0.3, easy_t=True, t_s=0.07, bt_s=0.07), 0.05),
    (2, 1, 32, 16, 16, 8, dict(t_t=0.5, bt_t=0.7), 0.02),
    (3, 2, 32, 17, 19, 4, {}, 0.25),                 # HW % 4 != 0: scalar loads on both maps
    (1, 2, 20, 17, 19, 5, dict(easy_s=True, easy_t=True), 0.1),
    (2, 3, 128, 9, 11, 8, dict(m_s=0.2, m_t=0.4), 0.02),
]


@pytest.mark.parametrize("cfg", MATRIX, ids=[f"k{m[5]}c{m[2]}hw{m[3] * m[4]}b{m[0]}{m[1]}" for m in MATRIX])
def test_equals_the_composition(cfg):
    b_s, b_t, c, h, w, k, kw, th = cfg
    d = case(b_s, b_t, c, h, w, k, seed=hash(cfg[:6]) % 10000)
    mods = modules(k, **kw)
    ref = run(composition, d, mods, k, th)
    out = run(fused, d, mods, k, th)
    assert_same(out, ref)
    assert 0 < int(out["mask"].sum()) < out["mask"].numel()


def test_mixed_load_widths():
    """A source map at a misaligned offset (scalar loads) and a vec4 target map: one launch per map, same results."""
    k, c, h, w = 4, 32, 16, 16
    d = case(2, 2, c, h, w, k, seed=3)
    base = torch.cat([torch.zeros(1, device=dev()), d["ft_s"].reshape(-1)])
    mods = modules(k)
    res = []
    for fn in (composition, fused):
        buf = base.clone().requires_grad_(True)
        ft = d["ft_t"].clone().requires_grad_(True)
        x = dict(d, ft_s=buf[1:].view(2, c, h, w), ft_t=ft)
        assert x["ft_s"].data_ptr() % 16 != 0 and x["ft_s"].is_contiguous()
        loss_s, loss_t, centres, hard, mask = fn(x, mods, k, 0.25)
        (W_S * loss_s + W_T * loss_t).backward()
        res.append(dict(loss_s=loss_s.detach(), loss_t=loss_t.detach(), centres=centres.detach(), hard=hard, mask=mask,
                        g_s=buf.grad, g_t=ft.grad))
    assert_same(res[1], res[0])


def test_absent_class_keeps_its_ema_row():
    k = 4
    d = case(2, 2, 32, 16, 16, k, seed=11, absent=True)
    mods = modules(k)
    out = run(fused, d, mods, k, 0.25)
    assert_same(out, run(composition, d, mods, k, 0.25))
    torch.testing.assert_close(out["centres"][k - 1], d["centres"][k - 1], rtol=1e-6, atol=1e-7)


def test_threshold_that_selects_no_pixel():
    k = 4
    d = case(2, 2, 32, 16, 16, k, seed=12)
    mods = modules(k)
    out = run(fused, d, mods, k, 2.5)
    assert_same(out, run(composition, d, mods, k, 2.5))
    assert int(out["mask"].sum()) == 0 and float(out["loss_t"]) == 0.0


@pytest.mark.parametrize("which", ["source", "target"])
def test_only_one_loss_back_propagated(which):
    k = 5
    d = case(2, 3, 32, 16, 16, k, seed=13)
    mods = modules(k)
    out = run(fused, d, mods, k, 0.1, which=which)
    assert_same(out, run(composition, d, mods, k, 0.1, which=which))
    assert (out["g_t"] is None) == (which == "source") and (out["g_s"] is None) == (which == "target")


def test_cfg4_shard_vs_oracle():
    """configs[3] per GPU of an 8-GPU run: 16 x 32 x 224 x 224 per map, K = 4, the trainer's margins 0.4 / 0.2; losses,
    centres and gradients against the oracle in fp32 (the target loss on the step's own pseudo labels, which are checked
    against the oracle's separately)."""
    k, b, c, h = 4, 16, 32, 224
    d = case(b, b, c, h, h, k, seed=404)
    from slcl.loss import MPCL
    mods = (MPCL(dev(), num_class=k, temperature=0.07, m=0.4, base_temperature=0.07),
            MPCL(dev(), num_class=k, temperature=0.07, m=0.2, base_temperature=0.07))
    out = run(fused, d, mods, k, 0.25)
    cen_o = O.update_class_center_iter(d["ft_s"], d["labels_s"], d["centres"], m=0.9, num_class=k)
    torch.testing.assert_close(out["centres"], cen_o, rtol=1e-4, atol=1e-6)
    hard_o, mask_o = O.generate_pseudo_label(d["ft_t"], cen_o, 0.25)
    assert float((hard_o != out["hard"]).float().mean()) < 1e-4
    assert float((mask_o != out["mask"]).float().mean()) < 1e-4
    fs, ft = d["ft_s"].clone().requires_grad_(True), d["ft_t"].clone().requires_grad_(True)
    spec = lambda mod: O.MarginSpec(num_class=k, temperature=mod.temperature, m=mod.m, base_temperature=mod.base_temperature)
    ls = O.mpcl_loss_calc(fs, d["labels_s"], cen_o, spec(mods[0]), tag='source')
    lt = O.mpcl_loss_calc(ft, out["hard"], cen_o, spec(mods[1]), pixel_sel_loc=out["mask"], tag='target')
    (W_S * ls + W_T * lt).backward()
    torch.testing.assert_close(out["loss_s"], ls.detach(), rtol=1e-4, atol=0)
    torch.testing.assert_close(out["loss_t"], lt.detach(), rtol=1e-4, atol=0)
    for got, ref in ((out["g_s"], fs.grad), (out["g_t"], ft.grad)):
        torch.testing.assert_close(got, ref, rtol=1e-4, atol=1e-4 * float(ref.abs().max()))


def test_launch_count():
    """An eager step is at most 5 kernels forward and 1 backward, and nothing else reaches the GPU: every CUDA event of
    the step is counted (the upstream gradients are passed in, so autograd's seed fills are not part of the step)."""
    from torch.profiler import ProfilerActivity, profile
    k = 4
    d = case(4, 4, 32, 64, 64, k, seed=93)
    mods = modules(k)
    run(fused, d, mods, k, 0.25)                                        # warm up
    x = dict(d, ft_s=d["ft_s"].clone().requires_grad_(True), ft_t=d["ft_t"].clone().requires_grad_(True))
    g_s, g_t = torch.full((), W_S, device=dev()), torch.full((), W_T, device=dev())
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        loss_s, loss_t, *_ = fused(x, mods, k, 0.25)
        torch.autograd.backward([loss_s, loss_t], [g_s, g_t])
        torch.cuda.synchronize()
    names = [ev.name for ev in prof.events() if ev.device_type == torch.autograd.DeviceType.CUDA]
    assert len(names) <= 6 and all("slcl" in n for n in names), names
    fin = [i for i, n in enumerate(names) if "mpscl_finalize_kernel" in n]
    assert len(fin) == 1 and fin[0] <= 4, names                         # sweep, reduce, prep, forward, finaliser
    assert len(names) - fin[0] - 1 == 1 and "mpscl_bwd_kernel" in names[-1], names


def test_no_host_sync_and_cuda_graph_replay():
    k = 4
    d = case(4, 3, 32, 64, 64, k, seed=92)
    mods = modules(k)
    eager = run(fused, d, mods, k, 0.25)
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        again = run(fused, d, mods, k, 0.25)
    finally:
        torch.cuda.set_sync_debug_mode(0)
    torch.cuda.synchronize()
    assert_same(again, eager)

    x = dict(d, ft_s=d["ft_s"].clone().requires_grad_(True), ft_t=d["ft_t"].clone().requires_grad_(True))

    def step():
        loss_s, loss_t, centres, hard, mask = fused(x, mods, k, 0.25)
        (W_S * loss_s + W_T * loss_t).backward()
        return loss_s.detach(), loss_t.detach(), centres, hard, mask
    side = torch.cuda.Stream(dev())
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        step()
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    x["ft_s"].grad = x["ft_t"].grad = None
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        static = step()
    for _ in range(2):
        x["ft_s"].grad.zero_()
        x["ft_t"].grad.zero_()
        graph.replay()
    torch.cuda.synchronize()
    for a, key in zip(static, ("loss_s", "loss_t", "centres", "hard", "mask")):
        assert torch.equal(a, eager[key]), key
    assert torch.equal(x["ft_s"].grad, eager["g_s"]) and torch.equal(x["ft_t"].grad, eager["g_t"])


# ---------------------------------------------------------------------------
# over the global batch: ranks are CUDA streams of one GPU exchanging through loopback mailboxes
# ---------------------------------------------------------------------------
def _on_streams(streams, fn):
    cur = torch.cuda.current_stream()
    out = []
    for r, st in enumerate(streams):
        st.wait_stream(cur)
        with torch.cuda.stream(st):
            out.append(fn(r))
    for st in streams:
        cur.wait_stream(st)
    return out


def _shards(d, sizes_s, sizes_t):
    bs = [sum(sizes_s[:r]) for r in range(len(sizes_s) + 1)]
    bt = [sum(sizes_t[:r]) for r in range(len(sizes_t) + 1)]
    return [dict(d, ft_s=d["ft_s"][bs[r]:bs[r + 1]], labels_s=d["labels_s"][bs[r]:bs[r + 1]],
                 ft_t=d["ft_t"][bt[r]:bt[r + 1]]) for r in range(len(sizes_s))], bs, bt


@pytest.mark.parametrize("world,sizes_s,sizes_t", [(2, [1, 3], [2, 1]), (3, [2, 1, 2], [1, 2, 2]),
                                                   (4, [1, 2, 1, 3], [2, 1, 1, 1])], ids=["w2", "w3", "w4"])
def test_sharded_equals_the_composition_and_the_global_batch(world, sizes_s, sizes_t):
    from slcl.peer import LoopbackMailboxes
    from slcl.seg import seg_losses
    from slcl.utils_ import cal_centroid
    k, c, h, w = 4, 32, 20, 24
    d = case(sum(sizes_s), sum(sizes_t), c, h, w, k, seed=31 + world)
    shards, bs, bt = _shards(d, sizes_s, sizes_t)
    mods = modules(k)
    glob = run(fused, d, mods, k, 0.25)
    preds = [torch.randn(s["ft_s"].shape[0], k, h, w, device=dev()) for s in shards]
    streams = [torch.cuda.Stream(dev()) for _ in range(world)]
    # load the exchanging kernels one kind per round: a kernel loaded on its first launch while a peer's kernel already
    # polls could keep the host from enqueueing the rank that kernel waits for
    warm = LoopbackMailboxes(world, dev(), timeout_s=20.0).boxes
    for fn in (lambda r: cal_centroid(shards[r]["ft_s"], shards[r]["labels_s"], n_class=k, group=warm[r]),
               lambda r: seg_losses(preds[r], shards[r]["labels_s"], group=warm[r]),
               lambda r: run(composition, shards[r], mods, k, 0.25, group=warm[r]),
               lambda r: run(fused, shards[r], mods, k, 0.25, group=warm[r])):
        _on_streams(streams, fn)
        torch.cuda.synchronize()
    assert all(bx.timeouts() == 0 for bx in warm)

    boxes = LoopbackMailboxes(world, dev(), timeout_s=20.0).boxes
    res, epochs = {}, {}

    def rank_fn(r):
        s = shards[r]
        # cal_centroid and seg_losses exchanges on the same mailbox around the step: the epochs interleave
        pre, _, _ = cal_centroid(s["ft_s"], s["labels_s"], n_class=k, group=boxes[r])
        seg = seg_losses(preds[r], s["labels_s"], group=boxes[r])
        res[r] = run(fused, s, mods, k, 0.25, group=boxes[r])
        post, _, _ = cal_centroid(s["ft_s"], s["labels_s"], n_class=k, group=boxes[r])
        res[r]["pre"], res[r]["post"], res[r]["seg"] = pre.detach(), post.detach(), [t.detach() for t in seg]
        res[r]["ref"] = run(composition, s, mods, k, 0.25, group=boxes[r])
    _on_streams(streams, rank_fn)
    torch.cuda.synchronize()
    assert all(bx.timeouts() == 0 for bx in boxes)
    e0 = [bx.epoch() for bx in boxes]
    _on_streams(streams, lambda r: run(fused, shards[r], mods, k, 0.25, group=boxes[r]))
    torch.cuda.synchronize()
    assert [bx.epoch() - e for bx, e in zip(boxes, e0)] == [2] * world          # two mailbox epochs per step

    cs_g, _, _ = cal_centroid(d["ft_s"], d["labels_s"], n_class=k)
    for r in range(world):
        out, ref = res[r], res[r]["ref"]
        assert_same({key: out[key] for key in ref}, ref)                # the composition with the same mailbox
        for key in ("loss_s", "loss_t", "centres"):
            assert torch.equal(out[key], res[0][key]), key               # identical bits on every rank
        torch.testing.assert_close(out["loss_s"], glob["loss_s"], rtol=1e-5, atol=0)
        torch.testing.assert_close(out["loss_t"], glob["loss_t"], rtol=1e-5, atol=0)
        torch.testing.assert_close(out["centres"], glob["centres"], rtol=1e-5, atol=1e-6)
        assert torch.equal(out["hard"], glob["hard"][bt[r] * h * w:bt[r + 1] * h * w])
        assert torch.equal(out["mask"], glob["mask"][bt[r] * h * w:bt[r + 1] * h * w])
        torch.testing.assert_close(out["g_s"], glob["g_s"][bs[r]:bs[r + 1]], rtol=1e-5, atol=1e-9)
        torch.testing.assert_close(out["g_t"], glob["g_t"][bt[r]:bt[r + 1]], rtol=1e-5, atol=1e-9)
        torch.testing.assert_close(out["pre"], cs_g, rtol=1e-5, atol=1e-6)
        torch.testing.assert_close(out["post"], cs_g, rtol=1e-5, atol=1e-6)

    # the global pixel counts: the source weight sum of every rank's scal is the global N_s, exactly
    scal = torch.ops.slcl.mpscl_step_fwd(shards[0]["ft_s"], shards[0]["labels_s"].reshape(-1), shards[0]["ft_t"],
                                         d["centres"], 0.9, 0.25, k, 1.0, 1.0, 0.4, False, 1.0, 1.0, 0.2, False)[0]
    assert float(scal[2]) == shards[0]["ft_s"].shape[0] * h * w

    # the NCCL route's kernels: global centres from the summed class sums, per-rank pairs summed here in rank order,
    # then the finish kernel and the backward
    op = torch.ops.slcl
    sums = sum(op.class_sums(s["ft_s"], s["labels_s"].reshape(-1), None, False, 0.0, None, 1, k) for s in shards)
    cen = op.ema_finalize(sums, d["centres"], 0.9)
    torch.testing.assert_close(cen, glob["centres"], rtol=1e-5, atol=1e-6)
    loc = [op.mpscl_step_fwd_local(s["ft_s"], s["labels_s"].reshape(-1), s["ft_t"], cen, 0.25, k, 1.0, 1.0, 0.4, False,
                                   1.0, 1.0, 0.2, False) for s in shards]
    pairs = loc[0][0]
    for lo in loc[1:]:
        pairs = pairs + lo[0]
    assert float(pairs[0]) == d["ft_s"].shape[0] * h * w
    scal = op.mpscl_step_finish(pairs)
    torch.testing.assert_close(scal[0], glob["loss_s"], rtol=1e-5, atol=0)
    torch.testing.assert_close(scal[4], glob["loss_t"], rtol=1e-5, atol=0)
    for r, s in enumerate(shards):
        _, cstate, st_s, st_t, hard, mask = loc[r]
        assert torch.equal(hard, glob["hard"][bt[r] * h * w:bt[r + 1] * h * w])
        d_s, d_t = op.mpscl_step_bwd(s["ft_s"], s["ft_t"], st_s, st_t, cstate, scal, torch.full((1,), W_S, device=dev()),
                                     torch.full((1,), W_T, device=dev()), k)
        torch.testing.assert_close(d_s, glob["g_s"][bs[r]:bs[r + 1]], rtol=1e-5, atol=1e-9)
        torch.testing.assert_close(d_t, glob["g_t"][bt[r]:bt[r + 1]], rtol=1e-5, atol=1e-9)


def test_nccl_route_through_autograd(monkeypatch):
    """The NCCL branch of the autograd node end to end, in a process group of one (gloo is not needed: all_reduce is
    replaced by what an NCCL all-reduce hands every rank)."""
    import torch.distributed as dist
    import slcl.distributed as D
    from slcl import functional as SF
    k, c, h, w = 4, 32, 20, 24
    sizes_s, sizes_t = [1, 3, 2], [2, 2, 1]
    d = case(sum(sizes_s), sum(sizes_t), c, h, w, k, seed=61)
    shards, bs, bt = _shards(d, sizes_s, sizes_t)
    mods = modules(k)
    glob = run(fused, d, mods, k, 0.25)
    op = torch.ops.slcl
    sums = sum(op.class_sums(s["ft_s"], s["labels_s"].reshape(-1), None, False, 0.0, None, 1, k) for s in shards)
    cen = op.ema_finalize(sums, d["centres"], 0.9)
    pairs = sum(op.mpscl_step_fwd_local(s["ft_s"], s["labels_s"].reshape(-1), s["ft_t"], cen, 0.25, k, 1.0, 1.0, 0.4,
                                        False, 1.0, 1.0, 0.2, False)[0] for s in shards)
    calls = []
    monkeypatch.setattr(D, "all_reduce_sums", lambda t, group: (calls.append("sums"), sums)[1])

    def all_reduce(t, op=None, group=None):
        calls.append("pairs")
        t.copy_(pairs)
    monkeypatch.setattr(dist, "all_reduce", all_reduce)

    def nccl_step(x, *_a, **_k):
        c_ = lambda mod: (mod.temperature, mod.base_temperature, mod.m, mod.easy_margin)
        return SF.mpscl_step(x["ft_s"], x["labels_s"].reshape(-1), x["ft_t"], x["centres"], m=0.9, sel_threshold=0.25,
                             n_class=k, const_s=c_(mods[0]), const_t=c_(mods[1]), group=True)
    for r, s in enumerate(shards):
        calls.clear()
        out = run(nccl_step, s)
        assert calls == ["sums", "pairs"]                              # two collectives per step
        torch.testing.assert_close(out["loss_s"], glob["loss_s"], rtol=1e-5, atol=0)
        torch.testing.assert_close(out["loss_t"], glob["loss_t"], rtol=1e-5, atol=0)
        torch.testing.assert_close(out["centres"], glob["centres"], rtol=1e-5, atol=1e-6)
        torch.testing.assert_close(out["g_s"], glob["g_s"][bs[r]:bs[r + 1]], rtol=1e-5, atol=1e-9)
        torch.testing.assert_close(out["g_t"], glob["g_t"][bt[r]:bt[r + 1]], rtol=1e-5, atol=1e-9)
