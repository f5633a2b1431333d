"""slcl.loss.mccl_step: the MCCL loss section (Trainer_MCCL.py:275-326) in one forward and one backward call, against the
composition of drop-in calls it is defined as (cal_centroid x 3 + mccl_centroid_losses), the oracle, the sharded global
batch over loopback mailboxes and the NCCL route's kernels, a CUDA-graph replay and the launch count.

The sums come from the same sweeps and the same reduce order as the separate calls, so sums and counts are compared
bit for bit; the logits fixtures keep every certainty and arg-max decision away from its rounding edge (as
test_centroid_logits.py)."""
import pytest
import torch

from oracle import slcl_oracle as O

pytestmark = pytest.mark.gpu

THR = 0.6


def dev():
    return torch.device("cuda:0")


@pytest.fixture()
def no_tf32():
    old = (torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32)
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    yield
    torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = old


def close(a, b, rtol, atol=1e-7):
    torch.testing.assert_close(torch.as_tensor(a).double().cpu(), torch.as_tensor(b).double().cpu(), rtol=rtol, atol=atol)


def grad_close(a, b, rtol=1e-5, floor=0.1):
    b = torch.as_tensor(b).double()
    close(a, b, rtol=rtol, atol=rtol * (float(b.abs().max()) + 1e-30) * floor)


def logits(b, k, h, w, gen, scale=3.0):
    z = scale * torch.randn(b, k, h, w, device=dev(), generator=gen)
    for _ in range(100):
        p = torch.softmax(z, 1)
        top = torch.topk(z, 2, dim=1).values
        bad = ((p.amax(1) - THR).abs() < 1e-4) | ((top[:, 0] - top[:, 1]) < 1e-3)
        n_bad = int(bad.sum())
        if n_bad == 0:
            return z
        zp = z.permute(0, 2, 3, 1)
        zp[bad] = scale * torch.randn(n_bad, k, device=dev(), generator=gen)
        z = zp.permute(0, 3, 1, 2).contiguous()
    raise AssertionError("could not draw logits away from the decision edges")


def case(b, c, h, w, k, parts, from_logits, seed, empty_class=False, b_t=None, b_a=None):
    gen = torch.Generator(device=dev()).manual_seed(seed)
    b_t = b if b_t is None else b_t
    b_a = b if b_a is None else b_a
    d = dict(ft_s=torch.randn(b, c, h, w, device=dev(), generator=gen),
             labels_s=torch.randint(0, k, (b, h, w), device=dev(), generator=gen),
             ft_t=torch.randn(b_t, c, h, w, device=dev(), generator=gen),
             ft_a=torch.randn(b_a, c, h, w, device=dev(), generator=gen))
    z_t, z_a = logits(b_t, k, h, w, gen), logits(b_a, k, h, w, gen)
    if empty_class:                       # class k-1 never labelled in the source, never the arg-max in the targets
        d["labels_s"] = d["labels_s"].clamp(max=k - 2)
        z_t[:, k - 1] -= 30.0
        z_a[:, k - 1] -= 30.0
    d["pred_t"] = z_t if from_logits else torch.softmax(z_t, 1)
    d["pred_a"] = z_a if from_logits else torch.softmax(z_a, 1)
    d["part_id"] = (torch.randperm(b_t * h * w, device=dev(), generator=gen) % parts).to(torch.int32) if parts > 1 else None
    d["prev"] = torch.randn(k, c, device=dev(), generator=gen)
    return d


def composition(d, k, parts, from_logits, thr, weighted, prev, aug, split=False, bg=False):
    """The definition of mccl_step (Trainer_MCCL.py:275-326) through the drop-in calls."""
    from slcl.loss import mccl_centroid_losses
    from slcl.utils_ import cal_centroid
    cs, _, _ = cal_centroid(d["ft_s"], d["labels_s"], previous_centroid=d["prev"] if prev else None, momentum=0.9, n_class=k)
    cs = cs.detach()
    ct, _, _ = cal_centroid(d["ft_t"], d["pred_t"], pseudo_label=True, partition=parts, threshold=thr, weighted_ave=weighted,
                            n_class=k, part_id=d["part_id"], from_logits=from_logits)
    ca = None
    if aug:
        ca, _, _ = cal_centroid(d["ft_a"], d["pred_a"], pseudo_label=True, threshold=thr, weighted_ave=weighted, n_class=k,
                                from_logits=from_logits)
    total, terms = mccl_centroid_losses(cs, ct, ca, 1.0, 1.0, 4e-5, split=split, bg=bg)
    return total, terms, cs, ct, ca


def fused(d, k, parts, from_logits, thr, weighted, prev, aug, split=False, bg=False, group=None):
    from slcl.loss import mccl_step
    return mccl_step(d["ft_s"], d["labels_s"], d["ft_t"], d["pred_t"], d["ft_a"] if aug else None,
                     d["pred_a"] if aug else None, n_class=k, partition=parts, part_id=d["part_id"], threshold=thr,
                     weighted_ave=weighted, from_logits=from_logits, previous_centroid_s=d["prev"] if prev else None,
                     momentum=0.9, split=split, bg=bg, group=group)


def leaves(d):
    out = dict(d)
    for key in ("ft_s", "ft_t", "ft_a", "pred_t", "pred_a"):
        out[key] = d[key].clone().requires_grad_(True)
    return out


def run(fn, d, *args, **kw):
    x = leaves(d)
    total, terms, cs, ct, ca = fn(x, *args, **kw)
    total.backward()
    cat = lambda t: torch.cat(t) if isinstance(t, list) else t
    grads = {key: x[key].grad for key in ("ft_s", "ft_t", "ft_a", "pred_t", "pred_a")}
    return total.detach(), terms.detach(), cs.detach(), cat(ct).detach(), None if ca is None else ca.detach(), grads


def check_equal(a, b, aug):
    total, terms, cs, ct, ca, g = a
    total2, terms2, cs2, ct2, ca2, g2 = b
    close(cs, cs2, rtol=1e-6)
    close(ct, ct2, rtol=1e-6)
    if aug:
        close(ca, ca2, rtol=1e-6)
    close(total, total2, rtol=1e-6)
    close(terms, terms2, rtol=1e-6)
    assert g["ft_s"] is None
    for key in ("ft_t", "ft_a", "pred_t", "pred_a"):
        if g2[key] is None:
            assert g[key] is None, key
        else:
            grad_close(g[key], g2[key], rtol=1e-5)


def sums_of(d, k, parts, from_logits, thr, weighted, aug):
    """The separate calls' class sums, stacked in mccl_step's row order."""
    op = torch.ops.slcl
    s = [op.class_sums(d["ft_s"], d["labels_s"].reshape(-1), None, False, 0.0, None, 1, k),
         op.class_sums(d["ft_t"], None, d["pred_t"], weighted, thr, d["part_id"], parts, k, from_logits)]
    if aug:
        s.append(op.class_sums(d["ft_a"], None, d["pred_a"], weighted, thr, None, 1, k, from_logits))
    return torch.cat(s)


def step_sums(d, k, parts, from_logits, thr, weighted, aug, prev):
    losses, cen, sums, dcen = torch.ops.slcl.mccl_step_fwd(
        d["ft_s"], d["labels_s"], d["ft_t"], d["pred_t"], d["part_id"], d["ft_a"] if aug else None,
        d["pred_a"] if aug else None, d["prev"] if prev else None, parts, k, weighted, thr, from_logits, 0.9, False, False,
        True, 1.0, 1.0, 4e-5)
    return sums


MATRIX = [
    # (b, c, h, w, k, parts, from_logits, thr, weighted, prev, aug)
    (2, 32, 32, 32, 2, 1, True, None, True, True, True),
    (2, 32, 32, 32, 2, 2, False, THR, False, False, True),
    (2, 48, 24, 24, 4, 2, True, THR, True, True, True),
    (2, 48, 24, 24, 4, 1, False, None, True, False, False),
    (2, 32, 32, 32, 5, 2, True, None, False, True, False),
    (2, 32, 32, 32, 5, 1, False, THR, True, True, True),
    (2, 128, 16, 16, 8, 2, True, THR, True, False, True),        # P * K = 16 columns, C = 128
    (2, 32, 16, 16, 8, 1, False, None, False, True, True),
    (3, 32, 17, 19, 4, 2, True, THR, True, True, True),          # HW % 4 != 0: the v2 sweep and the scalar backward
    (3, 48, 17, 19, 5, 1, False, None, True, False, True),
]


@pytest.mark.parametrize("cfg", MATRIX, ids=[f"k{m[4]}p{m[5]}c{m[1]}{'L' if m[6] else 'P'}" for m in MATRIX])
def test_equals_the_composition(cfg):
    b, c, h, w, k, parts, from_logits, thr, weighted, prev, aug = cfg
    d = case(b, c, h, w, k, parts, from_logits, seed=hash(cfg) % 10000)
    ref = run(composition, d, k, parts, from_logits, thr, weighted, prev, aug)
    out = run(fused, d, k, parts, from_logits, thr, weighted, prev, aug)
    check_equal(out, ref, aug)
    t = 0.0 if thr is None else thr
    assert torch.equal(step_sums(d, k, parts, from_logits, t, weighted, aug, prev),
                       sums_of(d, k, parts, from_logits, t, weighted, aug))


@pytest.mark.parametrize("split,bg", [(True, False), (False, True), (True, True)])
def test_split_bg_and_an_empty_class(split, bg):
    k, parts = 4, 2
    d = case(2, 32, 32, 32, k, parts, True, seed=77, empty_class=True)
    ref = run(composition, d, k, parts, True, THR, True, True, True, split=split, bg=bg)
    out = run(fused, d, k, parts, True, THR, True, True, True, split=split, bg=bg)
    check_equal(out, ref, True)
    sums = step_sums(d, k, parts, True, THR, True, True, True)
    assert torch.equal(sums, sums_of(d, k, parts, True, THR, True, True))
    assert float(sums[k - 1, -1]) == 0.0                     # the empty source class


def test_generator_draws_the_same_partition_ids():
    from slcl.loss import mccl_step
    from slcl.utils_ import cal_centroid
    k, parts = 4, 2
    d = case(2, 32, 32, 32, k, parts, True, seed=5)
    ct_ref, _, _ = cal_centroid(d["ft_t"], d["pred_t"], pseudo_label=True, partition=parts, n_class=k, weighted_ave=True,
                                generator=torch.Generator(device=dev()).manual_seed(9), from_logits=True)
    _, _, _, ct, _ = mccl_step(d["ft_s"], d["labels_s"], d["ft_t"], d["pred_t"], n_class=k, partition=parts,
                               generator=torch.Generator(device=dev()).manual_seed(9))
    close(torch.cat(ct), torch.cat(ct_ref).detach(), rtol=1e-6)


def test_full_size_cfg5_vs_oracle(no_tf32):
    """configs[4] per GPU: 64 x 32 x 224 x 224 maps, K = 4, P = 2, logits, aug view; loss and gradients against the
    oracle (cal_centroid, ContrastiveLoss, cnr_loss, softmax) in fp32 on the GPU."""
    from slcl.loss import mccl_step
    k, parts, b, c, h = 4, 2, 64, 32, 224
    d = case(b, c, h, h, k, parts, True, seed=505)
    x = leaves(d)
    total, terms, cs, ct, ca = mccl_step(x["ft_s"], x["labels_s"], x["ft_t"], x["pred_t"], x["ft_a"], x["pred_a"], n_class=k,
                                         partition=parts, part_id=d["part_id"], threshold=THR)
    total.backward()
    got = (total.detach(), x["ft_t"].grad, x["ft_a"].grad, x["pred_t"].grad, x["pred_a"].grad)
    del x
    y = leaves(d)
    cs_o, _, _ = O.cal_centroid(y["ft_s"].detach(), y["labels_s"], n_class=k)
    ct_o, _, _ = O.cal_centroid(y["ft_t"], torch.softmax(y["pred_t"], 1), pseudo_label=True, weighted_ave=True,
                                partition=parts, n_class=k, threshold=THR, part_id=d["part_id"])
    ca_o, _, _ = O.cal_centroid(y["ft_a"], torch.softmax(y["pred_a"], 1), pseudo_label=True, weighted_ave=True, n_class=k,
                                threshold=THR)
    inter = sum(O.contrastive_loss(cs_o.detach(), t) for t in ct_o) / parts
    intra = sum(O.contrastive_loss(t, ca_o) for t in ct_o) / parts
    cnr = O.cnr_loss(cs_o.detach(), ct_o)
    ref = inter + intra + 4e-5 * cnr
    ref.backward()
    close(cs, cs_o.detach(), rtol=1e-4, atol=1e-6)
    close(got[0], ref.detach(), rtol=1e-4)
    close(terms, torch.stack([inter, intra, cnr]).detach(), rtol=1e-4, atol=1e-7)
    for a, key in zip(got[1:], ("ft_t", "ft_a", "pred_t", "pred_a")):
        grad_close(a, y[key].grad, rtol=1e-4)


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


def _shard(d, lo, hi, lo_a, hi_a, h, w):
    s = dict(d)
    for key in ("ft_s", "labels_s", "ft_t", "pred_t"):
        s[key] = d[key][lo:hi]
    s["ft_a"], s["pred_a"] = d["ft_a"][lo_a:hi_a], d["pred_a"][lo_a:hi_a]
    if d["part_id"] is not None:
        s["part_id"] = d["part_id"].reshape(-1, h * w)[lo:hi].reshape(-1)
    return s


@pytest.mark.parametrize("world,sizes", [(2, [1, 3]), (3, [2, 1, 2])], ids=["w2", "w3"])
def test_sharded_equals_the_global_batch(world, sizes):
    from slcl.peer import LoopbackMailboxes
    from slcl.utils_ import cal_centroid
    k, parts, c, h, w = 4, 2, 32, 20, 24
    b = sum(sizes)
    sizes_a = sizes[::-1]
    d = case(b, c, h, w, k, parts, True, seed=31 + world)
    bounds = [sum(sizes[:r]) for r in range(world + 1)]
    bounds_a = [sum(sizes_a[:r]) for r in range(world + 1)]
    shards = [_shard(d, bounds[r], bounds[r + 1], bounds_a[r], bounds_a[r + 1], h, w) for r in range(world)]
    glob = run(fused, d, k, parts, True, THR, True, True, True)
    sums_g = step_sums(d, k, parts, True, THR, True, True, True)

    streams = [torch.cuda.Stream(dev()) for _ in range(world)]
    _on_streams(streams, lambda r: run(fused, shards[r], k, parts, True, THR, True, True, True))
    torch.cuda.synchronize()
    # load the exchanging kernels one kind per round: a kernel loaded on its first launch while a peer's kernel already
    # polls could keep the host from enqueueing the rank that kernel waits for
    warm = LoopbackMailboxes(world, dev(), timeout_s=20.0).boxes
    _on_streams(streams, lambda r: cal_centroid(shards[r]["ft_s"], shards[r]["labels_s"], n_class=k, group=warm[r]))
    torch.cuda.synchronize()
    _on_streams(streams, lambda r: run(fused, shards[r], k, parts, True, THR, True, True, True, group=warm[r]))
    torch.cuda.synchronize()
    assert all(bx.timeouts() == 0 for bx in warm)
    mb = LoopbackMailboxes(world, dev(), timeout_s=20.0)
    boxes = mb.boxes
    res = {}

    def rank_fn(r):
        s = shards[r]
        # a cal_centroid exchange on the same mailbox before and after the step: the epochs interleave
        pre, _, _ = cal_centroid(s["ft_s"], s["labels_s"], n_class=k, group=boxes[r])
        res[r] = run(fused, s, k, parts, True, THR, True, True, True, group=boxes[r])
        post, _, _ = cal_centroid(s["ft_s"], s["labels_s"], n_class=k, group=boxes[r])
        sums = torch.ops.slcl.mccl_step_fwd(s["ft_s"], s["labels_s"], s["ft_t"], s["pred_t"], s["part_id"], s["ft_a"],
                                            s["pred_a"], s["prev"], parts, k, True, THR, True, 0.9, False, False, True, 1.0,
                                            1.0, 4e-5, *boxes[r].args())[2]
        res[r] = res[r] + (pre.detach(), post.detach(), sums)
    _on_streams(streams, rank_fn)
    torch.cuda.synchronize()
    assert all(bx.timeouts() == 0 for bx in boxes)
    cs_g, _, _ = cal_centroid(d["ft_s"], d["labels_s"], n_class=k)
    for r in range(world):
        total, terms, cs, ct, ca, g, pre, post, sums = res[r]
        assert torch.equal(sums[:, -1], sums_g[:, -1])                  # pixel counts / weight sums of the GLOBAL batch
        close(sums, sums_g, rtol=1e-9, atol=1e-9)
        close(total, glob[0], rtol=1e-5)
        close(terms, glob[1], rtol=1e-5)
        for a, bb in zip((cs, ct, ca), glob[2:5]):
            close(a, bb, rtol=1e-5, atol=1e-6)
        lo, hi, lo_a, hi_a = bounds[r], bounds[r + 1], bounds_a[r], bounds_a[r + 1]
        grad_close(g["ft_t"], glob[5]["ft_t"][lo:hi])
        grad_close(g["pred_t"], glob[5]["pred_t"][lo:hi])
        grad_close(g["ft_a"], glob[5]["ft_a"][lo_a:hi_a])
        grad_close(g["pred_a"], glob[5]["pred_a"][lo_a:hi_a])
        close(pre, cs_g, rtol=1e-5, atol=1e-6)
        close(post, cs_g, rtol=1e-5, atol=1e-6)
        for a, bb in zip(res[r][:5], res[0][:5]):                         # identical bits on every rank
            assert torch.equal(a, bb)

    # the NCCL route's kernels: per-rank sums summed here in rank order, then the finish kernel and the backward
    op = torch.ops.slcl
    loc = [op.mccl_step_fwd_local(s["ft_s"], s["labels_s"], s["ft_t"], s["pred_t"], s["part_id"], s["ft_a"], s["pred_a"],
                                  parts, k, True, THR, True) for s in shards]
    tot = loc[0]
    for s in loc[1:]:
        tot = tot + s
    assert torch.equal(tot[:, -1], sums_g[:, -1])
    losses, cen, dcen = op.mccl_step_finish(tot, True, d["prev"], parts, k, 0.9, False, False, True, 1.0, 1.0, 4e-5)
    close(losses[0], glob[0], rtol=1e-5)
    close(cen[k:(parts + 1) * k], glob[3], rtol=1e-5, atol=1e-6)
    one = torch.ones(1, device=dev())
    for r, s in enumerate(shards):
        df_t, dp_t, df_a, dp_a = op.mccl_step_bwd(s["ft_t"], s["pred_t"], s["part_id"], s["ft_a"], s["pred_a"], parts, k, True,
                                                  THR, True, tot, dcen, one, True)
        grad_close(df_t, glob[5]["ft_t"][bounds[r]:bounds[r + 1]])
        grad_close(dp_a, glob[5]["pred_a"][bounds_a[r]:bounds_a[r + 1]])


def test_nccl_route_through_autograd(monkeypatch):
    """The NCCL branch of the autograd node end to end (local sums -> all_reduce_sums -> finish kernel, then the
    backward): ranks run one after another, and all_reduce_sums returns the ranks' local sums added in rank order, what
    an NCCL all-reduce hands every rank."""
    import slcl.distributed as D
    from slcl import functional as SF
    k, parts, c, h, w = 4, 2, 32, 20, 24
    sizes, sizes_a = [1, 3, 2], [2, 3, 1]
    b = sum(sizes)
    d = case(b, c, h, w, k, parts, True, seed=61)
    bounds = [sum(sizes[:r]) for r in range(len(sizes) + 1)]
    bounds_a = [sum(sizes_a[:r]) for r in range(len(sizes) + 1)]
    shards = [_shard(d, bounds[r], bounds[r + 1], bounds_a[r], bounds_a[r + 1], h, w) for r in range(len(sizes))]
    glob = run(fused, d, k, parts, True, THR, True, True, True)
    op = torch.ops.slcl
    loc = [op.mccl_step_fwd_local(s["ft_s"], s["labels_s"], s["ft_t"], s["pred_t"], s["part_id"], s["ft_a"], s["pred_a"],
                                  parts, k, True, THR, True) for s in shards]
    tot = loc[0]
    for s in loc[1:]:
        tot = tot + s
    seen = []

    def all_reduce_sums(sums, group):
        assert group is True
        seen.append(sums)
        return tot
    monkeypatch.setattr(D, "all_reduce_sums", all_reduce_sums)

    def nccl_step(x):
        total, terms, cen, sums = SF.mccl_step(x["ft_s"], x["labels_s"], x["ft_t"], x["pred_t"], x["part_id"], x["ft_a"],
                                               x["pred_a"], x["prev"], n_partitions=parts, n_class=k, weighted=True,
                                               threshold=THR, from_logits=True, momentum=0.9, split=False, bg=False,
                                               norm=True, inter_w=1.0, intra_w=1.0, cnr_w=4e-5, group=True)
        return total, terms, cen[:k], cen[k:(parts + 1) * k], cen[(parts + 1) * k:]
    for r, s in enumerate(shards):
        total, terms, cs, ct, ca, g = run(nccl_step, s)
        assert torch.equal(seen[-1], loc[r])                          # the local sums of this rank went to the all-reduce
        close(total, glob[0], rtol=1e-5)
        close(terms, glob[1], rtol=1e-5)
        for a, bb in zip((cs, ct, ca), glob[2:5]):
            close(a, bb, rtol=1e-5, atol=1e-6)
        assert g["ft_s"] is None
        grad_close(g["ft_t"], glob[5]["ft_t"][bounds[r]:bounds[r + 1]])
        grad_close(g["pred_t"], glob[5]["pred_t"][bounds[r]:bounds[r + 1]])
        grad_close(g["ft_a"], glob[5]["ft_a"][bounds_a[r]:bounds_a[r + 1]])
        grad_close(g["pred_a"], glob[5]["pred_a"][bounds_a[r]:bounds_a[r + 1]])


def test_no_host_sync_and_cuda_graph_replay():
    k, parts = 4, 2
    d = case(4, 32, 64, 64, k, parts, True, seed=92)
    eager = run(fused, d, k, parts, True, THR, True, True, True)
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        again = run(fused, d, k, parts, True, THR, True, True, True)
    finally:
        torch.cuda.set_sync_debug_mode(0)
    torch.cuda.synchronize()
    check_equal(again, eager, True)

    x = leaves(d)

    def step():
        total, *_ = fused(x, k, parts, True, THR, True, True, True)
        total.backward()
        return total.detach()
    side = torch.cuda.Stream(dev())
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        step()
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    for key in ("ft_t", "ft_a", "pred_t", "pred_a"):
        x[key].grad = None
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        static_total = step()
    for _ in range(2):
        graph.replay()
    torch.cuda.synchronize()
    close(static_total, eager[0], rtol=1e-6, atol=0.0)
    for key in ("ft_t", "ft_a", "pred_t", "pred_a"):
        grad_close(x[key].grad, eager[5][key], rtol=1e-6)


def test_launch_count():
    """With part_id given, an eager step is at most 4 kernels forward (one sweep per set, the tail) and 3 backward, and
    nothing else reaches the GPU: every CUDA event of the step is counted (the upstream gradient is passed in, so
    autograd's seed fill is not part of the step)."""
    from torch.profiler import ProfilerActivity, profile
    k, parts = 4, 2
    d = case(4, 32, 64, 64, k, parts, True, seed=93)
    run(fused, d, k, parts, True, THR, True, True, True)              # warm up
    x = leaves(d)
    g = torch.ones((), device=dev())
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        total, *_ = fused(x, k, parts, True, THR, True, True, True)
        total.backward(g)
        torch.cuda.synchronize()
    names = [ev.name for ev in prof.events() if ev.device_type == torch.autograd.DeviceType.CUDA]
    assert len(names) <= 7 and all("slcl" in n for n in names), names
    tail = [i for i, n in enumerate(names) if "mccl_step_tail_kernel" in n]
    assert len(tail) == 1 and tail[0] <= 3, names                      # the sweeps and the tail: forward
    assert "mccl_step_bwd_prep_kernel" in names[tail[0] + 1], names    # then the backward
    assert len(names) - tail[0] - 1 <= 3, names
