"""Pixel <-> pixel losses over the global batch of data-parallel ranks (``group=`` of ``sampled_supcon_loss``,
``SupConLoss(group=)``, ``LocalConLoss(group=)``).

Ranks are CUDA streams of one GPU exchanging through loopback mailboxes (``slcl.peer.LoopbackMailboxes`` with a row
region): the bulk all-gather kernels and the protocol are those N processes run over NVLink, only the transport differs.
Each rank runs in its own host thread, as a rank would in its own process (the first labelled call of a module reduces the
label range across ranks on the host).  The reference is the same loss on ONE rank over the whole batch.
"""
import threading

import pytest
import torch

from oracle import cases
from oracle import slcl_oracle as O

pytestmark = pytest.mark.gpu

T = 0.7


def dev():
    return torch.device("cuda:0")


def close(a, b, rtol, atol=0.0):
    torch.testing.assert_close(torch.as_tensor(a).double().cpu(), torch.as_tensor(b).double().cpu(), rtol=rtol, atol=atol)


def grad_close(a, b, rtol=1e-4, floor=1.0):
    """rtol per element with an absolute floor of floor * rtol * max|b|.  The floor is the full rtol * max|grad| here, not
    the tenth of it the single-rank parity tests use: the sweeps round each G = exp(S - shift) tile to bf16, and the column
    shift comes from Zs, which the sharded and the unsharded problem sum in different fp32 orders.  So an element whose
    G is near a bf16 rounding boundary moves by one bf16 ulp of that one term (measured: <= 3e-5 max|grad| at world 4)."""
    b = torch.as_tensor(b).double()
    close(a, b, rtol=rtol, atol=rtol * (float(b.abs().max()) + 1e-30) * floor)


def boxes_for(world, rows_bytes, timeout_s=20.0):
    from slcl.peer import LoopbackMailboxes
    return LoopbackMailboxes(world, dev(), timeout_s=timeout_s, rows_bytes=rows_bytes).boxes


def on_ranks(world, fn, boxes, rows_bytes=None):
    """fn(rank, box) for every rank, each in its own thread on its own stream, with boxes[rank]; results in rank order.

    With ``rows_bytes`` the ranks first run fn once on a separate, throw-away set of mailboxes (short time-out, results
    dropped): CUDA loads a kernel's module at its first launch and may wait for the context to go idle while doing so,
    which the polling kernel of another rank (one GPU, ranks as streams) would prevent until it times out.  That pass only
    gets every kernel loaded; ``boxes`` -- their epochs and counters -- are untouched by it, and whatever goes wrong in the
    real pass is reported."""
    if rows_bytes is not None:
        spare = boxes_for(world, rows_bytes, timeout_s=2.0)
        try:
            _threads(world, lambda r: fn(r, spare[r]))
        except Exception:          # noqa: BLE001 - a pass on throw-away mailboxes; the real pass below reports
            pass
        torch.cuda.synchronize()
    return _threads(world, lambda r: fn(r, boxes[r]))


def _threads(world, fn):
    streams = [torch.cuda.Stream(dev()) for _ in range(world)]
    cur = torch.cuda.current_stream(dev())
    for st in streams:
        st.wait_stream(cur)
    out, errs = [None] * world, []

    def run(r):
        try:
            torch.cuda.set_device(dev())
            with torch.cuda.stream(streams[r]):
                out[r] = fn(r)
        except BaseException as e:          # noqa: BLE001 - re-raised on the main thread
            errs.append(e)
    threads = [threading.Thread(target=run, args=(r,)) for r in range(world)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    for st in streams:
        cur.wait_stream(st)
    torch.cuda.synchronize()
    if errs:
        raise errs[0]
    return out


def shard(t, world, r):
    per = t.shape[0] // world
    return t[r * per:(r + 1) * per]


# ---------------------------------------------------------------------------------------------------------------------
# sampled_supcon_loss(group=)
# ---------------------------------------------------------------------------------------------------------------------
def _sampled_case(world, seed, n_anchor=256, n_contrast=1024, k=4):
    g = cases.g(seed)
    b_l, c, h, w = 2, 64, 32, 32
    feat = torch.randn(b_l * world, c, h, w, generator=g).to(dev())
    lab = torch.randint(0, k, (b_l * world, h, w), generator=g).to(dev())
    return feat, lab, n_anchor, n_contrast, k


def _draws(lab, world, n_anchor, n_contrast, k, seed0):
    """Each rank's own class-balanced draw (its own generator), and the rank-major union in global pixel indices."""
    from slcl.p2p import sample_class_balanced
    a_all, c_all = [], []
    for r in range(world):
        lr = shard(lab, world, r)
        a, cc = sample_class_balanced(lr, n_anchor, n_contrast, k, torch.Generator(dev()).manual_seed(seed0 + r))
        a_all.append(a + r * lr.numel())
        c_all.append(cc + r * lr.numel())
    return torch.cat(a_all), torch.cat(c_all)


def _run_sampled(feat, lab, world, boxes, n_anchor, n_contrast, k, analytic, seed0):
    from slcl.p2p import global_record_bytes, sampled_supcon_loss

    def rank(r, box):
        f = shard(feat, world, r).clone().requires_grad_(True)
        loss = sampled_supcon_loss(f, shard(lab, world, r), n_anchor, n_contrast, k, T,
                                   torch.Generator(dev()).manual_seed(seed0 + r), analytic=analytic, group=box)
        loss.backward()
        return loss.detach(), f.grad
    return on_ranks(world, rank, boxes, global_record_bytes(n_anchor, n_contrast, feat.shape[1]))


@pytest.mark.parametrize("world,analytic", [(2, True), (2, False), (4, True), (4, False), (8, True)])
def test_sampled_supcon_global_equals_union_reference(world, analytic):
    from slcl.p2p import global_record_bytes, sampled_supcon_loss
    feat, lab, na, nc, k = _sampled_case(world, 300 + world)
    boxes = boxes_for(world, global_record_bytes(na, nc, feat.shape[1]))
    got = _run_sampled(feat, lab, world, boxes, na, nc, k, analytic, 900)
    a_idx, c_idx = _draws(lab, world, na, nc, k, 900)
    fg = feat.clone().requires_grad_(True)
    ref = sampled_supcon_loss(fg, lab, na, nc, k, T, anchor_idx=a_idx, contrast_idx=c_idx, analytic=analytic)
    ref.backward()
    assert all(bx.timeouts() == 0 and bx.mismatches() == 0 for bx in boxes)
    for r in range(world):
        assert torch.equal(got[r][0], got[0][0])                         # identical bits on every rank
        close(got[r][0], ref, rtol=1e-5)
        grad_close(got[r][1], shard(fg.grad, world, r), rtol=1e-4)
    # and the oracle on the union (bf16 GEMM inputs: 2e-2)
    fo, lab_o = feat.cpu(), lab.reshape(-1).cpu()
    ai, ci = a_idx.cpu(), c_idx.cpu()
    want = O.supcon_rect(O.gather_unit_rows(fo, ai), O.gather_unit_rows(fo, ci), lab_o[ai], lab_o[ci], ai, ci, T)
    close(got[0][0], want, rtol=2e-2)


def test_sampled_supcon_global_short_rank_is_nan_everywhere():
    from slcl.p2p import global_record_bytes
    world = 2
    feat, lab, na, nc, k = _sampled_case(world, 41)
    lab[lab.shape[0] // 2:] = 200                     # rank 1: 96 labelled pixels for 1024 contrast rows: its draw comes up short
    lab[lab.shape[0] // 2, :3] = 3
    boxes = boxes_for(world, global_record_bytes(na, nc, feat.shape[1]))
    got = _run_sampled(feat, lab, world, boxes, na, nc, k, True, 5)
    assert all(torch.isnan(got[r][0]) for r in range(world))
    assert all(bx.timeouts() == 0 for bx in boxes)


def test_rank_that_never_calls_gives_nan_and_timeout():
    from slcl.p2p import global_record_bytes, sampled_supcon_loss
    feat, lab, na, nc, k = _sampled_case(2, 43)
    box = boxes_for(2, global_record_bytes(na, nc, feat.shape[1]), timeout_s=0.3)[0]
    loss = sampled_supcon_loss(shard(feat, 2, 0), shard(lab, 2, 0), na, nc, k, T, torch.Generator(dev()).manual_seed(1),
                               group=box)                                     # rank 1 never calls
    torch.cuda.synchronize()
    assert torch.isnan(loss)
    assert box.timeouts() >= 1
    with pytest.raises(RuntimeError):
        box.check()


def test_ranks_with_different_row_counts_give_nan_and_counted_error():
    from slcl.p2p import global_record_bytes, sampled_supcon_loss
    world = 2
    feat, lab, na, nc, k = _sampled_case(world, 47)
    boxes = boxes_for(world, global_record_bytes(na, nc, feat.shape[1]))

    def rank(r, box):         # rank 1 draws half as many anchors
        return sampled_supcon_loss(shard(feat, world, r), shard(lab, world, r), na if r == 0 else na // 2, nc, k, T,
                                   torch.Generator(dev()).manual_seed(r), group=box)
    got = on_ranks(world, rank, boxes, global_record_bytes(na, nc, feat.shape[1]))
    assert all(torch.isnan(x) for x in got)
    assert all(bx.mismatches() >= 1 for bx in boxes)


def test_record_larger_than_row_slot_is_refused():
    from slcl.p2p import sampled_supcon_loss
    feat, lab, na, nc, k = _sampled_case(2, 53)
    box = boxes_for(2, 4096)[0]
    with pytest.raises(ValueError):
        sampled_supcon_loss(shard(feat, 2, 0), shard(lab, 2, 0), na, nc, k, T, torch.Generator(dev()).manual_seed(0), group=box)


# ---------------------------------------------------------------------------------------------------------------------
# SupConLoss / LocalConLoss(group=)
# ---------------------------------------------------------------------------------------------------------------------
def _module_case(world, seed, labels):
    g = cases.g(seed)
    b_l, v, c, h, w = 2, 2, 32, 16, 16
    feat = torch.nn.functional.normalize(torch.randn(b_l * world, v, c, h, w, generator=g), dim=2).to(dev())
    lab = torch.randint(0, 4, (b_l * world, v, h, w), generator=g)
    if labels == "skewed":               # class 3 only on rank 0; rank world-1 has no foreground at all
        lab[lab == 3] = 2
        lab[0, :, :8, :8] = 3
        lab[-b_l:] = 0
    elif labels == "out_of_range_on_one_rank":         # (both views: the row has a positive, its loss is finite)
        lab[-1, :, 0, 0] = 9
    return feat, lab.to(dev())


def _rows_bytes(feat, stride=1):
    from slcl.p2p import global_record_bytes
    b, v, c, h, w = feat.shape
    m = b * v * (-(-h // stride)) * (-(-w // stride))
    return global_record_bytes(m, m, c, same_rows=True)


@pytest.mark.parametrize("world,labels", [(2, "random"), (4, "random"), (2, "skewed"), (4, "skewed"), (2, "none"),
                                          (4, "none"), (2, "out_of_range_on_one_rank")])
def test_supcon_and_localcon_global_equal_unsharded(world, labels):
    from slcl.p2p import LocalConLoss, SupConLoss
    feat, lab = _module_case(world, 500 + world, labels)
    use_lab = labels != "none"
    boxes = boxes_for(world, _rows_bytes(feat))

    fg = feat.clone().requires_grad_(True)
    lab_all = lab if use_lab else None
    ref = SupConLoss(temperature=T)(fg, lab_all), LocalConLoss(temperature=T, stride=4)(fg, lab_all)
    (ref[0] + 2 * ref[1]).backward()

    def rank(r, box):         # SupConLoss: group at construction; LocalConLoss: group per call
        sup, loc = SupConLoss(temperature=T, group=box), LocalConLoss(temperature=T, stride=4)
        f = shard(feat, world, r).clone().requires_grad_(True)
        lb = shard(lab, world, r) if use_lab else None
        out = sup(f, lb), loc(f, lb, group=box)
        (out[0] + 2 * out[1]).backward()
        return [o.detach() for o in out], f.grad, sup, loc
    got = on_ranks(world, rank, boxes, _rows_bytes(feat))
    mods, locs = [g_[2] for g_ in got], [g_[3] for g_ in got]
    assert all(bx.timeouts() == 0 and bx.mismatches() == 0 for bx in boxes)
    if labels == "out_of_range_on_one_rank":          # every rank took the general sweeps, like the unsharded module
        assert all(m._classes.auto == 0 and lc.supconloss._classes.auto == 0 for m, lc in zip(mods, locs))
    elif use_lab:
        assert all(m._classes.auto == 8 and lc.supconloss._classes.auto == 8 for m, lc in zip(mods, locs))
    for r in range(world):
        for a, b in zip(got[r][0], ref):
            close(a, b, rtol=1e-5, atol=1e-7)
        assert torch.equal(got[r][0][0], got[0][0][0]) and torch.equal(got[r][0][1], got[0][0][1])
        grad_close(got[r][1], shard(fg.grad, world, r), rtol=1e-4)


def test_two_losses_before_one_backward_then_more_steps():
    """Two different group= losses forwarded before one backward, then three more steps: everything the backward reads is
    a private copy, so slot reuse by later exchanges cannot disturb it."""
    from slcl.p2p import SupConLoss, global_record_bytes, sampled_supcon_loss
    world = 2
    feat5, lab5 = _module_case(world, 71, "random")
    feat, lab, na, nc, k = _sampled_case(world, 73)
    rows = max(_rows_bytes(feat5), global_record_bytes(na, nc, feat.shape[1]))
    boxes = boxes_for(world, rows)
    mods = {}
    for step in range(4):
        seed0 = 100 * step
        a_idx, c_idx = _draws(lab, world, na, nc, k, seed0)
        f5g, fg = feat5.clone().requires_grad_(True), feat.clone().requires_grad_(True)
        l1 = SupConLoss(temperature=T, n_class=4)(f5g, lab5)
        l2 = sampled_supcon_loss(fg, lab, na, nc, k, T, anchor_idx=a_idx, contrast_idx=c_idx)
        (l1 + 3 * l2).backward()

        def rank(r, box):     # the same module object on every step of a rank
            sup = mods.setdefault(id(box), SupConLoss(temperature=T, n_class=4, group=box))
            f5 = shard(feat5, world, r).clone().requires_grad_(True)
            f = shard(feat, world, r).clone().requires_grad_(True)
            x1 = sup(f5, shard(lab5, world, r))
            x2 = sampled_supcon_loss(f, shard(lab, world, r), na, nc, k, T, torch.Generator(dev()).manual_seed(seed0 + r),
                                     group=box)
            (x1 + 3 * x2).backward()
            return x1.detach(), x2.detach(), f5.grad, f.grad
        got = on_ranks(world, rank, boxes, rows if step == 0 else None)
        for r in range(world):
            close(got[r][0], l1, rtol=1e-5)
            close(got[r][1], l2, rtol=1e-5)
            grad_close(got[r][2], shard(f5g.grad, world, r))
            grad_close(got[r][3], shard(fg.grad, world, r))
    assert all(bx.timeouts() == 0 and bx.mismatches() == 0 for bx in boxes)


def test_localcon_global_without_foreground_on_any_rank_is_zero():
    """LocalConLoss's "no foreground -> 0" early-out over the global batch: no rank has foreground."""
    from slcl.p2p import LocalConLoss
    world = 2
    feat, lab = _module_case(world, 81, "random")
    lab = torch.zeros_like(lab)
    fg = feat.clone().requires_grad_(True)
    ref = LocalConLoss(temperature=T, stride=4)(fg, lab)
    ref.backward()
    boxes = boxes_for(world, _rows_bytes(feat))

    def rank(r, box):
        f = shard(feat, world, r).clone().requires_grad_(True)
        out = LocalConLoss(temperature=T, stride=4)(f, shard(lab, world, r), group=box)
        out.backward()
        return out.detach(), f.grad
    got = on_ranks(world, rank, boxes, _rows_bytes(feat))
    assert float(ref) == 0.0 and all(bx.timeouts() == 0 for bx in boxes)
    for r in range(world):
        assert float(got[r][0]) == 0.0
        assert torch.equal(got[r][1], shard(fg.grad, world, r))


def test_row_exchanges_interleaved_with_scalar_exchanges_on_one_mailbox():
    """The mailbox's epoch counter is shared: scalar group= exchanges (cal_centroid, update_class_center_iter) before and
    between the pixel <-> pixel losses must neither stall the row exchange nor change any result."""
    from slcl import utils_ as U
    from slcl.p2p import LocalConLoss, global_record_bytes, sampled_supcon_loss
    world = 2
    feat, lab, na, nc, k = _sampled_case(world, 91)
    feat5, lab5 = _module_case(world, 93, "random")
    cen = torch.randn(k, feat.shape[1], generator=cases.g(95)).to(dev())
    rows = max(_rows_bytes(feat5), global_record_bytes(na, nc, feat.shape[1]))
    boxes = boxes_for(world, rows)
    a_idx, c_idx = _draws(lab, world, na, nc, k, 700)
    fg, f5g = feat.clone().requires_grad_(True), feat5.clone().requires_grad_(True)
    want_c, _, _ = U.cal_centroid(feat, lab, n_class=k)
    want_e = U.update_class_center_iter(feat, lab, cen, m=.9, num_class=k)
    l1 = sampled_supcon_loss(fg, lab, na, nc, k, T, anchor_idx=a_idx, contrast_idx=c_idx)
    l2 = LocalConLoss(temperature=T, stride=4)(f5g, lab5)
    (l1 + l2).backward()

    def rank(r, box):
        f, f5 = shard(feat, world, r).clone().requires_grad_(True), shard(feat5, world, r).clone().requires_grad_(True)
        c1, _, _ = U.cal_centroid(shard(feat, world, r), shard(lab, world, r), n_class=k, group=box)
        e1 = U.update_class_center_iter(shard(feat, world, r), shard(lab, world, r), cen, m=.9, num_class=k, group=box)
        x1 = sampled_supcon_loss(f, shard(lab, world, r), na, nc, k, T, torch.Generator(dev()).manual_seed(700 + r),
                                 group=box)
        c2, _, _ = U.cal_centroid(shard(feat, world, r), shard(lab, world, r), n_class=k, group=box)
        e2 = U.update_class_center_iter(shard(feat, world, r), shard(lab, world, r), cen, m=.9, num_class=k, group=box)
        x2 = LocalConLoss(temperature=T, stride=4)(f5, shard(lab5, world, r), group=box)   # + its label-range exchange
        c3, _, _ = U.cal_centroid(shard(feat, world, r), shard(lab, world, r), n_class=k, group=box)
        (x1 + x2).backward()
        return x1.detach(), x2.detach(), f.grad, f5.grad, (c1, c2, c3), (e1, e2)
    got = on_ranks(world, rank, boxes, rows)
    assert all(bx.timeouts() == 0 and bx.mismatches() == 0 for bx in boxes)
    for r in range(world):
        close(got[r][0], l1, rtol=1e-5)
        close(got[r][1], l2, rtol=1e-5)
        grad_close(got[r][2], shard(fg.grad, world, r))
        grad_close(got[r][3], shard(f5g.grad, world, r))
        for c in got[r][4]:
            close(c, want_c, rtol=1e-5, atol=1e-6)
        for e in got[r][5]:
            close(e, want_e, rtol=1e-5, atol=1e-6)
