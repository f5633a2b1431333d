"""Segmentation losses over the global batch of data-parallel ranks (``group=`` of ``seg_losses``, ``loss_calc``,
``dice_loss``, ``jaccard_loss``).

Ranks are CUDA streams of one GPU exchanging through loopback mailboxes (``slcl.peer.LoopbackMailboxes``): the finaliser
kernel and the protocol are those N processes run over NVLink, only the transport differs.  Each rank runs in its own host
thread, as it would in its own process.  The reference is the same call on ONE rank over the ranks' batches concatenated
in rank order, and the oracle (fp32, on the GPU) where the labels are all inside [0, K).

This file sorts after ``test_p2p_global*.py`` on purpose: ranks-as-streams tests depend on which kernels the process has
already loaded, and every test here loads the seg kernels it needs on a one-rank mailbox before its ranks start.
"""
import threading

import pytest
import torch

from oracle import cases
from oracle import slcl_oracle as O

pytestmark = pytest.mark.gpu

W3 = (1.0, 0.5, 2.0)          # upstream weights of {ce, dice, jaccard}: every coefficient of the backward is exercised


def dev():
    return torch.device("cuda:0")


def close(a, b, rtol, atol=0.0):
    torch.testing.assert_close(torch.as_tensor(a).double().cpu(), torch.as_tensor(b).double().cpu(), rtol=rtol, atol=atol)


def grad_close(a, b, rtol=1e-5, floor=1.0):
    """rtol per element with an absolute floor of floor * rtol * max|b| (elements near zero carry the absolute error of
    the large terms they cancel)."""
    b = torch.as_tensor(b).double()
    close(a, b, rtol=rtol, atol=rtol * (float(b.abs().max()) + 1e-30) * floor)


def boxes_for(world, timeout_s=20.0, capacity_words=None):
    from slcl.peer import LoopbackMailboxes
    kw = {} if capacity_words is None else {"capacity_words": capacity_words}
    return LoopbackMailboxes(world, dev(), timeout_s=timeout_s, **kw).boxes


def warm_seg(parts):
    """Load every seg kernel the ranks will launch before they start: CUDA loads a kernel at its first launch and may wait
    for the context to go idle, which another rank's polling kernel (one GPU, ranks as streams) would prevent.  The
    op-level peer entry on a ONE-rank mailbox has nothing to wait for; the NCCL-route kernels and the torch kernels of a
    local forward + backward come along."""
    from slcl import ops, seg
    box = boxes_for(1)[0]
    g = torch.tensor(W3, device=dev())
    for z, lab in parts:
        z = z.detach()
        _, stats, vec = ops.seg_fwd_peer(z, lab, *box.args())
        ops.seg_bwd_global(z, lab, stats, vec, g)
        _, vec = ops.seg_fwd_local(z, lab)
        ops.seg_finish(vec, z.shape[1])
        zz = z.clone().requires_grad_(True)
        (seg.seg_losses(zz, lab) * g).sum().backward()
    torch.cuda.synchronize()


def on_ranks(world, fn, boxes, spare_pass=False):
    """fn(rank, box) for every rank, each in its own thread on its own stream, with boxes[rank]; results in rank order.
    ``spare_pass``: first run fn once on throw-away mailboxes (short time-out, results dropped) so that the kernels of the
    OTHER group= calls fn makes are loaded too; ``boxes`` are untouched by it."""
    if spare_pass:
        spare = boxes_for(world, timeout_s=2.0)
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


def spans(sizes):
    lo, out = 0, []
    for s in sizes:
        out.append((lo, lo + s))
        lo += s
    return out


def _case(sizes, k, h, w, seed):
    gen = cases.g(seed)
    n = sum(sizes)
    z = (1.5 * torch.randn(n, k, h, w, generator=gen)).to(dev())
    lab = torch.randint(0, k, (n, h, w), generator=gen).to(dev())
    return z, lab


def _single(z, lab):
    """seg_losses on ONE rank over the whole batch: (losses, dlogits of sum(W3 * losses))."""
    from slcl import seg
    zz = z.clone().requires_grad_(True)
    out = seg.seg_losses(zz, lab)
    (out * torch.tensor(W3, device=dev())).sum().backward()
    return out.detach(), zz.grad


def _oracle(z, lab):
    """The oracle in fp32 on the GPU (its dice one-hot is built on the default device)."""
    zo = z.clone().requires_grad_(True)
    with dev():
        parts = torch.stack([O.loss_calc(zo, lab), O.dice_loss(zo, lab), O.jaccard_loss(lab, zo)])
    (parts * torch.tensor(W3, device=dev())).sum().backward()
    return parts.detach(), zo.grad


def _run_peer(z, lab, sizes, boxes):
    from slcl import seg
    world = len(sizes)
    sp = spans(sizes)
    g = torch.tensor(W3, device=dev())
    warm_seg([(z[lo:hi], lab[lo:hi]) for lo, hi in sp])

    def rank(r, box):
        lo, hi = sp[r]
        zr = z[lo:hi].clone().requires_grad_(True)
        out = seg.seg_losses(zr, lab[lo:hi], group=box)
        (out * g).sum().backward()
        return out.detach(), zr.grad
    got = on_ranks(world, rank, boxes)
    assert all(bx.timeouts() == 0 for bx in boxes)
    return got


def _check(got, sizes, want, rtol=1e-5):
    losses, dz = want
    for r, (lo, hi) in enumerate(spans(sizes)):
        assert torch.equal(got[r][0], got[0][0])                 # identical bits on every rank
        close(got[r][0], losses, rtol=rtol, atol=1e-7)
        grad_close(got[r][1], dz[lo:hi], rtol=rtol)


# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("hw", [(33, 33), (32, 40)])          # HW % 4 != 0 (scalar path) and HW % 4 == 0 (vec4 path)
@pytest.mark.parametrize("k", [2, 4, 5, 8])
@pytest.mark.parametrize("world", [2, 3, 4])
def test_peer_route_equals_global_batch(world, k, hw):
    h, w = hw
    sizes = [2] * world
    z, lab = _case(sizes, k, h, w, 100 * world + 10 * k + h)
    got = _run_peer(z, lab, sizes, boxes_for(world))
    _check(got, sizes, _single(z, lab))
    _check(got, sizes, _oracle(z, lab))


def test_uneven_shards():
    """8 images over 3 ranks as slcl.distributed.shard_range splits them (3/3/2): the image count travels in the vector."""
    from slcl.distributed import shard_range
    sizes = [hi - lo for lo, hi in (shard_range(8, r, 3) for r in range(3))]
    assert sizes == [3, 3, 2]
    z, lab = _case(sizes, 4, 24, 20, 7001)
    got = _run_peer(z, lab, sizes, boxes_for(3))
    _check(got, sizes, _single(z, lab))
    _check(got, sizes, _oracle(z, lab))


def test_ignored_labels_concentrated_on_one_rank():
    """Labels -100 and K (outside [0, K): not counted by the cross entropy) mostly on rank 0, every pixel of rank 1
    ignored, none on rank 2; the CE denominator is the global count of counted pixels."""
    k = 4
    sizes = [2, 2, 2]
    z, lab = _case(sizes, k, 33, 33, 7002)
    gen = cases.g(7003)
    drop = (torch.rand(2, 33, 33, generator=gen) < 0.7).to(dev())
    kind = (torch.rand(2, 33, 33, generator=gen) < 0.5).to(dev())
    lab[0:2] = torch.where(drop, torch.where(kind, torch.full_like(lab[0:2], -100), torch.full_like(lab[0:2], k)), lab[0:2])
    lab[2:4] = -100
    got = _run_peer(z, lab, sizes, boxes_for(3))
    _check(got, sizes, _single(z, lab))
    assert torch.isfinite(got[0][0]).all()


def test_class_present_on_one_rank_only():
    """Jaccard's per-class union is global: class 3 exists only in rank 1's labels."""
    k = 4
    sizes = [2, 2, 2]
    z, lab = _case(sizes, k, 32, 32, 7004)
    lab[0:2] = lab[0:2] % 3
    lab[4:6] = lab[4:6] % 3
    assert bool((lab[2:4] == 3).any())
    got = _run_peer(z, lab, sizes, boxes_for(3))
    _check(got, sizes, _single(z, lab))
    _check(got, sizes, _oracle(z, lab))


def test_group_none_and_world_of_one_are_the_single_rank_call():
    """group=None, a one-rank mailbox and True without a process group run slcl_seg_fwd / slcl_seg_bwd unchanged."""
    from slcl import ops, seg
    z, lab = _case([3], 5, 33, 33, 7005)
    g = torch.tensor(W3, device=dev())
    losses, stats = ops.seg_fwd(z, lab)
    dz = ops.seg_bwd(z, lab, stats, g)
    one = boxes_for(1)[0]
    for group in (None, one, True):
        zz = z.clone().requires_grad_(True)
        out = seg.seg_losses(zz, lab, group=group)
        (out * g).sum().backward()
        assert torch.equal(out.detach(), losses)
        assert torch.equal(zz.grad, dz)
    assert one.epoch() == 0
    zz = z.clone().requires_grad_(True)
    assert torch.equal(seg.loss_calc(zz, lab, 0, True, group=None).detach(), losses[0] + losses[2])
    assert torch.equal(seg.dice_loss(zz, lab, group=None).detach(), losses[1])
    assert torch.equal(seg.jaccard_loss(lab, zz, group=None).detach(), losses[2])


def test_nccl_route_kernels_without_nccl():
    """The NCCL route's pieces with the all-reduce done here: local vectors summed in rank order, the finishing kernel and
    the global backward.  Summed in rank order like the peer finaliser, the vector and the losses equal the peer route's
    bit for bit."""
    from slcl import ops
    sizes = [3, 3, 2]
    k = 5
    z, lab = _case(sizes, k, 33, 33, 7006)
    g = torch.tensor(W3, device=dev())
    locs = [ops.seg_fwd_local(z[lo:hi], lab[lo:hi]) for lo, hi in spans(sizes)]
    vec = torch.zeros_like(locs[0][1])
    for _, v in locs:
        vec += v
    losses = ops.seg_finish(vec, k)
    dz = torch.cat([ops.seg_bwd_global(z[lo:hi], lab[lo:hi], st, vec, g) for (lo, hi), (st, _) in zip(spans(sizes), locs)])
    ref_l, ref_dz = _single(z, lab)
    close(losses, ref_l, rtol=1e-5, atol=1e-7)
    grad_close(dz, ref_dz)
    assert vec[2 * k + 3].item() == 8.0

    sp = spans(sizes)
    boxes = boxes_for(3)
    warm_seg([(z[lo:hi], lab[lo:hi]) for lo, hi in sp])

    def rank(r, box):
        lo, hi = sp[r]
        return ops.seg_fwd_peer(z[lo:hi], lab[lo:hi], *box.args())
    got = on_ranks(3, rank, boxes)
    assert all(bx.timeouts() == 0 for bx in boxes)
    for r in range(3):
        assert torch.equal(got[r][2], vec)
        assert torch.equal(got[r][0], losses)
        assert torch.equal(got[r][1], locs[r][0])                 # stats stay per local image


def test_peer_route_has_no_host_sync():
    """Forward and backward of the peer route wait for nothing on the host: a second call runs under
    torch.cuda.set_sync_debug_mode("error")."""
    from slcl import seg
    world, sizes = 2, [2, 2]
    z, lab = _case(sizes, 4, 32, 32, 7007)
    boxes = boxes_for(world)
    sp = spans(sizes)
    g = torch.tensor(W3, device=dev())
    ins = [z[lo:hi].clone().requires_grad_(True) for lo, hi in sp]
    labs = [lab[lo:hi] for lo, hi in sp]
    warm_seg(list(zip(ins, labs)))

    def first(r, box):
        (seg.seg_losses(ins[r], labs[r], group=box) * g).sum().backward()
    on_ranks(world, first, boxes)
    for f in ins:
        f.grad = None
    ready, done = threading.Barrier(world), threading.Barrier(world)

    def second(r):
        ready.wait()
        if r == 0:
            torch.cuda.set_sync_debug_mode("error")
        ready.wait()
        try:
            out = seg.seg_losses(ins[r], labs[r], group=boxes[r])
            (out * g).sum().backward()
        finally:
            done.wait()
            if r == 0:
                torch.cuda.set_sync_debug_mode("default")
        return out.detach()
    got = _threads(world, second)
    assert all(bx.timeouts() == 0 for bx in boxes)
    assert [bx.epoch() for bx in boxes] == [2, 2]
    ref_l, ref_dz = _single(z, lab)
    for r, (lo, hi) in enumerate(sp):
        assert torch.equal(got[r], got[0])
        close(got[r], ref_l, rtol=1e-5, atol=1e-7)
        grad_close(ins[r].grad, ref_dz[lo:hi])


def test_interleaved_with_other_exchanges_over_three_steps():
    """loss_calc(group=) between mpcl_loss_calc(group=) and cal_centroid(group=) on one mailbox, three steps: each call is
    one exchange (the epoch advances by 3 a step on every rank) and no result changes."""
    from slcl import seg
    from slcl import utils_ as U
    from slcl.loss import MPCL, mpcl_loss_calc
    world, sizes, k, c, h, w = 2, [2, 2], 4, 32, 16, 16
    gen = cases.g(7008)
    feat = torch.randn(sum(sizes), c, h, w, generator=gen).to(dev())
    cen = torch.randn(k, c, generator=gen).to(dev())
    z = (1.5 * torch.randn(sum(sizes), k, h, w, generator=gen)).to(dev())
    lab0 = torch.randint(0, k, (sum(sizes), h, w), generator=gen).to(dev())
    boxes = boxes_for(world)
    sp = spans(sizes)
    mods = [MPCL(dev(), num_class=k, temperature=.1, m=.4, base_temperature=1.0) for _ in range(world)]
    for step in range(3):
        lab = (lab0 + step) % k
        warm_seg([(z[lo:hi], lab[lo:hi]) for lo, hi in sp])
        want_c, _, _ = U.cal_centroid(feat, lab, n_class=k)
        fg, zg = feat.clone().requires_grad_(True), z.clone().requires_grad_(True)
        want_m = mpcl_loss_calc(fg, lab, cen, mods[0], tag='source')
        want_s = seg.loss_calc(zg, lab, 0, True)
        (want_m + want_s).backward()
        e0 = [bx.epoch() for bx in boxes]

        def rank(r, box):
            lo, hi = sp[r]
            f, zr = feat[lo:hi].clone().requires_grad_(True), z[lo:hi].clone().requires_grad_(True)
            c1, _, _ = U.cal_centroid(feat[lo:hi], lab[lo:hi], n_class=k, group=box)
            s1 = seg.loss_calc(zr, lab[lo:hi], 0, True, group=box)
            m1 = mpcl_loss_calc(f, lab[lo:hi], cen, mods[r], tag='source', group=box)
            (m1 + s1).backward()
            return c1, s1.detach(), m1.detach(), f.grad, zr.grad
        got = on_ranks(world, rank, boxes, spare_pass=(step == 0))
        assert all(bx.timeouts() == 0 for bx in boxes)
        assert [bx.epoch() for bx in boxes] == [e + 3 for e in e0]
        for r, (lo, hi) in enumerate(sp):
            assert torch.equal(got[r][1], got[0][1])
            close(got[r][0], want_c, rtol=1e-5, atol=1e-6)
            close(got[r][1], want_s, rtol=1e-5, atol=1e-7)
            close(got[r][2], want_m, rtol=1e-4, atol=1e-6)
            grad_close(got[r][4], zg.grad[lo:hi])
            grad_close(got[r][3], fg.grad[lo:hi], rtol=1e-4, floor=0.1)


def test_undersized_mailbox_raises_before_any_launch():
    from slcl import ops, seg
    k = 8
    need = 2 * ops.seg_vec_len(k)
    boxes = boxes_for(2, capacity_words=need - 2)
    z, lab = _case([2], k, 16, 16, 7009)
    torch.cuda.synchronize()
    before = boxes[0].buf.clone()
    with pytest.raises(ValueError, match="capacity_words"):
        seg.seg_losses(z, lab, group=boxes[0])
    with pytest.raises(ValueError, match="capacity_words"):
        ops.seg_fwd_peer(z, lab, *boxes[0].args())
    torch.cuda.synchronize()
    assert torch.equal(boxes[0].buf, before) and boxes[0].epoch() == 0
