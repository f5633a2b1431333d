"""BlockConLoss over the global batch of data-parallel ranks (``BlockConLoss(group=)``).

Ranks are CUDA streams of one GPU exchanging through loopback mailboxes, with the harness of tests/test_p2p_global.py.
The reference is ``BlockConLoss`` on ONE rank over the ranks' batches concatenated: every tile's problem is the union of
that tile's rows on all ranks.  (The file name sorts after test_p2p_global.py on purpose: ranks as streams of one GPU
depend on the CUDA streams and cached index tensors the process already holds, so these tests run after that file's
and leave its cases the process history they were written against.)
"""
import threading

import pytest
import torch
import torch.nn.functional as F

import test_p2p_global as base
from oracle import cases
from oracle import slcl_oracle as O
from test_p2p_global import boxes_for, close, dev, grad_close, on_ranks, shard

pytestmark = pytest.mark.gpu

T = 0.7
BS = 32


@pytest.fixture
def no_tf32():
    old = (torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32)
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    yield
    torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = old


def _case(world, seed, hw=64, c=32, b_l=1):
    """Per rank (b_l, 2, c, hw, hw), unit feature vectors, labels in [0, 4)."""
    g = cases.g(seed)
    feat = F.normalize(torch.randn(b_l * world, 2, c, hw, hw, generator=g), dim=2)
    lab = torch.randint(0, 4, (b_l * world, 2, hw, hw), generator=g)
    return feat.to(dev()), lab.to(dev())


def _rows_bytes(feat_rank, bs=BS):
    from slcl.p2p import global_record_bytes
    b, v, c, h, w = feat_rank.shape
    div = w // bs
    m = b * v * div * div * bs * bs
    return global_record_bytes(m, m, c, same_rows=True, n_batch=div * div)


def _unsharded(feat, lab, n_class=None):
    from slcl.p2p import BlockConLoss
    f = feat.clone().requires_grad_(True)
    out = BlockConLoss(T, BS, n_class=n_class)(f, lab)
    out.backward()
    return out.detach(), f.grad


def _sharded(feat, lab, world, n_class=None, boxes=None):
    """Every rank's (loss, gradient of its shard, module)."""
    from slcl.p2p import BlockConLoss
    rb = _rows_bytes(shard(feat, world, 0))
    boxes = boxes if boxes is not None else boxes_for(world, rb)

    def rank(r, box):
        mod = BlockConLoss(T, BS, n_class=n_class, group=box)
        f = shard(feat, world, r).clone().requires_grad_(True)
        out = mod(f, None if lab is None else shard(lab, world, r))
        out.backward()
        return out.detach(), f.grad, mod
    got = on_ranks(world, rank, boxes, rb)
    assert all(bx.timeouts() == 0 and bx.mismatches() == 0 for bx in boxes)
    return got


def _check(got, ref, world, rtol=1e-5):
    for r in range(world):
        assert torch.equal(got[r][0], got[0][0])                          # identical bits on every rank
        close(got[r][0], ref[0], rtol=rtol, atol=1e-7)
        grad_close(got[r][1], shard(ref[1], world, r), rtol=1e-4)


@pytest.mark.parametrize("world", [2, 4])
@pytest.mark.parametrize("mode", ["stock", "general", "unlabelled"])
def test_blockcon_global_equals_unsharded(world, mode):
    """Stock signature (class-index labels -> analytic sweeps), n_class = 0 (general sweeps) and labels=None."""
    feat, lab = _case(world, 610 + world)
    lab = None if mode == "unlabelled" else lab
    n_class = 0 if mode == "general" else None
    ref = _unsharded(feat, lab, n_class)
    got = _sharded(feat, lab, world, n_class)
    if mode == "stock":
        assert all(g_[2].supconloss._classes.auto == 8 for g_ in got)       # label range reduced over the ranks
    _check(got, ref, world)
    if world == 2 and mode == "stock":          # and the oracle on the union (bf16 GEMM inputs: 2e-2)
        close(got[0][0], O.block_con_loss(feat.cpu(), lab.cpu(), T, BS), rtol=2e-2)


def test_blockcon_global_foreground_skew():
    """Tile (0, 0) has foreground on rank 0 only, tile (1, 1) on no rank: the first counts with rank 0's rows as its only
    weighted anchors, the second is skipped; both decided over the union."""
    world = 2
    feat, lab = _case(world, 631)
    lab[1:, :, :BS, :BS] = 0
    lab[:1, :, :BS, :BS] = torch.randint(1, 4, (1, 2, BS, BS), generator=cases.g(632)).to(dev())
    lab[:, :, BS:, BS:] = 0
    ref = _unsharded(feat, lab)
    _check(_sharded(feat, lab, world), ref, world)
    ref0 = _unsharded(feat, lab, n_class=0)
    _check(_sharded(feat, lab, world, n_class=0), ref0, world)


def test_blockcon_global_without_foreground_on_any_rank_is_zero():
    world = 2
    feat, lab = _case(world, 641)
    lab = torch.zeros_like(lab)
    ref = _unsharded(feat, lab)
    assert float(ref[0]) == 0.0 and not bool(ref[1].any())
    for r_loss, r_grad, _ in _sharded(feat, lab, world):
        assert float(r_loss) == 0.0
        assert not bool(r_grad.any())


def _oracle_fp32(feat, lab):
    """O.block_con_loss on the GPU in fp32 (loss and gradient), one tile's graph at a time: the mean over the tiles with
    foreground, as utils/loss.py:430-466."""
    div = feat.shape[-1] // BS
    f = feat.clone().requires_grad_(True)
    tiles = [(slice(i * BS, (i + 1) * BS), slice(j * BS, (j + 1) * BS)) for i in range(div) for j in range(div)]
    kept = [(sh, sw) for sh, sw in tiles if int(lab[:, :, sh, sw].sum()) != 0]
    total = torch.zeros((), dtype=torch.float64, device=feat.device)
    for sh, sw in kept:
        part = O.supcon_loss(f[:, :, :, sh, sw], lab[:, :, sh, sw], T) / len(kept)
        part.backward()
        total += part.detach().double()
    return total, f.grad


def test_blockcon_global_beyond_the_old_anchor_bound(no_tf32):
    """World 4 at the reference's per-rank shape (1, 2, 32, 224, 224): 49 tiles, 401 408 global anchors (the sweeps
    refused more than 262 143 before).  The unsharded (4, 2, 32, 224, 224) call is itself checked against the fp32
    oracle on the GPU."""
    world = 4
    feat, lab = _case(world, 651, hw=224)
    ref = _unsharded(feat, lab)
    want, want_grad = _oracle_fp32(feat, lab)
    close(ref[0], want, rtol=2e-2)
    base.grad_close(ref[1], want_grad, rtol=2e-2, floor=0.5)
    _check(_sharded(feat, lab, world), ref, world)


@pytest.mark.parametrize("shape,bs,batched", [((1, 2, 16, 36, 36), 12, True), ((1, 2, 32, 64, 64), 32, False)])
def test_blockcon_global_refuses_per_tile_loop_shapes(shape, bs, batched):
    """288 rows per tile (not whole 128-row tiles), or batched = False: ValueError on every rank, before any exchange
    (not even the label-range exchange of a module without n_class)."""
    from slcl.p2p import BlockConLoss
    world = 2
    boxes = boxes_for(world, 1 << 20)
    epochs = [bx.epoch() for bx in boxes]
    feat = torch.randn((shape[0] * world,) + shape[1:], device=dev())
    lab = torch.randint(0, 4, (shape[0] * world, shape[1]) + shape[3:], device=dev())
    for r, box in enumerate(boxes):
        mod = BlockConLoss(T, bs)
        mod.batched = batched
        with pytest.raises(ValueError):
            mod(shard(feat, world, r), shard(lab, world, r), group=box)
    torch.cuda.synchronize()
    assert [bx.epoch() for bx in boxes] == epochs


def test_blockcon_global_second_call_has_no_host_sync():
    """With a fixed n_class nothing in forward or backward waits for the host: the call is capturable and overlaps."""
    from slcl.p2p import BlockConLoss
    world = 2
    feat, lab = _case(world, 661)
    rb = _rows_bytes(shard(feat, world, 0))
    boxes = boxes_for(world, rb)
    mods = [BlockConLoss(T, BS, n_class=4) for r in range(world)]
    ins = [(shard(feat, world, r).clone().requires_grad_(True), shard(lab, world, r)) for r in range(world)]

    def first(r, box):
        mods[r](*ins[r], group=box).backward()
    on_ranks(world, first, boxes, rb)
    for f, _ in ins:
        f.grad = None
    ready, done = threading.Barrier(world), threading.Barrier(world)

    def second(r):
        ready.wait()
        if r == 0:
            torch.cuda.set_sync_debug_mode("error")
        ready.wait()
        try:
            out = mods[r](*ins[r], group=boxes[r])
            out.backward()
        finally:
            done.wait()
            if r == 0:
                torch.cuda.set_sync_debug_mode("default")
        return out.detach()
    got = base._threads(world, second)
    ref = _unsharded(feat, lab, n_class=4)
    assert all(bx.timeouts() == 0 and bx.mismatches() == 0 for bx in boxes)
    for r in range(world):
        close(got[r], ref[0], rtol=1e-5, atol=1e-7)
        grad_close(ins[r][0].grad, shard(ref[1], world, r))


def test_blockcon_global_interleaved_with_other_exchanges_then_more_steps():
    """BlockConLoss(group=) between SupConLoss(group=) and a scalar cal_centroid(group=) on one mailbox, three steps with
    the same modules: the shared epoch sequence neither stalls an exchange nor changes a result."""
    from slcl import utils_ as U
    from slcl.p2p import BlockConLoss, SupConLoss, global_record_bytes
    world, k = 2, 4
    feat, lab = _case(world, 671)
    b, v, c, h, w = feat.shape
    m_sup = (b // world) * v * h * w
    rows = max(_rows_bytes(shard(feat, world, 0)), global_record_bytes(m_sup, m_sup, c, same_rows=True))
    boxes = boxes_for(world, rows)
    mods = {}
    for step in range(3):
        fs = F.normalize(feat + 0.1 * step, dim=2)
        ls = (lab + step) % k
        f4, l4 = fs.reshape(b * v, c, h, w), ls.reshape(b * v, h, w)
        want_c, _, _ = U.cal_centroid(f4, l4, n_class=k)
        fg = fs.clone().requires_grad_(True)
        l1 = SupConLoss(temperature=T)(fg, ls)
        l2 = BlockConLoss(T, BS)(fg, ls)
        (l1 + 2 * l2).backward()

        def rank(r, box):         # the same module objects on every step of a rank
            sup, blk = mods.setdefault(id(box), (SupConLoss(temperature=T, group=box), BlockConLoss(T, BS, group=box)))
            f = shard(fs, world, r).clone().requires_grad_(True)
            lr = shard(ls, world, r)
            c1, _, _ = U.cal_centroid(shard(f4, world, r), shard(l4, world, r), n_class=k, group=box)
            x1 = sup(f, lr)
            c2, _, _ = U.cal_centroid(shard(f4, world, r), shard(l4, world, r), n_class=k, group=box)
            x2 = blk(f, lr)
            c3, _, _ = U.cal_centroid(shard(f4, world, r), shard(l4, world, r), n_class=k, group=box)
            (x1 + 2 * x2).backward()
            return x1.detach(), x2.detach(), f.grad, (c1, c2, c3)
        got = on_ranks(world, rank, boxes, rows if step == 0 else None)
        assert all(bx.timeouts() == 0 and bx.mismatches() == 0 for bx in boxes)
        for r in range(world):
            assert torch.equal(got[r][1], got[0][1])
            close(got[r][0], l1, rtol=1e-5, atol=1e-7)
            close(got[r][1], l2, rtol=1e-5, atol=1e-7)
            grad_close(got[r][2], shard(fg.grad, world, r))
            for cc in got[r][3]:
                close(cc, want_c, rtol=1e-5, atol=1e-6)
