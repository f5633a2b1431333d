"""cal_centroid(..., pseudo_label=True, from_logits=True): soft-label centroids straight from the segmentor's logits, the
softmax done inside the class-sum sweep and the centroid backward.

The reference is autograd through ``torch.softmax(z, 1)`` followed by the probability path of ``cal_centroid`` (itself
pinned to the oracle by test_gpu_parity.py), and at full size the oracle on the GPU.  Our softmax and torch's may differ in
the last bits, so the fixtures keep every decision away from its rounding edge: a pixel whose largest probability lies
within 1e-4 of the certainty threshold, or whose two largest logits lie within 1e-3, is redrawn.  With that, certainty
and arg-max decisions agree exactly and the arg-max weight columns (pixel counts) are compared bit for bit.
"""
import pytest
import torch

from oracle import slcl_oracle as O

pytestmark = pytest.mark.gpu

RTOL = 1e-4
THR = 0.5


def dev():
    return torch.device("cuda:0")


def close(a, b, rtol=RTOL, atol=1e-6):
    torch.testing.assert_close(torch.as_tensor(a).double().cpu(), torch.as_tensor(b).double().cpu(), rtol=rtol, atol=atol)


def grad_close(a, b, rtol=RTOL, floor=0.1):
    """rtol per element with an absolute floor of floor * rtol * max|b| (as test_gpu_parity.grad_close)."""
    b = torch.as_tensor(b).double()
    close(a, b, rtol=rtol, atol=rtol * (float(b.abs().max()) + 1e-30) * floor)


def logits(b, k, h, w, gen, scale=3.0):
    """scale * randn logits [B, K, H, W] with every pixel away from a decision edge (see the module docstring)."""
    z = scale * torch.randn(b, k, h, w, device=dev(), generator=gen)
    for _ in range(100):
        p = torch.softmax(z, 1)
        top = torch.topk(z, 2, dim=1).values
        bad = ((p.amax(1) - THR).abs() < 1e-4) | ((top[:, 0] - top[:, 1]) < 1e-3)
        n_bad = int(bad.sum())
        if n_bad == 0:
            return z
        fresh = scale * torch.randn(n_bad, k, device=dev(), generator=gen)
        zp = z.permute(0, 2, 3, 1)
        zp[bad] = fresh
        z = zp.permute(0, 3, 1, 2).contiguous()
    raise AssertionError("could not draw logits away from the decision edges")


def part_ids(n, parts, gen):
    return (torch.randperm(n, device=dev(), generator=gen) % parts).to(torch.int32) if parts > 1 else None


def _centroids(U, f, lab, k, parts, pid, prev, thr, weighted, from_logits, group=None):
    out, _, _ = U.cal_centroid(f, lab, previous_centroid=prev, momentum=0.9, pseudo_label=True, n_class=k, partition=parts,
                               threshold=thr, weighted_ave=weighted, part_id=pid, group=group, from_logits=from_logits)
    return torch.cat(out) if isinstance(out, list) else out


SHAPES = [(4, 32, 64, 64), (2, 128, 32, 32), (8, 32, 33, 33)]      # vec4 / TMA sweep, C = 128, scalar path (HW % 4 != 0)


@pytest.mark.parametrize("shape", SHAPES, ids=["vec4", "c128", "scalar"])
@pytest.mark.parametrize("parts", [1, 2])
@pytest.mark.parametrize("k", [2, 4, 5, 8])
def test_centroids_and_gradients_from_logits_equal_the_softmax_path(shape, parts, k):
    """Forward (centroids, class-sum weight column) and backward (dF, dlogits) of from_logits=True against autograd
    through torch.softmax + cal_centroid on the probabilities, with and without previous_centroid, threshold None / 0.5,
    weighted_ave True / False."""
    from slcl import utils_ as U
    op = torch.ops.slcl
    b, c, h, w = shape
    gen = torch.Generator(device=dev()).manual_seed(1000 * k + 10 * parts + c + h)
    feat = torch.randn(b, c, h, w, device=dev(), generator=gen)
    z = logits(b, k, h, w, gen)
    pid = part_ids(b * h * w, parts, gen)
    gcen = torch.randn(parts * k, c, device=dev(), generator=gen)
    prev_t = torch.randn(k, c, device=dev(), generator=gen)
    for with_prev in (False, True):
        prev = None if not with_prev else (prev_t if parts == 1 else [prev_t, 0.5 * prev_t])
        for thr in (None, THR):
            for weighted in (True, False):
                f1, z1 = feat.clone().requires_grad_(True), z.clone().requires_grad_(True)
                got = _centroids(U, f1, z1, k, parts, pid, prev, thr, weighted, True)
                (got * gcen).sum().backward()
                f2, z2 = feat.clone().requires_grad_(True), z.clone().requires_grad_(True)
                want = _centroids(U, f2, torch.softmax(z2, 1), k, parts, pid, prev, thr, weighted, False)
                (want * gcen).sum().backward()
                tag = (with_prev, thr, weighted)
                close(got, want)
                grad_close(f1.grad, f2.grad)
                if weighted:
                    grad_close(z1.grad, z2.grad)
                else:
                    assert z1.grad is None or float(z1.grad.abs().sum()) == 0.0
                t = 0.0 if thr is None else thr
                s1 = op.class_sums(feat, None, z, weighted, t, pid, parts, k, True)
                s2 = op.class_sums(feat, None, torch.softmax(z, 1), weighted, t, pid, parts, k)
                if weighted:
                    close(s1, s2, rtol=1e-5, atol=1e-4)
                else:
                    assert torch.equal(s1[:, -1], s2[:, -1]), tag            # pixel counts: bit-exact
                    close(s1[:, :-1], s2[:, :-1], rtol=1e-5, atol=1e-4)


def test_v2_sweep_from_logits(monkeypatch):
    """The register-tiled sweep (SLCL_CLASS_SUMS_V2=1) on a vec4 shape, next to the default TMA sweep."""
    op = torch.ops.slcl
    gen = torch.Generator(device=dev()).manual_seed(77)
    b, c, h, w, k, parts = 2, 48, 32, 32, 5, 2
    feat = torch.randn(b, c, h, w, device=dev(), generator=gen)
    z = logits(b, k, h, w, gen)
    pid = part_ids(b * h * w, parts, gen)
    for v2 in ("0", "1"):
        monkeypatch.setenv("SLCL_CLASS_SUMS_V2", v2)
        for weighted, thr in ((True, 0.0), (True, THR), (False, THR)):
            s1 = op.class_sums(feat, None, z, weighted, thr, pid, parts, k, True)
            s2 = op.class_sums(feat, None, torch.softmax(z, 1), weighted, thr, pid, parts, k)
            close(s1, s2, rtol=1e-5, atol=1e-4)
            if not weighted:
                assert torch.equal(s1[:, -1], s2[:, -1])


@pytest.fixture()
def no_tf32():
    old = (torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32)
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    yield
    torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = old


def test_full_size_cfg5_from_logits_vs_oracle(no_tf32):
    """configs[4] per GPU (64 x 32 x 224 x 224, K = 4, P = 2, threshold 0.5, weighted): centroids, dF and dlogits against
    the oracle on softmax(logits), evaluated on the GPU in fp32; the arg-max pixel counts per partition are exact."""
    from slcl import utils_ as U
    gen = torch.Generator(device=dev()).manual_seed(505)
    b, c, h, w, k, parts = 64, 32, 224, 224, 4, 2
    feas = torch.randn(b, c, h, w, device=dev(), generator=gen)
    z = logits(b, k, h, w, gen)
    part = part_ids(b * h * w, parts, gen)
    gcen = torch.randn(parts * k, c, device=dev(), generator=gen)
    fo, zo = feas.clone().requires_grad_(True), z.clone().requires_grad_(True)
    ref, _, _ = O.cal_centroid(fo, torch.softmax(zo, 1), pseudo_label=True, weighted_ave=True, partition=parts, n_class=k,
                               threshold=THR, part_id=part)
    (torch.cat(ref) * gcen).sum().backward()
    f, zz = feas.clone().requires_grad_(True), z.clone().requires_grad_(True)
    out, _, _ = U.cal_centroid(f, zz, pseudo_label=True, weighted_ave=True, partition=parts, n_class=k, threshold=THR,
                               part_id=part, from_logits=True)
    (torch.cat(out) * gcen).sum().backward()
    close(torch.cat(out), torch.cat(ref).detach())
    grad_close(f.grad, fo.grad)
    grad_close(zz.grad, zo.grad)
    del fo, zo, ref
    sums = torch.ops.slcl.class_sums(feas, None, z, False, THR, part, parts, k, True)
    p = torch.softmax(z, 1)
    cert = (p.amax(1).reshape(-1) >= THR).long()
    want = torch.bincount(part.long() * k + p.argmax(1).reshape(-1), weights=cert.double(), minlength=parts * k)
    assert torch.equal(sums[:, -1], want)


def _mccl_section(feats, lab_s, target_inputs, parts, k, from_logits, pids):
    """Trainer_MCCL's loss section from the decoder outputs: hard source centroids, P-partition centroids of the target
    view and centroids of the augmented view from their soft labels, every centroid term through mccl_centroid_losses."""
    from slcl.loss import mccl_centroid_losses
    from slcl.utils_ import cal_centroid
    cs, _, _ = cal_centroid(feats[0], lab_s, n_class=k)
    soft = [t if from_logits else torch.softmax(t, 1) for t in target_inputs]
    ct, _, _ = cal_centroid(feats[1], soft[0], pseudo_label=True, weighted_ave=True, partition=parts, n_class=k, threshold=THR,
                            part_id=pids[0], from_logits=from_logits)
    ca, _, _ = cal_centroid(feats[2], soft[1], pseudo_label=True, weighted_ave=True, n_class=k, threshold=THR,
                            from_logits=from_logits)
    total, _ = mccl_centroid_losses(cs, ct, ca, inter_w=1.0, intra_w=1.0, cnr_w=4e-5)
    return total


def _section_inputs(b=4, c=32, h=64, k=4, parts=2, seed=91):
    gen = torch.Generator(device=dev()).manual_seed(seed)
    feats = [torch.randn(b, c, h, h, device=dev(), generator=gen) for _ in range(3)]
    lab_s = torch.randint(0, k, (b, h, h), device=dev(), generator=gen)
    zs = [logits(b, k, h, h, gen) for _ in range(2)]
    pids = [part_ids(b * h * h, parts, gen)]
    return feats, lab_s, zs, pids


def test_mccl_section_from_logits_equals_softmax_section():
    """The loss and the gradients into the three feature maps and both logit maps."""
    k, parts = 4, 2
    feats, lab_s, zs, pids = _section_inputs(k=k, parts=parts)
    res = []
    for from_logits in (True, False):
        f = [t.clone().requires_grad_(True) for t in feats]
        z = [t.clone().requires_grad_(True) for t in zs]
        loss = _mccl_section(f, lab_s, z, parts, k, from_logits, pids)
        loss.backward()
        res.append((loss.detach(), [t.grad for t in f], [t.grad for t in z]))
    (l1, df1, dz1), (l2, df2, dz2) = res
    close(l1, l2, rtol=1e-5)
    for a, b in zip(df1 + dz1, df2 + dz2):
        grad_close(a, b)


def test_no_host_sync_and_cuda_graph_replay():
    k, parts = 4, 2
    feats, lab_s, zs, pids = _section_inputs(k=k, parts=parts, seed=92)

    def leaves():
        return [t.clone().requires_grad_(True) for t in feats], [t.clone().requires_grad_(True) for t in zs]

    f, z = leaves()
    eager = _mccl_section(f, lab_s, z, parts, k, True, pids)
    eager.backward()
    torch.cuda.synchronize()
    f2, z2 = leaves()
    torch.cuda.set_sync_debug_mode("error")
    try:
        loss = _mccl_section(f2, lab_s, z2, parts, k, True, pids)
        loss.backward()
    finally:
        torch.cuda.set_sync_debug_mode(0)
    torch.cuda.synchronize()
    close(loss, eager, rtol=1e-6, atol=0.0)

    # the whole section (forward + autograd backward) in one CUDA graph; fresh leaves so that their AccumulateGrad nodes
    # are born on the capture stream
    gf, gz = leaves()

    def step():
        out = _mccl_section(gf, lab_s, gz, parts, k, True, pids)
        out.backward()
        return out.detach()
    side = torch.cuda.Stream(dev())
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        step()
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    for t in gf + gz:
        t.grad = None
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        static_loss = step()
    for _ in range(2):
        graph.replay()
    torch.cuda.synchronize()
    close(static_loss, eager, rtol=1e-6, atol=0.0)
    for a, b in zip(gf + gz, f + z):
        grad_close(a.grad, b.grad, rtol=1e-6)


# ---------------------------------------------------------------------------
# over the global batch: ranks are CUDA streams of one GPU exchanging through loopback mailboxes
# (slcl.peer.LoopbackMailboxes), as in test_gpu_parity.test_sharded_class_centres_and_centroids_equal_global
# ---------------------------------------------------------------------------
def _on_streams(streams, fn):
    """fn(rank) enqueued on streams[rank] for every rank, nothing synchronises in between; returns the results."""
    cur = torch.cuda.current_stream()
    out = []
    for r, st in enumerate(streams):
        st.wait_stream(cur)
        with torch.cuda.stream(st):
            out.append(fn(r))
    for st in streams:
        cur.wait_stream(st)
    return out


@pytest.mark.parametrize("world", [2, 4])
def test_sharded_from_logits_equals_the_global_batch(world):
    from slcl import utils_ as U
    from slcl.peer import LoopbackMailboxes
    op = torch.ops.slcl
    b, c, h, w, k, parts = 2 * world, 32, 24, 20, 4, 2
    gen = torch.Generator(device=dev()).manual_seed(31 + world)
    feat = torch.randn(b, c, h, w, device=dev(), generator=gen)
    z = logits(b, k, h, w, gen)
    part = part_ids(b * h * w, parts, gen)
    gcen = torch.randn(parts * k, c, device=dev(), generator=gen)
    per = b // world
    sl = lambda t, r: t[r * per:(r + 1) * per]
    pix = lambda t, r: t.reshape(b, -1)[r * per:(r + 1) * per].reshape(-1)

    # the global batch on one rank; loads every kernel the ranks launch before any of them polls a mailbox
    fg, zg = feat.clone().requires_grad_(True), z.clone().requires_grad_(True)
    cen_g = _centroids(U, fg, zg, k, parts, part, None, THR, True, True)
    (cen_g * gcen).sum().backward()
    sums_g = op.class_sums(feat, None, z, False, THR, part, parts, k, True)

    def warm(r):
        f = sl(feat, r).clone().requires_grad_(True)
        zz = sl(z, r).clone().requires_grad_(True)
        (_centroids(U, f, zz, k, parts, pix(part, r), None, THR, True, True) * gcen).sum().backward()
        op.centroids_fwd(sl(feat, r), None, sl(z, r), False, THR, pix(part, r), parts, k, None, 0.9, from_logits=True)
    streams = [torch.cuda.Stream(dev()) for _ in range(world)]
    _on_streams(streams, warm)
    torch.cuda.synchronize()

    boxes = LoopbackMailboxes(world, dev(), timeout_s=20.0).boxes
    res = {}

    def rank_fn(r):
        f = sl(feat, r).clone().requires_grad_(True)
        zz = sl(z, r).clone().requires_grad_(True)
        cen = _centroids(U, f, zz, k, parts, pix(part, r), None, THR, True, True, group=boxes[r])
        (cen * gcen).sum().backward()
        _, _, sums = op.centroids_fwd(sl(feat, r), None, sl(z, r), False, THR, pix(part, r), parts, k, None, 0.9,
                                      *boxes[r].args(), from_logits=True)
        res[r] = (cen.detach(), f.grad, zz.grad, sums)
    _on_streams(streams, rank_fn)
    torch.cuda.synchronize()
    assert all(bx.timeouts() == 0 for bx in boxes)
    for r in range(world):
        cen, df, dz, sums = res[r]
        assert torch.equal(sums[:, -1], sums_g[:, -1])                   # arg-max x certainty pixel counts: GLOBAL, exact
        close(cen, cen_g.detach(), rtol=1e-5)
        grad_close(df, sl(fg.grad, r), rtol=1e-5)
        grad_close(dz, sl(zg.grad, r), rtol=1e-5)
        assert torch.equal(cen, res[0][0])                                 # identical bits on every rank

    # the NCCL route's kernels: per-rank class sums from logits, summed here in rank order, finalised, and the backward
    # of each shard against the global sums
    sums_w_g = op.class_sums(feat, None, z, True, THR, part, parts, k, True)
    loc = [op.class_sums(sl(feat, r), None, sl(z, r), True, THR, pix(part, r), parts, k, True) for r in range(world)]
    tot = loc[0]
    for s in loc[1:]:
        tot = tot + s
    close(tot, sums_w_g, rtol=1e-6, atol=1e-6)
    cen_n, _ = op.centroid_finalize(tot, None, 0.9, parts, k)
    close(cen_n, cen_g.detach(), rtol=1e-5)
    for r in range(world):
        df, dz = op.centroid_bwd(sl(feat, r), None, sl(z, r), True, THR, pix(part, r), parts, k, gcen, tot, 1.0, True, True)
        grad_close(df, sl(fg.grad, r), rtol=1e-5)
        grad_close(dz, sl(zg.grad, r), rtol=1e-5)
