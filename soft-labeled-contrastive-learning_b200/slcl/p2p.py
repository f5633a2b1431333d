"""Pixel <-> pixel supervised contrastive losses on the tensor-core path.

Drop-ins for the reference's ``SupConLoss`` / ``LocalConLoss`` / ``BlockConLoss``
(utils/loss.py:315-466, duplicated at utils/losses.py:95-239) plus the sampled
rectangular variant of SURVEY.md 8(c)-3 (``sampled_supcon_loss``).  Rows are
gathered from the NCHW map into bf16 K-major rows, similarities run as
tcgen05 GEMMs with fp32 accumulation and a fused soft-max epilogue; the M x M
matrix of the reference (:342-349) is never materialised.
"""
from __future__ import annotations

from typing import Optional

import torch
import torch.nn as nn

from . import ops  # noqa: F401

_ops = ops.dispatch          # eager: op bodies directly; compiled: torch.ops.slcl
_SORT_MIN_ROWS = 8192        # one-row-set problems at least this large are gathered sorted by label (see p2p_loss)
AUTO_N_CLASS = 8             # labelled SupCon family without an explicit n_class: analytic sweeps for labels in [0, 8)


class _AutoClasses:
    """Lets the STOCK signatures (``SupConLoss()``, ``LocalConLoss()``: no ``n_class`` argument) reach the analytic
    tensor-core sweeps.  Those need class-index labels in [0, n_class), n_class <= 8 -- true for every label map of the
    reference (4 or 5 classes, config.py:9) but not guaranteed by the signature.  The first labelled call of a module
    checks the range once on the host (one synchronisation in the module's lifetime).  Should a label leave the range
    in a later call the loss comes out NaN, never silently wrong, and at no cost: in these losses every row is an
    anchor, an anchor whose label is outside [0, n_class) has no class table, so the finishing kernel sees n_i = 0
    positives and its row loss is 0/0 -- which the weighted sum carries to the result whatever the row's weight.
    ``n_class=0`` in the constructor forces the general sweeps (any integer labels), ``n_class=k`` trusts the caller."""

    def __init__(self, n_class):
        self.fixed = n_class            # None = auto
        self.auto = None                # decided at the first labelled call

    def resolve(self, labels, exchange=None):
        """-> (n_class for the sweeps, device flag `labels in range` or None -- None since the kernels' own NaN covers it).
        With an ``exchange`` (``group=``) the range is reduced over the ranks, so every rank takes the same sweeps."""
        if self.fixed is not None:
            return int(self.fixed), None
        if labels is None:
            return 0, None
        if self.auto is None:
            if exchange is None:
                lo, hi = int(labels.min()), int(labels.max())        # once per module
            else:
                lo, hi = exchange.label_range(labels)
            self.auto = AUTO_N_CLASS if (lo >= 0 and hi < AUTO_N_CLASS) else 0
        if self.auto == 0:
            return 0, None
        return self.auto, None


def _guard(loss, in_range):
    return loss if in_range is None else torch.where(in_range, loss, torch.full_like(loss, float("nan")))



class _P2PLoss(torch.autograd.Function):
    """loss(feat) for anchor rows idx_a and contrast rows idx_b of an NCHW map (appendix A.6).

    ``n_class`` > 0 selects the analytic sweeps (include/slcl.h): labels are class indices in [0, n_class), ids
    unique; the forward then also produces U and the per-class row sums, and the backward is one sweep."""

    @staticmethod
    def forward(ctx, feat, idx_a, idx_b, meta_a, meta_b, weight, temperature, normalize, same_rows, n_class, selfcol,
                selfrow, n_batch, rowmaps):
        fm = feat.detach().contiguous()
        c = fm.shape[1]
        b_bf16, _, inv_b = _ops.gather_unit_rows(fm, idx_b, normalize, True, False)
        if same_rows:
            a_bf16, inv_a = b_bf16, inv_b
        else:
            a_bf16, _, inv_a = _ops.gather_unit_rows(fm, idx_a, normalize, True, False)
        if normalize:
            shift = torch.full_like(inv_a, 1.0 / temperature)
        else:   # upper bound of S_ij: |a_i| max_j |b_j| / T
            shift = _ops.p2p_shift(inv_a, inv_b, temperature)
        keep = n_class > 0 and ctx.needs_input_grad[0]
        loss, stats, state = _ops.p2p_fwd(a_bf16, b_bf16, meta_a, meta_b, shift, weight, temperature, n_class, selfcol, keep,
                                          n_batch)
        ctx.save_for_backward(fm, idx_a, idx_b, meta_a, meta_b, weight, a_bf16, b_bf16, inv_a, inv_b, shift, stats, state,
                              selfcol, selfrow, rowmaps)
        ctx.cfg = (temperature, normalize, same_rows, c, n_class, n_batch)
        return loss[0]

    @staticmethod
    def backward(ctx, grad_out):
        (fm, idx_a, idx_b, meta_a, meta_b, weight, a_bf16, b_bf16, inv_a, inv_b, shift, stats, state, selfcol,
         selfrow, rowmaps) = ctx.saved_tensors
        temperature, normalize, same_rows, c, n_class, n_batch = ctx.cfg
        if not ctx.needs_input_grad[0]:
            return (None,) * 14
        d_a, d_b = _ops.p2p_bwd(a_bf16, b_bf16, c, meta_a, meta_b, shift, weight, temperature, stats,
                                grad_out.reshape(1), True, True, n_class, selfcol, selfrow, state, n_batch)
        if rowmaps is not None and not same_rows:
            # pixel -> row maps at hand and the rows cover a good share of the map: write the whole gradient map from the
            # pixel side (coalesced, no atomics, no zero-fill) instead of scattering 4-byte elements
            dfeat = _ops.scatter_rows_by_map(fm, normalize, rowmaps[0], d_a.contiguous(), inv_a, rowmaps[1], d_b.contiguous(), inv_b)
            return (dfeat,) + (None,) * 13
        dfeat = torch.zeros_like(fm)
        if same_rows:       # anchors and contrast rows are the same gathered rows: one scatter of the summed row gradients
            _ops.scatter_rows_bwd(fm, idx_b, normalize, d_a + d_b, inv_b, dfeat)
        else:
            _ops.scatter_rows_bwd(fm, idx_a, normalize, d_a, inv_a, dfeat)
            _ops.scatter_rows_bwd(fm, idx_b, normalize, d_b, inv_b, dfeat)
        return (dfeat,) + (None,) * 13


_INT_MIN = -2 ** 31


class _Exchange:
    """The ``group=`` argument of the pixel <-> pixel losses: all-gather of byte records over NVLink peer memory
    (``slcl.peer.PeerMailbox`` built with ``rows_bytes``; ``slcl_peer_allgather``) or NCCL (``True`` / a ProcessGroup)."""

    def __init__(self, group):
        from .peer import PeerMailbox
        if isinstance(group, PeerMailbox):
            self.box, self.pg = group, None
            self.world, self.rank = group.world, group.rank
        else:
            import torch.distributed as dist
            self.box, self.pg = None, (None if group is True else group)
            self.world, self.rank = dist.get_world_size(self.pg), dist.get_rank(self.pg)

    def allgather(self, record, status):
        """uint8 record [n] -> [world, n] in rank order.  ``status`` (int32 [1]) turns non-zero when a peer timed out or
        sent a record whose 16-byte key differs (peer route: the caller's result is then NaN)."""
        if self.box is not None:
            return _ops.peer_allgather(record, status, *self.box.args(), *self.box.rows_args())
        import torch.distributed as dist
        # NCCL cannot gather records of different sizes: compare the keys first and refuse on the host
        keys = torch.empty((self.world, 16), dtype=torch.uint8, device=record.device)
        dist.all_gather_into_tensor(keys, record[:16].contiguous(), group=self.pg)
        if not bool((keys == record[:16]).all()):
            raise ValueError("group= pixel<->pixel loss: the ranks passed row sets of different sizes")
        out = torch.empty((self.world, record.numel()), dtype=torch.uint8, device=record.device)
        dist.all_gather_into_tensor(out, record, group=self.pg)
        return out

    def label_range(self, labels):
        """(min, max) of the labels over all ranks: one exchange and one host synchronisation."""
        lohi = torch.stack([labels.min(), -labels.max()]).long()
        rec, _ = _pack([_key(labels.device, 0, 0, 0, 3), lohi])
        status = torch.zeros(1, dtype=torch.int32, device=labels.device)
        got = self.allgather(rec, status)[:, 16:32].contiguous().view(torch.int64)
        if int(status[0]) != 0:
            raise RuntimeError("group= pixel<->pixel loss: the label-range exchange failed (peer timed out or shapes differ)")
        lo, nhi = got.amin(0).tolist()
        return lo, -nhi


def _exchange(group):
    """None (today's single-rank path) for no group or a world of one."""
    if group is None:
        return None
    x = _Exchange(group)
    return x if x.world > 1 else None


def _key(dev, a, m, dp, flags):
    """16-byte record key (int32 {A, M, dp, flags}): equal on every rank iff the records have the same layout."""
    def build():          # filled on the device: a host copy would synchronise the stream in the middle of the exchanges
        k = torch.zeros(4, dtype=torch.int32, device=dev)
        for i, v in enumerate((a, m, dp, flags)):
            k[i] = v
        return k
    return _cached(("key", a, m, dp, flags, str(dev)), build)


def _pack(parts):
    """tensors -> (uint8 record, layout); every part starts on a 16-byte boundary."""
    chunks, layout, off = [], [], 0
    for t in parts:
        b = t.contiguous().view(-1).view(torch.uint8)
        n = b.numel()
        chunks.append(b)
        if n % 16:
            chunks.append(b.new_zeros(16 - n % 16))
        layout.append((off, n, t.dtype, tuple(t.shape)))
        off += n + (-n) % 16
    return torch.cat(chunks), layout


def _unpack(gathered, layout, i, n_batch=1):
    """Part i of every rank's record, concatenated along the first dimension (a private copy): in rank order, or, for a
    part whose rows fall into ``n_batch`` equal block-diagonal batches, batch-major -- [batch][rank][rows of the batch] --
    so that every batch's rows of all ranks are contiguous.  The reordering is a strided view in front of the one copy."""
    off, n, dtype, shape = layout[i]
    part = gathered[:, off:off + n]
    if n_batch > 1:
        part = part.view(gathered.shape[0], n_batch, n // n_batch).transpose(0, 1)
    return part.contiguous().view(dtype).reshape((-1,) + shape[1:])


def _pad_meta_rows(meta):
    out = torch.full(((meta.shape[0] + 63) // 64 * 64, 2), _INT_MIN, dtype=torch.int32, device=meta.device)
    out[:meta.shape[0]] = meta
    return out


def global_record_bytes(n_anchor: int, n_contrast: int, channels: int, same_rows: bool = False, n_batch: int = 1) -> int:
    """Send-slot size (``rows_bytes`` of ``PeerMailbox`` / ``LoopbackMailboxes``) that a ``group=`` pixel <-> pixel loss with
    this many anchors / contrast rows per rank and ``channels`` feature channels needs.  ``n_batch``: block-diagonal
    batches (``BlockConLoss``: div^2 tiles), each of which carries its own table of per-class sums."""
    p16 = lambda n: (n + 15) // 16 * 16
    dp = (channels + 63) // 64 * 64
    rows = lambda r: r * dp * 2 + p16(r * 8) + p16(r * 4)
    first = 16 + 16 + rows(n_contrast) + (0 if same_rows else rows(n_anchor))
    second = 16 + 16 + max(3 * p16(n_anchor * 4) + p16(n_batch * AUTO_N_CLASS * (dp + 1) * 4), p16(n_anchor * 12))
    return max(first, second)


def _global_self_maps(selfcol, selfrow, na, m, world, rank, n_batch):
    """The local self maps carried into the global row index spaces, whose order is [batch][rank][row of the batch]
    (rank-major for n_batch = 1): -> (local anchors -> global contrast rows [na], global contrast rows -> local anchors
    [m world], global anchors -> local contrast rows [na world], local contrast rows -> global anchors [m]); -1 = no self
    pair (a self pair never crosses ranks)."""
    ra, rb = na // n_batch, m // n_batch

    def to_global(i, rows):          # local (batch t, row k) -> global t world rows + rank rows + k
        i = i.long()
        return torch.where(i >= 0, (i // rows) * (world * rows) + rank * rows + i % rows, i).to(torch.int32)

    selfrow_g = torch.full((n_batch, world, rb), -1, dtype=torch.int32, device=selfcol.device)
    selfrow_g[:, rank] = selfrow.view(n_batch, rb)
    a_selfcol_g = torch.full((n_batch, world, ra), -1, dtype=torch.int32, device=selfcol.device)
    a_selfcol_g[:, rank] = selfcol.view(n_batch, ra)
    return to_global(selfcol, rb), selfrow_g.view(-1), a_selfcol_g.view(-1), to_global(selfrow, ra)


class _P2PGlobal(torch.autograd.Function):
    """loss(feat) of the pixel <-> pixel problem over the GLOBAL batch of ``x.world`` ranks (INTEGRATION.md section 4).

    Anchors and contrast rows are the union of every rank's rows in rank order; ``meta_*`` carry ids that are unique across
    ranks.  With ``n_batch`` > 1 block-diagonal batches (BlockConLoss's tiles) each rank's rows are batch-major, and the
    union is ordered [batch][rank][row of the batch]: batch z of the global problem is batch z of every rank.
    Forward: all-gather {rows, meta, norms, short flag} -> weights / shifts of the global problem -> this rank's
    anchors x all contrast rows (slcl_p2p_fwd) -> all-gather {loss partial, per-anchor backward constants}.  Backward, no
    exchange: d_a = this rank's anchors x all contrast rows, d_b = all anchors x this rank's contrast rows (slcl_p2p_bwd with
    a state assembled from the gathered constants), so this rank gets exactly its shard of the global gradient."""

    @staticmethod
    def forward(ctx, feat, idx_a, idx_b, meta_a, meta_b, short, temperature, normalize, same_rows, n_class, selfcol, selfrow,
                uniform_weight, zero_if_empty, x, rowmaps, n_batch, maps_key):
        fm = feat.detach().contiguous()
        c = fm.shape[1]
        dev = fm.device
        W, r, T = x.world, x.rank, n_batch
        b_l, _, inv_b = _ops.gather_unit_rows(fm, idx_b, normalize, True, False)
        if same_rows:
            a_l, inv_a = b_l, inv_b
        else:
            a_l, _, inv_a = _ops.gather_unit_rows(fm, idx_a, normalize, True, False)
        na, m, dp = a_l.shape[0], b_l.shape[0], b_l.shape[1]
        flags = int(same_rows) | int(normalize) << 1 | n_class << 2 | (T - 1) << 6
        parts = [_key(dev, na, m, dp, flags), short.reshape(1).to(torch.int32), b_l, meta_b[:m], inv_b]
        if not same_rows:
            parts += [a_l, meta_a[:na], inv_a]
        rec, lay = _pack(parts)
        status = torch.zeros(1, dtype=torch.int32, device=dev)
        g1 = x.allgather(rec, status)
        b_g, meta_b_g, inv_b_g = _unpack(g1, lay, 2, T), _pad_meta_rows(_unpack(g1, lay, 3, T)), _unpack(g1, lay, 4, T)
        if same_rows:
            a_g, meta_a_g, inv_a_g = b_g, meta_b_g, inv_b_g
        else:
            a_g, meta_a_g, inv_a_g = _unpack(g1, lay, 5, T), _pad_meta_rows(_unpack(g1, lay, 6, T)), _unpack(g1, lay, 7, T)
        short_any = (_unpack(g1, lay, 1) != 0).any()
        na_g, m_g = na * W, m * W
        if uniform_weight:
            w_g = torch.full((na_g,), 1.0 / na_g, device=dev)
        else:         # fg_i / sum fg over the anchors of all ranks (per batch, averaged over the batches with foreground)
            w_g, _ = _ops.tile_weights(meta_a_g, na_g, T, bool(zero_if_empty))
        mine = lambda t: t.view(T, W, -1)[:, r].reshape(-1)          # this rank's rows of every batch
        w_l = mine(w_g)
        if normalize:
            shift_g = torch.full((na_g,), 1.0 / temperature, device=dev)
        else:         # |a_i| max_j |b_j| / T over the contrast rows of all ranks
            shift_g = _ops.p2p_shift(inv_a_g, inv_b_g, temperature)
        shift_l = mine(shift_g)
        analytic = n_class > 0
        selfcol_f = selfrow_g = a_selfcol_g = b_selfrow_l = None
        if selfcol is not None:        # the local self maps, moved into the global row index spaces
            build = lambda: _global_self_maps(selfcol, selfrow, na, m, W, r, T)
            # maps_key: the self maps are a pure function of the geometry it names (cached like the row indices)
            selfcol_f, selfrow_g, a_selfcol_g, b_selfrow_l = (build() if maps_key is None else
                                                              _cached(("global_self_maps", maps_key, W, r, T), build))
        loss_l, stats_l, state_l = _ops.p2p_fwd(a_l, b_g, meta_a, meta_b_g, shift_l, w_l, temperature, n_class, selfcol_f,
                                                analytic, T)
        parts2 = [_key(dev, na, m, dp, flags), loss_l]
        if analytic:
            off = ops.p2p_state_layout(na, dp)
            f32 = lambda name, n: state_l[off[name]:off[name] + 4 * n].view(torch.float32)
            parts2 += [f32("alpha", na), f32("beta", na), f32("colshift", na), f32("absum", T * n_class * (dp + 1))]
        else:
            parts2 += [stats_l]
        rec2, lay2 = _pack(parts2)
        g2 = x.allgather(rec2, status)
        partials = _unpack(g2, lay2, 1)
        loss = partials[0]
        for q in range(1, W):          # rank order: identical bits on every rank
            loss = loss + partials[q]
        loss = torch.where((status[0] != 0) | short_any, torch.full_like(loss, float("nan")), loss)
        if analytic:
            # per-anchor constants batch-major like the anchors; the ABsum tables stay rank-major (summed in rank order)
            state_g = _ops.p2p_state_assemble(_unpack(g2, lay2, 2, T), _unpack(g2, lay2, 3, T), _unpack(g2, lay2, 4, T),
                                              _unpack(g2, lay2, 5).reshape(W, -1), dp, n_class, T)
            stats_g = stats_l          # (not read by the analytic backward with a state)
        else:
            state_g, stats_g = None, _unpack(g2, lay2, 2, T).reshape(na_g, 3)
        ctx.save_for_backward(fm, idx_a, idx_b, a_l, b_l, a_g, b_g, meta_a, meta_b, meta_a_g, meta_b_g, inv_a, inv_b, shift_l,
                              shift_g, w_l, w_g, stats_l, stats_g, state_l, state_g, selfcol_f, selfrow_g, a_selfcol_g,
                              b_selfrow_l, rowmaps)
        ctx.cfg = (temperature, normalize, same_rows, c, n_class, T)
        return loss

    @staticmethod
    def backward(ctx, grad_out):
        (fm, idx_a, idx_b, a_l, b_l, a_g, b_g, meta_a, meta_b, meta_a_g, meta_b_g, inv_a, inv_b, shift_l, shift_g, w_l, w_g,
         stats_l, stats_g, state_l, state_g, selfcol_f, selfrow_g, a_selfcol_g, b_selfrow_l, rowmaps) = ctx.saved_tensors
        temperature, normalize, same_rows, c, n_class, T = ctx.cfg
        none = (None,) * 17
        if not ctx.needs_input_grad[0]:
            return (None,) + none
        g = grad_out.reshape(1)
        d_a, _ = _ops.p2p_bwd(a_l, b_g, c, meta_a, meta_b_g, shift_l, w_l, temperature, stats_l, g, True, False, n_class,
                              selfcol_f, selfrow_g, state_l if n_class > 0 else None, T)
        _, d_b = _ops.p2p_bwd(a_g, b_l, c, meta_a_g, meta_b, shift_g, w_g, temperature, stats_g, g, False, True, n_class,
                              a_selfcol_g, b_selfrow_l, state_g, T)
        if rowmaps is not None and not same_rows:
            return (_ops.scatter_rows_by_map(fm, normalize, rowmaps[0], d_a.contiguous(), inv_a, rowmaps[1], d_b.contiguous(),
                                             inv_b),) + none
        dfeat = torch.zeros_like(fm)
        if same_rows:
            _ops.scatter_rows_bwd(fm, idx_b, normalize, d_a + d_b, inv_b, dfeat)
        else:
            _ops.scatter_rows_bwd(fm, idx_a, normalize, d_a, inv_a, dfeat)
            _ops.scatter_rows_bwd(fm, idx_b, normalize, d_b, inv_b, dfeat)
        return (dfeat,) + none


def _offset_ids(meta, n, offset):
    """{label, id} rows with the ids of the first n rows moved by `offset` (ids unique across ranks)."""
    if offset:
        meta[:n, 1] += offset
    return meta


def p2p_loss(feat, idx_a, idx_b, lab_a, lab_b, id_a, id_b, weight, temperature, normalize, same_rows=False, n_class=0,
             selfcol=None, selfrow=None, n_batch=1, metas=None, id_bound=None):
    """``same_rows``: anchors and contrast rows are the same gathered rows (one gather); their labels may
    still differ (ISCL compares query labels with the anchors' dominant labels).
    ``n_batch`` > 1: block-diagonal batches -- rows [z R/n, (z+1) R/n) of both sides only see each other (R/n a
    multiple of 128; either mode -- the analytic sweeps keep one table of per-class sums per batch).
    ``n_class`` in 1..8: labels are class indices in [0, n_class) and ids are unique -> analytic sweeps; the
    self-pair maps are derived from the ids unless given.
    ``metas``: the {label, id} rows (``ops.rows_meta`` / ``ops.pad_meta``) when the caller has built them already
    (``lab_*`` are then unused); ``id_bound``: the ids are int64 in [0, id_bound) (pixel indices) -> the self-pair maps
    come from two lookup tables instead of a sort."""
    if same_rows and n_class == 0 and n_batch == 1 and metas is None and idx_a.numel() >= _SORT_MIN_ROWS:
        # General labels over ONE large row set (SupCon family, ISCL): the sums are order-invariant, so gather the rows
        # sorted by contrast label -- label-uniform column tiles take the sweeps' fast path -- and hand the kernels the
        # self maps (row i is its own contrast row), which takes the id tests out of the sweeps.  (Small or batched
        # problems are launch-bound: the sort would cost more than it saves.)
        n = idx_a.numel()
        order = torch.argsort(lab_b.long(), stable=True)
        same_labels = lab_b is lab_a
        idx_a = idx_b = idx_a[order]
        lab_b = lab_b[order]
        lab_a = lab_b if same_labels else lab_a[order]
        weight = weight[order]
        id_a = id_b = torch.arange(n, device=feat.device, dtype=torch.int32)
        selfcol = selfrow = id_a
    rowmaps = None
    if metas is not None:
        meta_a, meta_b = metas
    else:
        meta_a = ops.pad_meta(lab_a, id_a)
        meta_b = meta_a if (same_rows and lab_b is lab_a) else ops.pad_meta(lab_b, id_b)
    if n_class > 0 and selfcol is None:
        if same_rows:
            selfcol = torch.arange(idx_a.numel(), device=feat.device, dtype=torch.int32)
            selfrow = selfcol
        elif id_bound is not None:
            selfcol, selfrow, tables = _ops.self_maps_bounded(id_a, id_b, int(id_bound))
            n_pix = feat.shape[0] * feat.shape[2] * feat.shape[3]
            if id_a is idx_a and id_b is idx_b and int(id_bound) == n_pix and (idx_a.numel() + idx_b.numel()) * 4 >= n_pix:
                rowmaps = tables          # the ids ARE the pixel indices: the tables are pixel -> row maps
        else:
            selfcol, selfrow = ops.self_maps(id_a, id_b)
    return _P2PLoss.apply(feat, idx_a.contiguous(), idx_b.contiguous(), meta_a, meta_b, weight.float().contiguous(),
                          float(temperature), bool(normalize), bool(same_rows), int(n_class), selfcol, selfrow, int(n_batch),
                          rowmaps)


_INDEX_CACHE = {}          # row-index tensors per geometry: pure functions of the shapes, rebuilt ~20 small torch ops a call


def _cached(key, build):
    hit = _INDEX_CACHE.get(key)
    if hit is None:
        if len(_INDEX_CACHE) > 64:
            _INDEX_CACHE.clear()
        hit = _INDEX_CACHE[key] = build()
    return hit


def _view_major_rows(b: int, v: int, h: int, w: int, ys: torch.Tensor, xs: torch.Tensor, device) -> torch.Tensor:
    """Pixel indices (into the [b*v, c, h, w] memory-order map) of the reference's row order
    ``cat(unbind(features, dim=1), dim=0)`` (utils/loss.py:337-343) restricted to rows ys, cols xs."""
    grid = (ys.view(-1, 1) * w + xs.view(1, -1)).reshape(-1)                      # [hs*ws]
    img = (torch.arange(b, device=device).view(1, -1) * v + torch.arange(v, device=device).view(-1, 1)).reshape(-1)
    return (img.view(-1, 1) * (h * w) + grid.view(1, -1)).reshape(-1)             # (v, b, y, x) order


def _supcon(features, labels, temperature, ys, xs, zero_if_no_foreground=False, n_class=0, geom=None, x=None):
    if features.ndim <= 3:                                                          # :334-336
        raise ValueError('`features` needs to be [bsz, n_views, ...],'
                         'at least 4 dimensions are required')
    if features.ndim != 5:
        raise ValueError("slcl SupConLoss expects [bsz, n_views, c, h, w] features")
    b, v, c, h, w = features.shape
    dev = features.device
    fmap = features.reshape(b * v, c, h, w)
    if geom is not None:          # ys / xs are a pure function of `geom`: reuse the index tensors of the previous call
        idx, ids = _cached(("rows", b, v, h, w, geom, str(dev)),
                           lambda: (lambda i: (i, torch.arange(i.numel(), device=dev, dtype=torch.int32)))(
                               _view_major_rows(b, v, h, w, ys(), xs(), dev)))
    else:
        idx = _view_major_rows(b, v, h, w, ys, xs, dev)
        ids = torch.arange(idx.numel(), device=dev, dtype=torch.int32)
    m = idx.numel()
    if x is not None:
        return _supcon_global(fmap, labels, idx, ids, m, v, temperature, zero_if_no_foreground, n_class, x)
    if labels is not None:
        # {label, pixel index} rows and the foreground weights fg / sum fg (:352-358, :382-384) in three launches;
        # zero_if_no_foreground: LocalConLoss / BlockConLoss early-out (:405-407, :439-440), without a host sync
        meta = _ops.rows_meta(labels.reshape(-1).long(), idx)
        weight, _ = _ops.tile_weights(meta, m, 1, bool(zero_if_no_foreground))
        if n_class > 0:
            return p2p_loss(fmap, idx, idx, None, None, ids, ids, weight, temperature, normalize=False, same_rows=True,
                            n_class=n_class, metas=(meta, meta))
        lab = meta[:m, 0]                 # general sweeps: p2p_loss may sort the rows by label and rebuilds the metadata
        return p2p_loss(fmap, idx, idx, lab, lab, ids, ids, weight, temperature, normalize=False, same_rows=True, n_class=0)
    lab = (ids % (m // v)).to(torch.int32)                                          # :360-361 same pixel, other views
    weight = torch.full((m,), 1.0 / m, device=dev)                                  # :386
    return p2p_loss(fmap, idx, idx, lab, lab, ids, ids, weight, temperature, normalize=False, same_rows=True, n_class=0)


def _supcon_global(fmap, labels, idx, ids, m, v, temperature, zero_if_no_foreground, n_class, x, n_batch=1, geom=None):
    """SupCon over the union of every rank's rows (rank-major): ids are pixel indices offset by the rank's pixel count
    (labelled), or row indices offset by the rank's row count with "same pixel, other view" labels offset likewise.
    ``n_batch`` > 1: BlockConLoss's block-diagonal tiles -- tile z of the global problem holds tile z's rows of every rank
    (global order [tile][rank][view, image, y, x], see _unpack), so the ids above are unique within every tile across
    ranks; ``geom`` names the row geometry, of which the self maps are then a pure function (cached)."""
    n_pix = fmap.shape[0] * fmap.shape[2] * fmap.shape[3]
    if max(n_pix, m) * x.world >= 2 ** 31:
        raise ValueError("group=: the global row / pixel ids must fit in int32")
    no_short = torch.zeros((), dtype=torch.bool, device=fmap.device)
    if labels is not None:
        meta = _offset_ids(_ops.rows_meta(labels.reshape(-1).long(), idx), m, x.rank * n_pix)
        selfcol = ids if n_class > 0 else None          # ids = arange(m): row i is its own contrast row
        return _P2PGlobal.apply(fmap, idx, idx, meta, meta, no_short, float(temperature), False, True, int(n_class), selfcol,
                                selfcol, False, bool(zero_if_no_foreground), x, None, n_batch, geom)
    per = m // (v * n_batch)
    meta = ops.pad_meta(ids % per + x.rank * per, ids + x.rank * m)
    return _P2PGlobal.apply(fmap, idx, idx, meta, meta, no_short, float(temperature), False, True, 0, None, None, True, False,
                            x, None, n_batch, None)


class SupConLoss(nn.Module):
    """Reference utils/loss.py:315-387.  ``contrast_mode`` / ``base_temperature`` are stored and
    unused there too."""

    def __init__(self, temperature=0.07, contrast_mode='all', base_temperature=0.07, n_class=None, group=None):
        super().__init__()
        self.temperature = temperature
        self.contrast_mode = contrast_mode
        self.base_temperature = base_temperature
        # extension: 1..8 = labels are class indices in [0, n_class) -> analytic tensor-core sweeps; 0 = general sweeps
        # (any integer labels); None (default) = decided from the labels themselves (_AutoClasses)
        self.n_class = n_class
        self._classes = _AutoClasses(n_class)
        # extension (INTEGRATION.md section 4): None = this batch only.  True / a ProcessGroup (NCCL) or a
        # slcl.peer.PeerMailbox built with rows_bytes (NVLink peer memory): every forward gets this rank's shard of a
        # data-parallel batch and returns SupCon over the GLOBAL batch -- every rank's rows are anchors and contrast rows,
        # in rank order; every rank returns the same loss and gets its shard of the gradient.  All ranks pass equal
        # shapes, make the same sequence of group= calls and back-propagate the same grad_out.  A constructor argument
        # here because SupConLoss.forward is a drop-in whose parameter list stays exactly the reference's (features,
        # labels); LocalConLoss, which has no such constraint, also takes it per call.  Without n_class, the sweeps are
        # chosen once, at the first labelled call, from the label range over all ranks of that call's group.
        self.group = group

    def forward(self, features, labels=None):
        if features.ndim <= 3:
            raise ValueError('`features` needs to be [bsz, n_views, ...],'
                             'at least 4 dimensions are required')
        h, w = features.shape[-2:]
        dev = features.device
        x = _exchange(self.group)
        n_class, in_range = self._classes.resolve(labels, x)
        return _guard(_supcon(features, labels, self.temperature, lambda: torch.arange(h, device=dev),
                              lambda: torch.arange(w, device=dev), n_class=n_class, geom=("all",), x=x), in_range)


class LocalConLoss(nn.Module):
    """Reference utils/loss.py:390-413: stride-subsampled SupCon."""

    def __init__(self, temperature=0.7, stride=4, n_class=None, group=None):
        super().__init__()
        self.temp = temperature
        # group: as SupConLoss's (the default of forward's group)
        self.supconloss = SupConLoss(temperature=self.temp, n_class=n_class, group=group)
        self.stride = stride

    def forward(self, features, labels=None, group=None):
        """``group`` (extension; INTEGRATION.md section 4): the data-parallel group of this call -- None = the one given to
        the constructor (None there too: this batch only); True / a ProcessGroup (NCCL) or a ``slcl.peer.PeerMailbox``
        built with ``rows_bytes``: the loss of the GLOBAL batch, as ``SupConLoss(group=)``.  The "no foreground -> 0"
        early-out then holds only when no rank has foreground.  Without ``n_class`` the sweeps are chosen once per module,
        at its first labelled call, from the label range over all ranks of that call's group."""
        h, w = features.shape[-2:]
        dev = features.device
        st = self.stride
        x = _exchange(self.supconloss.group if group is None else group)
        n_class, in_range = self.supconloss._classes.resolve(labels, x)
        return _guard(_supcon(features, labels, self.temp, lambda: torch.arange(0, h, st, device=dev),
                              lambda: torch.arange(0, w, st, device=dev), zero_if_no_foreground=True, n_class=n_class,
                              geom=("stride", st), x=x), in_range)


class BlockConLoss(nn.Module):
    """Reference utils/loss.py:416-466: mean of SupCon over block_size x block_size tiles; tiles whose
    labels are all background are skipped (decided on the device, no per-tile host sync)."""

    def __init__(self, temperature=0.7, block_size=32, n_class=None, group=None):
        super().__init__()
        self.block_size = block_size
        # group: as SupConLoss's (the default of forward's group)
        self.supconloss = SupConLoss(temperature=temperature, n_class=n_class, group=group)
        self.batched = True             # all tiles as one block-diagonal problem where the shape allows (False: per-tile loop)

    def forward(self, features, labels=None, group=None):
        """``group`` (extension; INTEGRATION.md section 4): the data-parallel group of this call -- None = the one given to
        the constructor (None there too: this batch only); True / a ProcessGroup (NCCL) or a ``slcl.peer.PeerMailbox``
        built with ``rows_bytes``: the loss of the GLOBAL batch, i.e. BlockConLoss of the ranks' batches concatenated.
        Every tile's problem is then the union of that tile's rows on all ranks, tile weights and the average over tiles
        with foreground are decided over that union, and "no foreground -> 0" holds only when no rank has foreground.
        The global form needs the block-diagonal layout (b v block_size^2 a multiple of 128, ``batched``): other shapes
        raise ValueError on every rank before anything is exchanged."""
        dev = features.device
        bs = self.block_size
        div = features.shape[-1] // bs                                               # :426-428
        t = self.supconloss.temperature
        if div == 0:
            return torch.zeros((), device=dev)
        x = _exchange(self.supconloss.group if group is None else group)
        batched = self.batched and features.ndim == 5 and (features.shape[0] * features.shape[1] * bs * bs) % 128 == 0
        if x is not None and not batched:
            raise ValueError("BlockConLoss(group=) needs [b, v, c, h, w] features with b * v * block_size^2 a multiple of "
                             "128 and batched = True (the per-tile loop would need div^2 exchanges)")
        n_class, in_range = self.supconloss._classes.resolve(labels, x)
        if batched:
            return _guard(self._forward_batched(features, labels, div, t, n_class, x), in_range)
        losses, flags = [], []
        for i in range(div):
            for j in range(div):
                ys = torch.arange(i * bs, (i + 1) * bs, device=dev)
                xs = torch.arange(j * bs, (j + 1) * bs, device=dev)
                losses.append(_supcon(features, labels, t, ys, xs, zero_if_no_foreground=True, n_class=n_class))
                if labels is not None:
                    flags.append((labels[:, :, i * bs:(i + 1) * bs, j * bs:(j + 1) * bs] != 0).any())
        stacked = torch.stack(losses)
        if labels is None:
            return stacked.mean()                                                    # :465 (general sweeps: no guard)
        keep = torch.stack(flags).float()
        return _guard((stacked * keep).sum() / keep.sum().clamp_min(1.0), in_range)   # :445-448 (0 when every tile is skipped)

    def _forward_batched(self, features, labels, div, t, n_class=0, x=None):
        """All div x div tiles as ONE block-diagonal problem (one launch per tensor-core sweep instead of div^2
        separate SupCon calls): rows are ordered (tile, view, image, y, x); the per-tile weighting of :445-448 /
        :465 -- fg_i / sum_tile fg, averaged over the tiles that have foreground -- is folded into the row weights.
        ``n_class`` > 0 (class-index labels): the analytic sweeps with one table of per-class sums per tile."""
        b, v, c, h, w = features.shape
        dev = features.device
        bs = self.block_size
        fmap = features.reshape(b * v, c, h, w)

        def build():
            ar = torch.arange(bs, device=dev)
            ti = torch.arange(div, device=dev)
            ys = (ti.view(-1, 1) * bs + ar.view(1, -1))                                  # [div, bs]
            grid = (ys.view(div, 1, bs, 1) * w + ys.view(1, div, 1, bs)).reshape(div * div, bs * bs)      # [tiles, bs*bs]
            img = (torch.arange(b, device=dev).view(1, -1) * v + torch.arange(v, device=dev).view(-1, 1)).reshape(-1)   # (v, b)
            i = (img.view(1, -1, 1) * (h * w) + grid.view(div * div, 1, bs * bs)).reshape(-1)           # (tile, v, b, y, x)
            return i, torch.arange(i.numel(), device=dev, dtype=torch.int32)
        geom = ("blocks", b, v, h, w, bs, div, str(dev))
        idx, ids = _cached(geom, build)
        n_tiles, m_tile = div * div, b * v * bs * bs
        if x is not None:
            return _supcon_global(fmap, labels, idx, ids, idx.numel(), v, t, True, n_class, x, n_tiles, geom)
        if labels is not None:
            meta = _ops.rows_meta(labels.reshape(-1).long(), idx)
            weight, _ = _ops.tile_weights(meta, idx.numel(), n_tiles, True)
            return p2p_loss(fmap, idx, idx, None, None, ids, ids, weight, t, normalize=False, same_rows=True,
                            n_class=n_class, n_batch=n_tiles, metas=(meta, meta))
        lab = (ids % (m_tile // v)).to(torch.int32)                                   # same pixel of the tile, other views
        weight = torch.full((idx.numel(),), 1.0 / (m_tile * n_tiles), device=dev)
        return p2p_loss(fmap, idx, idx, lab, lab, ids, ids, weight, t, normalize=False, same_rows=True, n_batch=n_tiles)


def sample_class_balanced(labels: torch.Tensor, n_anchor: int, n_contrast: int, n_class: int,
                          generator: Optional[torch.Generator] = None, return_counts: bool = False):
    """Class-balanced sampler (SURVEY.md 8(c)-3; north_star item 1), with NO host synchronisation.

    ONE permutation of all pixels is drawn from PyTorch's RNG stream -- ``torch.randperm(N, generator)``, on the label
    map's device unless the generator lives elsewhere -- and the labels are read in that order.  The stable per-class
    compaction of the permuted labels (CUDA kernel ``slcl_compact_by_class``, order bit-identical to ``torch.nonzero``)
    gives every pixel its rank within its class; class k contributes its first ``ceil(n / K)`` pixels in permutation
    order (class-major output), and slots a short class leaves open are filled with the next unpicked labelled pixels
    (the test-side restatement of this rule is ``sample_class_balanced`` of the CPU checker).  Output sizes are ``K * ceil(n / K)`` whatever the class
    counts, so nothing has to come back to the host.  Anchors use the same rule with their own quota (their per-class
    picks are a prefix of the contrast picks of that class).  Returns (anchor_idx, contrast_idx[, n_filled_anchor, n_filled_contrast])."""
    lab = labels.reshape(-1).long()
    n = lab.numel()
    dev = lab.device
    gen_dev = generator.device if generator is not None else dev
    perm = torch.randperm(n, generator=generator, device=gen_dev).to(dev)
    per_a = -(-n_anchor // n_class)
    per_c = -(-n_contrast // n_class)
    # labels in permutation order -> stable per-class compaction -> phase-1 prefix per class -> phase-2 fill, both quotas:
    # one C-ABI call (slcl_sample_balanced), ~13 launches where the torch formulation of the same rule took ~60
    a_idx, a_fill, c_idx, c_fill = _ops.sample_balanced(perm, lab, n_class, per_a, per_c)
    a_fill, c_fill = a_fill[0], c_fill[0]
    if return_counts:
        return a_idx, c_idx, a_fill, c_fill
    return a_idx, c_idx


def sampled_supcon_loss(feat: torch.Tensor, labels: torch.Tensor, n_anchor: int, n_contrast: int, n_class: int,
                        temperature: float = 0.7, generator: Optional[torch.Generator] = None,
                        anchor_idx: Optional[torch.Tensor] = None, contrast_idx: Optional[torch.Tensor] = None,
                        analytic: bool = True, group=None):
    """Sampled rectangular pixel <-> pixel loss (BASELINE.json configs[2]): anchors x contrast rows
    drawn class-balanced from an NCHW map, L2-normalised, bf16 tensor-core similarities.  The whole call -- draw,
    compaction, gather, sweeps -- runs without a host synchronisation; if the map holds fewer labelled pixels than the
    sample needs, the loss is NaN (decided on the device).

    ``group`` (extension; INTEGRATION.md section 4): ``feat`` / ``labels`` are this rank's shard of a data-parallel batch.
    Each rank draws its rows from its own shard with its own generator, exactly as without a group; the loss is the one of
    the union of all ranks' draws (anchors and contrast rows in rank order, weights fg_i / sum fg over all anchors), the same
    on every rank, and the gradient is this rank's shard of its gradient.  NaN on every rank if any rank is short of
    labelled pixels.  ``True`` / a ProcessGroup: NCCL; a ``slcl.peer.PeerMailbox`` built with ``rows_bytes >=
    global_record_bytes(...)``: NVLink peer memory.  All ranks pass equal shapes, make the same sequence of ``group=``
    calls and back-propagate the same grad_out."""
    short = None
    if anchor_idx is None or contrast_idx is None:
        anchor_idx, contrast_idx, a_fill, c_fill = sample_class_balanced(labels, n_anchor, n_contrast, n_class, generator,
                                                                          return_counts=True)
        short = (a_fill < anchor_idx.numel()) | (c_fill < contrast_idx.numel())
    lab = labels.reshape(-1).long()
    anchor_idx, contrast_idx = anchor_idx.reshape(-1).long(), contrast_idx.reshape(-1).long()
    x = _exchange(group)
    if x is not None:
        return _sampled_global(feat, lab, anchor_idx, contrast_idx, short, n_class, temperature, analytic, x)
    meta_a, meta_b = _ops.rows_meta(lab, anchor_idx), _ops.rows_meta(lab, contrast_idx)          # {label, pixel index}
    weight, _ = _ops.tile_weights(meta_a, anchor_idx.numel(), 1, False)          # fg / sum fg over the anchors
    # analytic sweeps need class-index labels (true here) and unique picks (distinct pixels of one permutation are)
    loss = p2p_loss(feat, anchor_idx, contrast_idx, None, None, anchor_idx, contrast_idx, weight, temperature, normalize=True,
                    n_class=n_class if (analytic and n_class <= 8) else 0, metas=(meta_a, meta_b), id_bound=lab.numel())
    if short is not None:
        loss = torch.where(short, torch.full_like(loss, float("nan")), loss)
    return loss


def _sampled_global(feat, lab, anchor_idx, contrast_idx, short, n_class, temperature, analytic, x):
    n_pix = lab.numel()
    if n_pix * x.world >= 2 ** 31:
        raise ValueError("group=: the global pixel ids must fit in int32")
    off = x.rank * n_pix                 # ids: pixel index in the rank-major global map
    meta_a = _offset_ids(_ops.rows_meta(lab, anchor_idx), anchor_idx.numel(), off)
    meta_b = _offset_ids(_ops.rows_meta(lab, contrast_idx), contrast_idx.numel(), off)
    n_cls = n_class if (analytic and n_class <= 8) else 0
    selfcol = selfrow = rowmaps = None
    if n_cls > 0:                         # self pairs live on one rank: the local maps, offset inside _P2PGlobal
        selfcol, selfrow, tables = _ops.self_maps_bounded(anchor_idx, contrast_idx, n_pix)
        if (anchor_idx.numel() + contrast_idx.numel()) * 4 >= n_pix:
            rowmaps = tables
    if short is None:
        short = torch.zeros((), dtype=torch.bool, device=feat.device)
    return _P2PGlobal.apply(feat, anchor_idx, contrast_idx, meta_a, meta_b, short, float(temperature), True, False, n_cls,
                            selfcol, selfrow, False, False, x, rowmaps, 1, None)


class InterpolatedSupervisedContrastiveLoss(nn.Module):
    """ISCL on [N, d] feature vectors (reference utils/losses.py:6-81; SURVEY.md 8(f)-4): mix-up supervised
    contrastive loss -- two label sets over the SAME Gram matrix, mixed with lambda.  Each term is one sweep of
    the tensor-core kernel with different row (query) labels and the dominant labels on the columns."""

    def __init__(self, temperature):
        super().__init__()
        self.temperature = temperature

    def forward(self, features, labels_1, labels_2, dominant_labels, lambdas, normalize=True):
        n, d = features.shape
        dev = features.device
        fmap = features.reshape(n, d, 1, 1)                 # rows [N,d] are an NCHW map with HW = 1
        idx = torch.arange(n, device=dev)
        ids = idx.to(torch.int32)
        lam = lambdas.to(torch.float32).reshape(-1)
        dom = dominant_labels.reshape(-1)
        t1 = p2p_loss(fmap, idx, idx, labels_1.reshape(-1), dom, ids, ids, lam / n, self.temperature, normalize, same_rows=True)
        t2 = p2p_loss(fmap, idx, idx, labels_2.reshape(-1), dom, ids, ids, (1.0 - lam) / n, self.temperature, normalize,
                      same_rows=True)
        return t1 + t2                                       # :55-59 (losses.mean())
