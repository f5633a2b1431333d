"""Drop-in for the contrastive-loss part of the reference's ``utils/loss.py``.

Same class / function names, argument meaning and error behaviour as the
reference (file:line cited per item); the arithmetic runs in libslcl.so.
"""
from __future__ import annotations

import math

import torch
import torch.nn as nn
import torch.nn.functional as F

from . import functional as SF
from . import p2p


class MPCL(nn.Module):
    """Pixel -> prototype margin InfoNCE.  Reference: utils/loss.py:469-573."""

    def __init__(self, device, num_class=5, temperature=0.07, m=0.5, base_temperature=0.07, easy_margin=False):
        super().__init__()
        self.num_class = num_class
        self.temperature = temperature
        self.base_temperature = base_temperature
        self.m = m
        self.cos_m = math.cos(m)
        self.sin_m = math.sin(m)
        self.th = math.cos(math.pi - m)
        self.mm = math.sin(math.pi - m) * m
        self.device = device
        self.easy_margin = easy_margin

    def _kw(self, normalize):
        return dict(n_class=self.num_class, temperature=self.temperature, base_temperature=self.base_temperature,
                    margin=self.m, easy_margin=self.easy_margin, normalize=normalize)

    def forward(self, features, labels, class_center_feas, pixel_sel_loc=None, mask=None):
        """features [N,1,C] unit rows; labels [N]; class_center_feas [C,K] unit
        columns; pixel_sel_loc [N]; mask [N,K] soft positives (utils/loss.py:484-573)."""
        if len(features.shape) < 3:                                     # :494-496
            raise ValueError('`features` needs to be [bsz, n_views, ...],'
                             'at least 3 dimensions are required')
        if len(features.shape) > 3:
            features = features.view(features.shape[0], features.shape[1], -1)
        if labels is not None and mask is not None:                     # :502-503
            raise ValueError('Cannot define both `labels` and `mask`')
        if features.shape[1] != 1:
            # the reference cannot run this either: mask.repeat(anchor_count, contrast_count) (:548) is [V*N, V*K] against
            # [V*N, K] logits, a RuntimeError from the broadcast at :552 -- same exception type, raised before any work
            raise RuntimeError(f"MPCL: n_views = {features.shape[1]} > 1 -- the size of tensor a ({self.num_class}) must match "
                               f"the size of tensor b ({features.shape[1] * self.num_class}) at non-singleton dimension 1 "
                               "(utils/loss.py:548-552); only n_views == 1 is defined")
        n = features.shape[0]
        if labels is None and mask is None:                             # :504-505  (eye(N) positives)
            if n != self.num_class:
                raise ValueError("labels=None and mask=None needs N == num_class (identity positive mask)")
            mask = torch.eye(n, dtype=torch.float32, device=features.device)
        if labels is not None:
            labels = labels.contiguous().view(-1).long()
            if labels.shape[0] != n:                                    # :511-512
                raise ValueError('Num of labels does not match num of features')
        else:
            mask = mask.float()
        rows = features[:, 0, :]
        centres = class_center_feas.transpose(0, 1)                     # [K, C]
        sel = None if pixel_sel_loc is None else pixel_sel_loc.view(-1)
        return SF.proto_loss(rows, labels, mask, sel, centres, rows_layout=True, **self._kw(normalize=False))


def mpcl_loss_calc(feas, labels, class_center_feas, loss_func, pixel_sel_loc=None, tag='source', group=None):
    """feas [B,C,h,w]; labels [B,H,W] (source) or [N] (target); class_center_feas
    [K,C]; loss_func an ``MPCL``.  Reference: utils/loss.py:576-605.  With an slcl
    ``MPCL`` the normalisation, the NCHW->NHWC copy and the loss are one fused
    kernel over the NCHW map; any other callable gets the reference call
    sequence.  ``group`` (addition): torch.distributed group (or True for the
    default group) over which the batch is sharded -- the loss becomes the mean
    over the GLOBAL batch (one 8-byte all-reduce), gradients follow."""
    n, c, fea_h, fea_w = feas.size()
    if tag == 'source' and (labels.size()[1] != fea_h or labels.size()[2] != fea_w):     # :585-590
        labels = labels.float()
        labels = F.interpolate(labels, size=fea_w, mode='nearest')
        labels = labels.permute(0, 2, 1).contiguous()
        labels = F.interpolate(labels, size=fea_h, mode='nearest')
        labels = labels.permute(0, 2, 1).contiguous()
    labels = labels.to(feas.device).reshape(-1).long()                                   # :592-593
    if isinstance(loss_func, MPCL):
        if labels.shape[0] != n * fea_h * fea_w:
            raise ValueError('Num of labels does not match num of features')
        sel = None if pixel_sel_loc is None else pixel_sel_loc.view(-1)
        return SF.proto_loss(feas, labels, None, sel, class_center_feas, rows_layout=False, group=group,
                             **loss_func._kw(normalize=True))
    unit = F.normalize(feas, p=2, dim=1).permute(0, 2, 3, 1).reshape(n * fea_h * fea_w, c).unsqueeze(1)
    centres = F.normalize(class_center_feas, p=2, dim=1).transpose(0, 1)
    return loss_func(unit, labels, centres, pixel_sel_loc=pixel_sel_loc)


def mpcl_target_step(feas_t, class_center_feas, loss_func, pixel_sel_th=.25, group=None, with_centroids=False,
                     weight_by_sel=False, previous_centroid=None, momentum=0.95):
    """Fused target step of trainer/Trainer_MPSCL.py:135,144 (an addition, SURVEY.md 8(f)-1):

        hard, mask = generate_pseudo_label(feas_t, class_center_feas, pixel_sel_th)
        loss = mpcl_loss_calc(feas_t, hard, class_center_feas, loss_func, pixel_sel_loc=mask, tag='target')

    in ONE read of ``feas_t`` (the reference reads and normalises it twice).  Returns ``(loss, hard, mask)``;
    gradients flow to ``feas_t`` only (the reference callers pass detached centres, :145).

    ``with_centroids=True`` adds, from the SAME read, the hard target centroids of the map under the pseudo labels it has
    just produced -- ``cal_centroid(feas_t, one_hot(hard), pseudo_label=True, weighted_ave=False)`` (utils/utils_.py:524-529),
    optionally restricted to the selected pixels (``weight_by_sel``) and EMA'd with ``previous_centroid`` -- and returns
    ``(loss, hard, mask, centroids [K, C])``; the centroids are differentiable w.r.t. ``feas_t``."""
    if not isinstance(loss_func, MPCL):
        raise TypeError("loss_func must be an slcl.loss.MPCL")
    kw = loss_func._kw(normalize=True)
    kw.pop("normalize")
    if with_centroids:
        return SF.proto_target_step_centroids(feas_t, class_center_feas, previous_centroid, pixel_sel_th,
                                              weight_by_sel=weight_by_sel, momentum=momentum, group=group, **kw)
    return SF.proto_target_step(feas_t, class_center_feas, pixel_sel_th, group=group, **kw)


def mpcl_source_step(feas_s, labels_s, class_center_feas, loss_func, m=.2, num_class=4, group=None):
    """Source side of trainer/Trainer_MPSCL.py:133,138 as one call (SURVEY.md 8(f)-1):

        centres = update_class_center_iter(feas_s, labels_s, class_center_feas, m)
        loss = mpcl_loss_calc(feas_s, labels_s, centres.detach(), loss_func, tag='source')

    The loss needs the centres of the WHOLE batch, so the map is walked twice by construction (class sums, then loss); what
    this call adds is residency: a map that fits in the 126 MB L2 (the per-GPU map of configs[3] does) is kept there by
    the first walk -- TMA loads with the default evict_normal policy, the loss forward with evict_last -- so the second
    and third walks (loss forward, loss backward) read it from L2, not from HBM.  Returns ``(centres, loss)``."""
    from .utils_ import update_class_center_iter
    if labels_s.shape[-2:] != feas_s.shape[-2:]:
        raise ValueError("labels must be at feature resolution (update_class_center_iter, utils/utils_.py:575-577)")
    centres = update_class_center_iter(feas_s, labels_s, class_center_feas, m=m, num_class=num_class, group=group)
    loss = mpcl_loss_calc(feas_s, labels_s, centres.detach(), loss_func, tag='source', group=group)
    return centres, loss


class ContrastiveLoss(nn.Module):
    """Centroid <-> centroid InfoNCE.  Reference: utils/loss.py:233-275.
    Bug-compatible: ``tau`` is stored and never used (:236 vs :264-265); the row
    range ends at the reference's hard-coded 4 (:266) when K == 4 and at K otherwise
    (the reference raises a shape error for K != 4)."""

    def __init__(self, tau=5, n_class=4, bg=False, norm=True):
        super().__init__()
        self._tau = tau
        self._norm = norm

    def forward(self, centroid_s, centroid_t, bg=False, split=False):
        k = centroid_s.shape[0]
        return SF.centroid_loss(centroid_s, centroid_t, mode=1 if split else 0, first_row=0 if bg else 1, n_rows=k,
                                norm=bool(self._norm))


def cnr_loss(centroid_s, centroid_t_list):
    """Centroid-norm regulariser written inline in the reference trainer
    (trainer/Trainer_MCCL.py:303-315): sum_p MSE(||t_p||, ||s||) / P."""
    if isinstance(centroid_t_list, torch.Tensor):
        centroid_t_list = [centroid_t_list]
    total = 0
    for ct in centroid_t_list:
        total = total + SF.centroid_loss(centroid_s, ct, mode=2, first_row=0, n_rows=centroid_s.shape[0], norm=False) \
            / len(centroid_t_list)
    return total


def mccl_centroid_losses(centroid_s, centroid_t, centroid_t_aug=None, inter_w=1.0, intra_w=1.0, cnr_w=4e-5, split=False, bg=False,
                         norm=True):
    """Every centroid <-> centroid term of one MCCL adaptation step (trainer/Trainer_MCCL.py:303-326) in ONE op (an
    addition; the drop-in ``ContrastiveLoss`` / ``cnr_loss`` calls stay available and give the same numbers):

        inter = sum_p ContrastiveLoss()(centroid_s, centroid_t[p], split=split) / P
        intra = sum_p ContrastiveLoss()(centroid_t[p], centroid_t_aug, split=split) / P        (if centroid_t_aug is given)
        cnr   = sum_p MSE(||centroid_t[p]||, ||centroid_s||) / P
        total = inter_w * inter + intra_w * intra + cnr_w * cnr

    ``centroid_t``: the list of P ``[K,C]`` tensors ``cal_centroid(..., partition=P)`` returns (or one tensor).  Returns
    ``(total, terms)`` with ``terms = [inter, intra, cnr]`` detached for logging.  Two kernel launches forward (all pairs in
    parallel blocks, then the weighted combination and ALL gradients), three small scalings backward -- instead of ~60."""
    if isinstance(centroid_t, torch.Tensor):
        centroid_t = [centroid_t]
    parts = torch.cat(list(centroid_t), dim=0) if len(centroid_t) > 1 else centroid_t[0]
    return SF.mccl_losses(centroid_s, parts, centroid_t_aug, n_partitions=len(centroid_t), split=split, bg=bg, norm=norm,
                          inter_w=inter_w, intra_w=intra_w, cnr_w=cnr_w)


def mccl_step(ft_s, labels_s, ft_t, pred_t, ft_t_aug=None, pred_t_aug=None, *, n_class=4, partition=2, part_id=None,
              generator=None, threshold=None, weighted_ave=True, from_logits=True, previous_centroid_s=None, momentum=0.95,
              inter_w=1.0, intra_w=1.0, cnr_w=4e-5, split=False, bg=False, norm=True, group=None):
    """The MCCL loss section of trainer/Trainer_MCCL.py:275-326, from the decoder outputs to the loss, as ONE forward and
    ONE backward call (an addition).  It is defined as this composition of the drop-in calls::

        cs, _, _ = cal_centroid(ft_s, labels_s, previous_centroid=previous_centroid_s, momentum=momentum, n_class=n_class)
        cs = cs.detach()
        ct, _, _ = cal_centroid(ft_t, pred_t, pseudo_label=True, partition=partition, threshold=threshold,
                                weighted_ave=weighted_ave, n_class=n_class, part_id=part_id, generator=generator,
                                from_logits=from_logits)
        ct_aug, _, _ = cal_centroid(ft_t_aug, pred_t_aug, pseudo_label=True, threshold=threshold,
                                    weighted_ave=weighted_ave, n_class=n_class, from_logits=from_logits)
        total, terms = mccl_centroid_losses(cs, ct, ct_aug, inter_w, intra_w, cnr_w, split=split, bg=bg, norm=norm)

    and returns ``(total, terms, cs, ct, ct_aug)``: ``total`` differentiable w.r.t. ``ft_t``, ``ft_t_aug``, ``pred_t`` and
    ``pred_t_aug`` (dL/dlogits with ``from_logits``, dL/dprobs otherwise); ``ft_s`` gets no gradient.  ``terms`` =
    ``[inter, intra, cnr]`` and the centroids are detached; ``ct`` is a list of ``partition`` tensors when
    ``partition > 1``; ``ct_aug`` is None without the augmented view (and there is then no intra term).

    The class sums of every set come from the same sweeps as ``cal_centroid``'s, reduced in the same order, and one tail
    kernel finalises the centroids and evaluates every centroid term: four launches forward when ``part_id`` is given,
    three backward, no host synchronisation.  ``group``: as ``cal_centroid`` / ``seg_losses`` -- the centroids and losses
    of the ranks' batches concatenated, with ONE exchange of all the sets' sums per step (inside the tail kernel for a
    ``slcl.peer.PeerMailbox``, one NCCL all-reduce for ``True`` / a ProcessGroup).

    Raises ``ValueError``, before any launch or exchange, for maps that are not contiguous float32 NCHW, channel counts
    that differ, ``n_class`` outside [2, 8] or ``partition * n_class > 16``, labels or ``pred`` not at the feature
    map's resolution, or a mailbox too small for the sums; the separate calls remain the route for those."""
    from .seg import _resolve_group
    from .utils_ import rmc_partition_ids
    from ._lib import MAX_CLASSES, MAX_WEIGHT_COLS
    from .peer import PeerMailbox
    k, parts = int(n_class), int(partition)
    if not (2 <= k <= MAX_CLASSES):
        raise ValueError(f"mccl_step: n_class must be in [2, {MAX_CLASSES}], got {k}")
    if parts < 1 or parts * k > MAX_WEIGHT_COLS:
        raise ValueError(f"mccl_step: partition * n_class must be at most {MAX_WEIGHT_COLS}, got {parts} * {k}")
    if (ft_t_aug is None) != (pred_t_aug is None):
        raise ValueError("mccl_step: ft_t_aug and pred_t_aug go together")
    maps = [("ft_s", ft_s), ("ft_t", ft_t)] + ([("ft_t_aug", ft_t_aug)] if ft_t_aug is not None else [])
    for name, m in maps:
        if not isinstance(m, torch.Tensor) or m.dim() != 4 or m.dtype != torch.float32 or not m.is_contiguous():
            raise ValueError(f"mccl_step: {name} must be a contiguous float32 [B, C, h, w] map")
    c, h, w = ft_s.shape[1:]
    for name, m in maps[1:]:
        if m.shape[1] != c:
            raise ValueError(f"mccl_step: {name} has {m.shape[1]} channels, ft_s has {c}")
        if tuple(m.shape[2:]) != (h, w):
            raise ValueError(f"mccl_step: {name} is {tuple(m.shape[2:])}, ft_s is {(h, w)}: the maps share one resolution")
    b_s, b_t = ft_s.shape[0], ft_t.shape[0]
    if labels_s.shape[-2:] != (h, w) or labels_s.numel() != b_s * h * w:
        raise ValueError(f"mccl_step: labels_s must be [B, h, w] = {(b_s, h, w)} at the feature map's resolution, "
                         f"got {tuple(labels_s.shape)}")
    for name, p, b in [("pred_t", pred_t, b_t)] + ([("pred_t_aug", pred_t_aug, ft_t_aug.shape[0])] if ft_t_aug is not None
                                                      else []):
        if tuple(p.shape) != (b, k, h, w) or p.dtype != torch.float32:
            raise ValueError(f"mccl_step: {name} must be float32 [B, K, h, w] = {(b, k, h, w)} at the feature map's "
                             f"resolution, got {tuple(p.shape)} {p.dtype}")
    if previous_centroid_s is not None and tuple(previous_centroid_s.shape) != (k, c):
        raise ValueError(f"mccl_step: previous_centroid_s must be [K, C] = {(k, c)}, got {tuple(previous_centroid_s.shape)}")
    if parts > 1 and part_id is not None and part_id.numel() != b_t * h * w:
        raise ValueError(f"mccl_step: part_id must hold B_t*h*w = {b_t * h * w} ids, got {part_id.numel()}")
    group = _resolve_group(group)
    rows = (parts + 1 + (ft_t_aug is not None)) * k
    if isinstance(group, PeerMailbox) and group.capacity_words < 2 * rows * (c + 1):
        raise ValueError(f"mccl_step: the sums of one step are {rows} x {c + 1} doubles; the mailbox needs capacity_words >= "
                         f"{2 * rows * (c + 1)}, this one has {group.capacity_words}")
    pid = None
    if parts > 1:
        pid = part_id if part_id is not None else rmc_partition_ids(b_t * h * w, parts, generator, ft_t.device)
        pid = pid.to(device=ft_t.device, dtype=torch.int32).reshape(-1)
    thr = float(threshold) if threshold is not None else 0.0
    total, terms, cen, _sums = SF.mccl_step(ft_s, labels_s.to(ft_s.device), ft_t, pred_t, pid, ft_t_aug, pred_t_aug,
                                            previous_centroid_s, n_partitions=parts, n_class=k, weighted=bool(weighted_ave),
                                            threshold=thr, from_logits=bool(from_logits), momentum=float(momentum),
                                            split=split, bg=bg, norm=norm, inter_w=inter_w, intra_w=intra_w, cnr_w=cnr_w,
                                            group=group)
    cs = cen[:k]
    ct = [cen[(p + 1) * k:(p + 2) * k] for p in range(parts)] if parts > 1 else cen[k:2 * k]
    ct_aug = cen[(parts + 1) * k:] if ft_t_aug is not None else None
    return total, terms, cs, ct, ct_aug


def mpscl_step(ft_s, labels_s, ft_t, class_center_feas, mpcl_src, mpcl_trg, *, m=0.9, num_class=4, pixel_sel_th=0.25,
               group=None):
    """The MPSCL loss section of trainer/Trainer_MPSCL.py:133-147 as ONE forward and ONE backward call (an addition).  It is
    defined as this composition of the drop-in calls::

        centres = update_class_center_iter(ft_s, labels_s, class_center_feas, m=m, num_class=num_class, group=group)
        hard, mask = generate_pseudo_label(ft_t, centres, pixel_sel_th)
        loss_s = mpcl_loss_calc(ft_s, labels_s, centres.detach(), mpcl_src, tag='source', group=group)
        loss_t = mpcl_loss_calc(ft_t, hard, centres.detach(), mpcl_trg, pixel_sel_loc=mask, tag='target', group=group)

    and returns ``(loss_s, loss_t, centres, hard, mask)`` with the same values.  ``loss_s`` is differentiable w.r.t.
    ``ft_s`` only, ``loss_t`` w.r.t. ``ft_t`` only; ``centres``, ``hard`` and ``mask`` are not differentiable.  The two
    ``MPCL`` modules may differ in margin, temperature, base temperature and ``easy_margin``.

    Five launches forward (class-sum sweep, reduce + EMA, unit centres, one prototype forward over both maps, one
    finaliser) and one backward (both maps; only the map whose loss receives a gradient), no host synchronisation.
    ``group``: as ``update_class_center_iter`` / ``mpcl_loss_calc`` -- two exchanges per step: the class sums, then both
    loss pairs at once (inside the reduce kernel and the finaliser for a ``slcl.peer.PeerMailbox``; two NCCL all-reduces
    for ``True`` / a ProcessGroup).  The backward exchanges nothing.

    Raises ``ValueError``, before any launch or exchange, for maps that are not contiguous float32 ``[B, C, h, w]``,
    channel counts or resolutions that differ between the maps (the batch sizes may differ), ``labels_s`` not at the
    feature resolution, ``class_center_feas`` not ``[num_class, C]`` or requiring grad, an ``MPCL`` whose ``num_class``
    is not ``num_class``, ``num_class`` outside [2, 8], or a mailbox too small for ``2 K (C+1)`` words; the separate
    calls remain the route for those."""
    from .seg import _resolve_group
    from ._lib import MAX_CLASSES
    from .peer import PeerMailbox
    k = int(num_class)
    if not (2 <= k <= MAX_CLASSES):
        raise ValueError(f"mpscl_step: num_class must be in [2, {MAX_CLASSES}], got {k}")
    for name, mod in (("mpcl_src", mpcl_src), ("mpcl_trg", mpcl_trg)):
        if not isinstance(mod, MPCL):
            raise TypeError(f"mpscl_step: {name} must be an slcl.loss.MPCL")
        if mod.num_class != k:
            raise ValueError(f"mpscl_step: {name}.num_class is {mod.num_class}, num_class is {k}")
    for name, t in (("ft_s", ft_s), ("ft_t", ft_t)):
        if not isinstance(t, torch.Tensor) or t.dim() != 4 or t.dtype != torch.float32 or not t.is_contiguous():
            raise ValueError(f"mpscl_step: {name} must be a contiguous float32 [B, C, h, w] map")
    b_s, c, h, w = ft_s.shape
    if ft_t.shape[1] != c:
        raise ValueError(f"mpscl_step: ft_t has {ft_t.shape[1]} channels, ft_s has {c}")
    if tuple(ft_t.shape[2:]) != (h, w):
        raise ValueError(f"mpscl_step: ft_t is {tuple(ft_t.shape[2:])}, ft_s is {(h, w)}: the maps share one resolution")
    if tuple(labels_s.shape[-2:]) != (h, w) or labels_s.numel() != b_s * h * w:
        raise ValueError(f"mpscl_step: labels_s must be [B, h, w] = {(b_s, h, w)} at the feature resolution "
                         f"(update_class_center_iter, utils/utils_.py:575-577), got {tuple(labels_s.shape)}")
    if not isinstance(class_center_feas, torch.Tensor) or tuple(class_center_feas.shape) != (k, c):
        raise ValueError(f"mpscl_step: class_center_feas must be [num_class, C] = {(k, c)}, "
                         f"got {tuple(getattr(class_center_feas, 'shape', ()))}")
    if class_center_feas.requires_grad:
        raise ValueError("mpscl_step: class_center_feas requires grad; the step's centres are a plain tensor (the "
                         "separate calls keep the graph through m * class_center_feas)")
    group = _resolve_group(group)
    if isinstance(group, PeerMailbox) and group.capacity_words < 2 * k * (c + 1):
        raise ValueError(f"mpscl_step: the class sums are {k} x {c + 1} doubles; the mailbox needs capacity_words >= "
                         f"{2 * k * (c + 1)}, this one has {group.capacity_words}")
    labels = labels_s.to(ft_s.device).reshape(-1).long()
    const = lambda mod: (float(mod.temperature), float(mod.base_temperature), float(mod.m), bool(mod.easy_margin))
    return SF.mpscl_step(ft_s, labels, ft_t, class_center_feas, m=m, sel_threshold=pixel_sel_th, n_class=k,
                         const_s=const(mpcl_src), const_t=const(mpcl_trg), group=group)


SupConLoss = p2p.SupConLoss
LocalConLoss = p2p.LocalConLoss
BlockConLoss = p2p.BlockConLoss
