"""Autograd wiring of the slcl custom ops (fused forward + closed-form backward).

Formulas: SURVEY.md appendix A; reference functions cited per class.
"""
from __future__ import annotations

from typing import List, Optional, Sequence, Tuple

import torch
from torch import Tensor

from . import ops  # noqa: F401  (registers torch.ops.slcl.*)

_ops = ops.dispatch          # eager: op bodies directly; compiled: torch.ops.slcl


def _peer_args(group):
    """The flat mailbox arguments when `group` is a PeerMailbox over more than one rank (the forward kernels then do the
    loss-pair exchange themselves, inside their finaliser), else ()."""
    from .peer import PeerMailbox
    if isinstance(group, PeerMailbox) and group.world > 1:
        return group.args()
    return ()


def _exchange_loss_pair(scal, has_sel: bool, group) -> None:
    """Data-parallel prototype loss: global mean = summed numerator / summed denominator (SURVEY.md 8(e)).
    ``group``: None (single process), True / a ProcessGroup (NCCL all-reduce of scal[2:4] + rescale), or a
    ``slcl.peer.PeerMailbox`` (exchange + rescale as ONE kernel over NVLink peer memory)."""
    if group is None:
        return
    from .peer import PeerMailbox
    if isinstance(group, PeerMailbox):
        return                       # exchanged inside the forward's finaliser kernel (_peer_args)
    import torch.distributed as dist
    if dist.is_initialized() and dist.get_world_size(None if group is True else group) > 1:
        dist.all_reduce(scal[2:4], op=dist.ReduceOp.SUM, group=None if group is True else group)
        _ops.proto_rescale(scal, has_sel)


class _ProtoLoss(torch.autograd.Function):
    """MPCL.forward (+ the normalise/layout work of mpcl_loss_calc): reference
    utils/loss.py:484-573, :592-601.  Backward: appendix A.1."""

    @staticmethod
    def forward(ctx, feat, labels, soft_mask, sel, centres, rows_layout, n_class, temperature, base_temperature, margin,
                easy_margin, normalize, group):
        scal, stash, cstate = _ops.proto_fwd(feat.detach(), labels, None if soft_mask is None else soft_mask.detach(),
                                             None if sel is None else sel.detach(), centres.detach(), rows_layout,
                                             n_class, temperature, base_temperature, margin, easy_margin, normalize,
                                             *_peer_args(group))
        _exchange_loss_pair(scal, sel is not None, group)
        ctx.soft = soft_mask is not None and soft_mask.requires_grad
        ctx.sel_grad = sel is not None and sel.requires_grad
        aux = ctx.soft or ctx.sel_grad          # (no reference caller differentiates these two: keep them only when asked)
        ctx.save_for_backward(feat, stash, cstate, scal, labels if aux else None, soft_mask if aux else None,
                              sel if aux else None)
        ctx.cfg = (rows_layout, n_class, normalize, temperature, base_temperature, margin, easy_margin)
        return scal[0]

    @staticmethod
    def backward(ctx, grad_out):
        feat, stash, cstate, scal, labels, soft_mask, sel = ctx.saved_tensors
        rows_layout, n_class, normalize, temperature, base_temperature, margin, easy_margin = ctx.cfg
        g = grad_out.reshape(1)
        dfeat = dcen = dmask = dsel = None
        if ctx.needs_input_grad[0]:
            dfeat = _ops.proto_bwd(feat.detach(), stash, cstate, scal, g, rows_layout, n_class, normalize)
        if ctx.needs_input_grad[4]:
            dcen = _ops.proto_bwd_centres(feat.detach(), stash, cstate, scal, g, rows_layout, n_class, normalize)
        if ctx.soft or ctx.sel_grad:          # utils/loss.py:516-517 / :558-565 as differentiable inputs: one more pass over feat
            dm, ds = _ops.proto_bwd_aux(feat.detach(), labels, None if soft_mask is None else soft_mask.detach(),
                                        None if sel is None else sel.detach(), cstate, scal, g, rows_layout, n_class,
                                        temperature, base_temperature, margin, easy_margin, normalize, ctx.soft, ctx.sel_grad)
            if ctx.soft:
                dmask = dm.reshape(soft_mask.shape).to(soft_mask.dtype)
            if ctx.sel_grad:
                dsel = ds.reshape(sel.shape).to(sel.dtype)
        return dfeat, None, dmask, dsel, dcen, None, None, None, None, None, None, None, None


class _ProtoTargetStep(torch.autograd.Function):
    """generate_pseudo_label + target mpcl_loss_calc fused (trainer/Trainer_MPSCL.py:135,144): one read of the
    target map in the forward; backward identical to _ProtoLoss."""

    @staticmethod
    def forward(ctx, feat, centres, sel_threshold, n_class, temperature, base_temperature, margin, easy_margin, group):
        scal, stash, cstate, label, sel = _ops.proto_fwd_target(feat.detach(), centres.detach(), sel_threshold, n_class,
                                                                temperature, base_temperature, margin, easy_margin,
                                                                *_peer_args(group))
        _exchange_loss_pair(scal, True, group)
        ctx.save_for_backward(feat, stash, cstate, scal)
        ctx.n_class = n_class
        ctx.mark_non_differentiable(label, sel)
        return scal[0], label, sel

    @staticmethod
    def backward(ctx, grad_out, _gl, _gs):
        feat, stash, cstate, scal = ctx.saved_tensors
        dfeat = None
        if ctx.needs_input_grad[0]:
            dfeat = _ops.proto_bwd(feat.detach(), stash, cstate, scal, grad_out.reshape(1), False, ctx.n_class, True)
        return dfeat, None, None, None, None, None, None, None, None


class _ProtoTargetStepCentroids(torch.autograd.Function):
    """The fused target step that also returns the hard target centroids of the map under its own pseudo labels
    (SURVEY.md 8(f)-1; trainer/Trainer_MPSCL.py:135,144 + cal_centroid, utils/utils_.py:524-529): ONE pass over the target
    map in the forward (slcl_target_step).  Backward: prototype-loss backward + centroid backward (appendix A.1 / A.4)."""

    @staticmethod
    def forward(ctx, feat, centres, previous, sel_threshold, weight_by_sel, n_class, temperature, base_temperature, margin,
                easy_margin, momentum, group):
        from .peer import PeerMailbox
        prev = None if previous is None else previous.detach()
        peer_ok = group is None or isinstance(group, PeerMailbox)
        if peer_ok and ops.target_step_supported(feat, n_class):
            peer = group.args() if group is not None else ()
            scal, stash, cstate, label, sel, sums, cen, _ = _ops.target_step(
                feat.detach(), centres.detach(), sel_threshold, weight_by_sel, n_class, temperature, base_temperature, margin,
                easy_margin, prev, momentum, *peer)
            wlab = torch.where(sel > 0, label, torch.full_like(label, -1)) if weight_by_sel else label
        else:       # shapes outside the tile kernel, or an NCCL group: the separate kernels (two reads of the map)
            scal, stash, cstate, label, sel = _ops.proto_fwd_target(feat.detach(), centres.detach(), sel_threshold, n_class,
                                                                    temperature, base_temperature, margin, easy_margin,
                                                                    *_peer_args(group))
            wlab = torch.where(sel > 0, label, torch.full_like(label, -1)) if weight_by_sel else label
            if peer_ok:
                cen, _, sums = _ops.centroids_fwd(feat.detach(), wlab, None, False, 0.0, None, 1, n_class, prev, momentum,
                                                  *(group.args() if group is not None else ()))
            else:
                from .distributed import all_reduce_sums
                sums = all_reduce_sums(_ops.class_sums(feat.detach(), wlab, None, False, 0.0, None, 1, n_class), group)
                cen, _ = _ops.centroid_finalize(sums, prev, momentum, 1, n_class)
        _exchange_loss_pair(scal, True, group)
        ctx.save_for_backward(feat, stash, cstate, scal, wlab, sums)
        ctx.cfg = (n_class, momentum, previous is not None)
        ctx.mark_non_differentiable(label, sel)
        return scal[0], label, sel, cen

    @staticmethod
    def backward(ctx, g_loss, _gl, _gs, g_cen):
        feat, stash, cstate, scal, wlab, sums = ctx.saved_tensors
        n_class, momentum, has_prev = ctx.cfg
        dfeat = dprev = None
        if ctx.needs_input_grad[0]:
            dfeat = _ops.proto_bwd(feat.detach(), stash, cstate, scal, g_loss.reshape(1), False, n_class, True)
            dcen, _ = _ops.centroid_bwd(feat.detach(), wlab, None, False, 0.0, None, 1, n_class, g_cen.contiguous(), sums,
                                        (1.0 - momentum) if has_prev else 1.0, False)
            dfeat = dfeat + dcen
        if has_prev and ctx.needs_input_grad[2]:
            dprev = momentum * g_cen
        return dfeat, None, dprev, None, None, None, None, None, None, None, None, None


def proto_target_step_centroids(feat: Tensor, centres: Tensor, previous: Optional[Tensor], sel_threshold: float, *,
                                weight_by_sel: bool, n_class: int, temperature: float, base_temperature: float, margin: float,
                                easy_margin: bool, momentum: float, group=None):
    return _ProtoTargetStepCentroids.apply(feat, centres, previous, float(sel_threshold), bool(weight_by_sel), n_class,
                                           temperature, base_temperature, margin, easy_margin, float(momentum), group)


def proto_target_step(feat: Tensor, centres: Tensor, sel_threshold: float, *, n_class: int, temperature: float,
                      base_temperature: float, margin: float, easy_margin: bool, group=None):
    return _ProtoTargetStep.apply(feat, centres, float(sel_threshold), n_class, temperature, base_temperature, margin,
                                  easy_margin, group)


def proto_loss(feat: Tensor, labels: Optional[Tensor], soft_mask: Optional[Tensor], sel: Optional[Tensor], centres: Tensor,
               *, rows_layout: bool, n_class: int, temperature: float, base_temperature: float, margin: float,
               easy_margin: bool, normalize: bool, group=None) -> Tensor:
    return _ProtoLoss.apply(feat, labels, soft_mask, sel, centres, rows_layout, n_class, temperature, base_temperature,
                            margin, easy_margin, normalize, group)


class _Centroids(torch.autograd.Function):
    """cal_centroid (reference utils/utils_.py:479-565, repaired; partitions per
    SURVEY.md 8(c)-2).  Forward = class sums (+ optional cross-rank all-reduce)
    + finalise; backward = appendix A.4.  from_logits: ``probs`` holds logits, the kernels apply the softmax and the
    backward returns dL/dlogits in its slot."""

    @staticmethod
    def forward(ctx, feat, labels, probs, previous, weighted, threshold, part_id, n_partitions, n_class, momentum, group,
                from_logits):
        from .peer import PeerMailbox
        prev = None if previous is None else previous.detach()
        if group is None or isinstance(group, PeerMailbox):
            # two launches: sweep, then reduce [+ exchange over the NVLink peer mailboxes] + finalise
            peer = group.args() if group is not None else ()
            cen, _inv_w, sums = _ops.centroids_fwd(feat.detach(), labels, None if probs is None else probs.detach(), weighted,
                                                   threshold, part_id, n_partitions, n_class, prev, momentum, *peer,
                                                   from_logits=from_logits)
        else:
            from .distributed import all_reduce_sums
            sums = _ops.class_sums(feat.detach(), labels, None if probs is None else probs.detach(), weighted, threshold,
                                   part_id, n_partitions, n_class, from_logits)
            sums = all_reduce_sums(sums, group)
            cen, _inv_w = _ops.centroid_finalize(sums, prev, momentum, n_partitions, n_class)
        ctx.save_for_backward(feat, labels, probs, part_id, sums)
        ctx.cfg = (weighted, threshold, n_partitions, n_class, momentum, previous is not None, from_logits)
        return cen

    @staticmethod
    def backward(ctx, grad_cen):
        feat, labels, probs, part_id, sums = ctx.saved_tensors
        weighted, threshold, n_partitions, n_class, momentum, has_prev, from_logits = ctx.cfg
        ema_scale = (1.0 - momentum) if has_prev else 1.0
        dfeat = dprobs = dprev = None
        need_dp = probs is not None and ctx.needs_input_grad[2] and weighted
        if ctx.needs_input_grad[0] or need_dp:
            dfeat, dp = _ops.centroid_bwd(feat.detach(), labels, None if probs is None else probs.detach(), weighted,
                                          threshold, part_id, n_partitions, n_class, grad_cen.contiguous(), sums,
                                          ema_scale, need_dp, from_logits)
            if need_dp:
                dprobs = dp
            if not ctx.needs_input_grad[0]:
                dfeat = None
        if has_prev and ctx.needs_input_grad[3]:
            dprev = momentum * grad_cen.reshape(n_partitions, n_class, -1).sum(0)
        return dfeat, None, dprobs, dprev, None, None, None, None, None, None, None, None


def centroids(feat: Tensor, labels: Optional[Tensor], probs: Optional[Tensor], previous: Optional[Tensor], *,
              weighted: bool, threshold: float, part_id: Optional[Tensor], n_partitions: int, n_class: int,
              momentum: float, group=None, from_logits: bool = False) -> Tensor:
    """-> [P*K, C] centroids (EMA'd with `previous` when given).  ``from_logits``: ``probs`` are the logits whose
    softmax over dim 1 is the soft label; its gradient is dL/dlogits."""
    return _Centroids.apply(feat, labels, probs, previous, weighted, threshold, part_id, n_partitions, n_class, momentum,
                            group, bool(from_logits))


class _CentroidLoss(torch.autograd.Function):
    """ContrastiveLoss.forward (utils/loss.py:241-275) / CNR (Trainer_MCCL.py:303-315):
    one launch yields the loss and both gradients (appendix A.5)."""

    @staticmethod
    def forward(ctx, cs, ct, mode, first_row, n_rows, norm):
        loss, ds, dt = _ops.centroid_loss(cs.detach(), ct.detach(), mode, first_row, n_rows, norm)
        ctx.save_for_backward(ds, dt)
        return loss[0]

    @staticmethod
    def backward(ctx, grad_out):
        ds, dt = ctx.saved_tensors
        return (grad_out * ds if ctx.needs_input_grad[0] else None,
                grad_out * dt if ctx.needs_input_grad[1] else None, None, None, None, None)


def centroid_loss(cs: Tensor, ct: Tensor, *, mode: int, first_row: int, n_rows: int, norm: bool) -> Tensor:
    return _CentroidLoss.apply(cs, ct, mode, first_row, n_rows, norm)


class _McclLosses(torch.autograd.Function):
    """inter / intra ContrastiveLoss over the target partitions + CNR (trainer/Trainer_MCCL.py:303-326) as one op: the
    forward also produces every gradient (appendix A.5), the backward only scales them."""

    @staticmethod
    def forward(ctx, cs, ct_parts, ct_aug, n_partitions, split, bg, norm, inter_w, intra_w, cnr_w):
        losses, ds, dt, da = _ops.mccl_losses(cs.detach(), ct_parts.detach(), None if ct_aug is None else ct_aug.detach(),
                                              n_partitions, split, bg, norm, inter_w, intra_w, cnr_w)
        ctx.save_for_backward(ds, dt, da)
        ctx.has_aug = ct_aug is not None
        terms = losses[1:].detach()
        ctx.mark_non_differentiable(terms)
        return losses[0], terms

    @staticmethod
    def backward(ctx, g, _g_terms):
        ds, dt, da = ctx.saved_tensors
        return (g * ds if ctx.needs_input_grad[0] else None, g * dt if ctx.needs_input_grad[1] else None,
                g * da if (ctx.has_aug and ctx.needs_input_grad[2]) else None, None, None, None, None, None, None, None)


def mccl_losses(cs: Tensor, ct_parts: Tensor, ct_aug: Optional[Tensor], *, n_partitions: int, split: bool, bg: bool, norm: bool,
                inter_w: float, intra_w: float, cnr_w: float):
    return _McclLosses.apply(cs, ct_parts, ct_aug, int(n_partitions), bool(split), bool(bg), bool(norm), float(inter_w),
                             float(intra_w), float(cnr_w))


class _McclStep(torch.autograd.Function):
    """The MCCL loss section (trainer/Trainer_MCCL.py:275-326) as one node: source, target and augmented-target centroids
    and every centroid term in one forward call, the target maps' gradients in one backward call.  The source map gets no
    gradient (the trainer detaches the source centroids, :277)."""

    @staticmethod
    def forward(ctx, feat_s, labels_s, feat_t, pred_t, part_id, feat_a, pred_a, previous_s, n_partitions, n_class, weighted,
                threshold, from_logits, momentum, split, bg, norm, inter_w, intra_w, cnr_w, group):
        from .peer import PeerMailbox
        d = lambda t: None if t is None else t.detach()
        sets = (feat_s.detach(), labels_s, feat_t.detach(), pred_t.detach(), part_id, d(feat_a), d(pred_a))
        loss_cfg = (momentum, split, bg, norm, inter_w, intra_w, cnr_w)
        if group is None or isinstance(group, PeerMailbox):
            peer = group.args() if group is not None else ()
            losses, cen, sums, dcen = _ops.mccl_step_fwd(*sets, d(previous_s), n_partitions, n_class, weighted, threshold,
                                                         from_logits, *loss_cfg, *peer)
        else:       # NCCL: local sums -> one all-reduce -> the tail without the reduce
            from .distributed import all_reduce_sums
            sums = all_reduce_sums(_ops.mccl_step_fwd_local(*sets, n_partitions, n_class, weighted, threshold, from_logits),
                                   group)
            losses, cen, dcen = _ops.mccl_step_finish(sums, feat_a is not None, d(previous_s), n_partitions, n_class,
                                                      *loss_cfg)
        ctx.save_for_backward(feat_t, pred_t, part_id, feat_a, pred_a, sums, dcen)
        ctx.cfg = (n_partitions, n_class, weighted, threshold, from_logits)
        terms = losses[1:]
        ctx.mark_non_differentiable(terms, cen, sums)
        # the outputs other than `total` get no gradient: no zero tensors (one fill launch each) for their slots
        ctx.set_materialize_grads(False)
        return losses[0], terms, cen, sums

    @staticmethod
    def backward(ctx, g, _g_terms, _g_cen, _g_sums):
        feat_t, pred_t, part_id, feat_a, pred_a, sums, dcen = ctx.saved_tensors
        n_partitions, n_class, weighted, threshold, from_logits = ctx.cfg
        need = ctx.needs_input_grad
        if g is None or not (need[2] or need[3] or need[5] or need[6]):
            return (None,) * 21
        d = lambda t: None if t is None else t.detach()
        df_t, dp_t, df_a, dp_a = _ops.mccl_step_bwd(feat_t.detach(), pred_t.detach(), part_id, d(feat_a), d(pred_a),
                                                    n_partitions, n_class, weighted, threshold, from_logits, sums, dcen,
                                                    g.reshape(1), bool(need[3] or need[6]))
        pick = lambda t, i: t if (need[i] and t.numel()) else None
        return (None, None, pick(df_t, 2), pick(dp_t, 3), None, pick(df_a, 5), pick(dp_a, 6)) + (None,) * 14


def mccl_step(feat_s: Tensor, labels_s: Tensor, feat_t: Tensor, pred_t: Tensor, part_id: Optional[Tensor],
              feat_a: Optional[Tensor], pred_a: Optional[Tensor], previous_s: Optional[Tensor], *, n_partitions: int,
              n_class: int, weighted: bool, threshold: float, from_logits: bool, momentum: float, split: bool, bg: bool,
              norm: bool, inter_w: float, intra_w: float, cnr_w: float, group=None):
    """-> (total, terms [3], centroids [rows, C] (source | target partitions | aug), sums [rows, C+1] fp64)."""
    return _McclStep.apply(feat_s, labels_s, feat_t, pred_t, part_id, feat_a, pred_a, previous_s, int(n_partitions),
                           int(n_class), bool(weighted), float(threshold), bool(from_logits), float(momentum), bool(split),
                           bool(bg), bool(norm), float(inter_w), float(intra_w), float(cnr_w), group)


class _MpsclStep(torch.autograd.Function):
    """The MPSCL loss section (trainer/Trainer_MPSCL.py:133-147) as one node: EMA class centres from the source map, pseudo
    labels of the target map and both prototype losses in one forward call; dF_s and dF_t in one backward launch.  The
    centres, pseudo labels and mask get no gradient (the trainer detaches the centres, :138 / :144)."""

    @staticmethod
    def forward(ctx, feat_s, labels_s, feat_t, old_centres, m, sel_threshold, n_class, const_s, const_t, group):
        from .peer import PeerMailbox
        fs, ft = feat_s.detach(), feat_t.detach()
        if group is None or isinstance(group, PeerMailbox):
            peer = group.args() if group is not None else ()
            scal, centres, cstate, stash_s, stash_t, label, sel = _ops.mpscl_step_fwd(
                fs, labels_s, ft, old_centres.detach(), m, sel_threshold, n_class, *const_s, *const_t, *peer)
        else:       # NCCL: class sums -> all-reduce -> EMA, the local forward, one all-reduce of both pairs, the finish
            import torch.distributed as dist
            from .distributed import all_reduce_sums
            sums = all_reduce_sums(_ops.class_sums(fs, labels_s, None, False, 0.0, None, 1, n_class), group)
            centres = _ops.ema_finalize(sums, old_centres.detach(), m)
            pairs, cstate, stash_s, stash_t, label, sel = _ops.mpscl_step_fwd_local(fs, labels_s, ft, centres, sel_threshold,
                                                                                    n_class, *const_s, *const_t)
            dist.all_reduce(pairs, op=dist.ReduceOp.SUM, group=None if group is True else group)
            scal = _ops.mpscl_step_finish(pairs)
        ctx.save_for_backward(feat_s, feat_t, stash_s, stash_t, cstate, scal)
        ctx.n_class = n_class
        ctx.mark_non_differentiable(centres, label, sel)
        # only the losses carry gradients, and one of them may get none: no zero tensors for the other slots
        ctx.set_materialize_grads(False)
        return scal[0], scal[4], centres, label, sel

    @staticmethod
    def backward(ctx, g_s, g_t, _gc, _gl, _gm):
        feat_s, feat_t, stash_s, stash_t, cstate, scal = ctx.saved_tensors
        need = ctx.needs_input_grad
        g_s = g_s.reshape(1) if (g_s is not None and need[0]) else None
        g_t = g_t.reshape(1) if (g_t is not None and need[2]) else None
        if g_s is None and g_t is None:
            return (None,) * 10
        d_s, d_t = _ops.mpscl_step_bwd(feat_s.detach(), feat_t.detach(), stash_s, stash_t, cstate, scal, g_s, g_t,
                                       ctx.n_class)
        return (d_s if g_s is not None else None, None, d_t if g_t is not None else None) + (None,) * 7


def mpscl_step(feat_s: Tensor, labels_s: Tensor, feat_t: Tensor, old_centres: Tensor, *, m: float, sel_threshold: float,
               n_class: int, const_s: Sequence, const_t: Sequence, group=None):
    """-> (loss_s, loss_t, centres [K, C], hard [N_t] int64, mask [N_t]).  ``const_s`` / ``const_t``: (temperature,
    base_temperature, margin, easy_margin) of each loss."""
    return _MpsclStep.apply(feat_s, labels_s, feat_t, old_centres, float(m), float(sel_threshold), int(n_class),
                            tuple(const_s), tuple(const_t), group)
