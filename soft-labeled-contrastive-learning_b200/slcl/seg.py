"""Segmentation losses next to the contrastive path (SURVEY.md 8(f)-2): drop-ins for the reference's
``loss_calc`` / ``jaccard_loss`` / ``dice_loss`` (utils/loss.py:11-103) and ``prob_2_entropy``
(utils/utils_.py:627-631).  One fused CUDA pass over the logits computes cross entropy, Dice and Jaccard
together (``seg_losses``); the drop-in functions pick what they need from it.  With ``group=`` they return the losses of
the global batch of data-parallel ranks (see ``seg_losses``)."""
from __future__ import annotations

import torch

from . import ops  # noqa: F401
from ._lib import MAX_CLASSES as _MAX_CLASSES
from .peer import PeerMailbox

_ops = ops.dispatch          # eager: op bodies directly; compiled: torch.ops.slcl


class _SegLosses(torch.autograd.Function):
    @staticmethod
    def forward(ctx, logits, labels, group):
        if group is None:
            losses, stats = _ops.seg_fwd(logits.detach(), labels)
            vec = None
        elif isinstance(group, PeerMailbox):          # exchanged inside the finaliser kernel
            losses, stats, vec = _ops.seg_fwd_peer(logits.detach(), labels, *group.args())
        else:                                         # NCCL: local vector -> all-reduce -> finishing kernel
            from .distributed import all_reduce_sums
            stats, vec = _ops.seg_fwd_local(logits.detach(), labels)
            vec = all_reduce_sums(vec, group)
            losses = _ops.seg_finish(vec, logits.shape[1])
        ctx.save_for_backward(logits, labels, stats, vec)
        return losses

    @staticmethod
    def backward(ctx, grad_losses):
        logits, labels, stats, vec = ctx.saved_tensors
        if not ctx.needs_input_grad[0]:
            return None, None, None
        if vec is None:
            return _ops.seg_bwd(logits.detach(), labels, stats, grad_losses.contiguous()), None, None
        return _ops.seg_bwd_global(logits.detach(), labels, stats, vec, grad_losses.contiguous()), None, None


def _resolve_group(group):
    """None (today's single-rank path) for no group, a world of one, or True without an initialised process group;
    else the PeerMailbox, True or the ProcessGroup."""
    if group is None:
        return None
    if isinstance(group, PeerMailbox):
        return group if group.world > 1 else None
    import torch.distributed as dist
    if group is not True and not (dist.is_available() and isinstance(group, dist.ProcessGroup)):
        raise TypeError(f"group must be None, True, a ProcessGroup or a slcl.peer.PeerMailbox, got {type(group).__name__}")
    if not dist.is_available() or not dist.is_initialized():
        return None
    return group if dist.get_world_size(None if group is True else group) > 1 else None


def _check_global_inputs(pred, label, group):
    """Shape checks of the group= path, made before anything is exchanged (a rank that raised after its peers had sent
    would leave them waiting)."""
    if pred.dim() != 4 or pred.dtype != torch.float32:
        raise ValueError("group= segmentation losses: pred must be float32 [B, K, H, W]")
    b, k, h, w = pred.shape
    if label.numel() != b * h * w:
        raise ValueError(f"group= segmentation losses: label must hold [B, H, W] = [{b}, {h}, {w}] values, "
                         f"got shape {tuple(label.shape)}")
    if k > _MAX_CLASSES:
        raise ValueError(f"segmentation losses support at most {_MAX_CLASSES} classes, got {k}")
    if isinstance(group, PeerMailbox) and group.capacity_words < 2 * ops.seg_vec_len(k):
        raise ValueError(f"group= segmentation losses over {k} classes need a mailbox with capacity_words >= "
                         f"{2 * ops.seg_vec_len(k)}, this one has {group.capacity_words}")


def seg_losses(pred: torch.Tensor, label: torch.Tensor, *, group=None) -> torch.Tensor:
    """[3] tensor {cross entropy, dice loss, jaccard loss} of logits ``pred`` [B,K,H,W] vs ``label`` [B,H,W]
    (or [B,1,H,W]) in one pass; differentiable w.r.t. ``pred``.

    ``group`` (addition): the batch is sharded over data-parallel ranks and the result is the three losses of the ranks'
    batches concatenated in rank order, identical bits on every rank; ``pred.grad`` is this rank's shard of the gradient.
    ``None`` or a world of one: the single-rank call.  ``True`` / a ProcessGroup: one NCCL all-reduce of 2K + 4 doubles.
    A ``slcl.peer.PeerMailbox``: the same sums exchanged inside the forward's finaliser kernel over NVLink peer memory (no
    collective, no host synchronisation).  Ranks may hold different batch sizes; K, H and W must agree.  The backward
    exchanges nothing.  All three losses come from ONE pass and ONE exchange, so a caller that needs two of them (CE +
    Dice, CE + Jaccard) calls this once rather than ``loss_calc`` and ``dice_loss`` (one exchange each)."""
    if pred.shape[1] < 2:
        raise NotImplementedError("num_classes == 1 (sigmoid branch of jaccard_loss, utils/loss.py:23-32) is not built")
    group = _resolve_group(group)
    if group is not None:
        _check_global_inputs(pred, label, group)
    return _SegLosses.apply(pred, label.to(pred.device), group)


def loss_calc(pred, label, gpu=0, jaccard=False, *, group=None):
    """utils/loss.py:46-66: CrossEntropyLoss (+ jaccard_loss).  ``group``: as ``seg_losses``."""
    out = seg_losses(pred, label, group=group)
    return out[0] + out[2] if jaccard else out[0]


def jaccard_loss(true, logits, eps=1e-7, *, group=None):
    """utils/loss.py:11-43 (eps is fixed at the reference default 1e-7).  ``group``: as ``seg_losses``."""
    if eps != 1e-7:
        raise NotImplementedError("jaccard_loss: only the reference default eps=1e-7 is built")
    return seg_losses(logits, true, group=group)[2]


def dice_loss(pred, target, *, group=None):
    """utils/loss.py:69-103.  ``group``: as ``seg_losses``."""
    return seg_losses(pred, target, group=group)[1]


class _EntropyMap(torch.autograd.Function):
    @staticmethod
    def forward(ctx, prob):
        ctx.save_for_backward(prob)
        return _ops.entropy_map(prob.detach())

    @staticmethod
    def backward(ctx, grad_out):
        (prob,) = ctx.saved_tensors
        return _ops.entropy_map_bwd(prob.detach(), grad_out.contiguous())


class _EntropyMapLogits(torch.autograd.Function):
    """The map from logits; saves the logits only and recomputes the softmax in the backward."""
    @staticmethod
    def forward(ctx, logits):
        ctx.save_for_backward(logits)
        return _ops.entropy_map_logits(logits.detach())

    @staticmethod
    def backward(ctx, grad_out):
        (logits,) = ctx.saved_tensors
        return _ops.entropy_map_logits_bwd(logits.detach(), grad_out)


def prob_2_entropy(prob, from_logits=False):
    """utils/utils_.py:627-631: weighted self-information map -p log2(p + 1e-7) / log2(C) of [N,C,H,W] probabilities.

    ``from_logits`` (addition): ``prob`` holds float32 logits [B, K, H, W] (2 <= K <= 8) and the call returns
    ``prob_2_entropy(torch.softmax(prob, 1))``, the gradient flowing into the logits; the softmax runs inside the map's
    forward and backward kernels (Trainer_MPSCL.py:171-172 without the ``F.softmax``)."""
    if not from_logits:
        return _EntropyMap.apply(prob)
    ops.check_entropy_logits(prob)
    if torch.is_grad_enabled() and prob.requires_grad:
        return _EntropyMapLogits.apply(prob)
    return _ops.entropy_map_logits(prob)
