"""Drop-in for the class-centre / centroid helpers of the reference's
``utils/utils_.py`` (:479-624)."""
from __future__ import annotations

from typing import Optional

import torch
import torch.nn.functional as F

from . import functional as SF
from . import ops

_ops = ops.dispatch          # eager: op bodies directly; compiled: torch.ops.slcl


def update_class_center_iter(cla_src_feas, batch_src_labels, class_center_feas, m=.2, num_class=4, group=None):
    """EMA class centres (reference utils/utils_.py:568-594).  One pass over the
    map instead of ``num_class`` masked passes; the empty-class rule (:585-588) is
    decided on the device, so there is no host sync.  ``group``: optional
    torch.distributed group -- the per-class sums/counts are all-reduced so every
    rank holds the centres of the global batch (SURVEY.md 8(e)); a ``slcl.peer.PeerMailbox`` does that exchange inside
    the reduce kernel over NVLink peer memory (no collective launch)."""
    feats = cla_src_feas.detach()
    labels = batch_src_labels.to(feats.device)
    if labels.shape != (feats.shape[0],) + tuple(feats.shape[2:]):
        raise ValueError("labels must be [B, h, w] at feature resolution")
    from .peer import PeerMailbox
    old = class_center_feas[:num_class]
    lab = labels.reshape(-1).long()
    if group is None or isinstance(group, PeerMailbox):
        # two launches: sweep, then reduce [+ exchange over the NVLink peer mailboxes] + EMA finalise
        new, _sums = _ops.class_centres_update(feats, lab, old.detach(), float(m), *(group.args() if group is not None else ()))
    else:
        from .distributed import all_reduce_sums
        sums = all_reduce_sums(_ops.class_sums(feats, lab, None, False, 0.0, None, 1, num_class), group)
        new = _ops.ema_finalize(sums, old.detach(), float(m))
    if class_center_feas.requires_grad:
        # the reference keeps the graph through `m * class_center_feas` (:592) and detaches the
        # old centre only in the empty-class branch (:586)
        new = new + m * (old - old.detach())
    return new


def generate_pseudo_label(cla_feas_trg, class_centers, pixel_sel_th=.25):
    """arg-max cosine label + (top1 - top2 > th) mask (reference utils/utils_.py:597-624)."""
    label, sel = _ops.pseudo_label(cla_feas_trg.detach(), class_centers.detach(), float(pixel_sel_th))
    return label, sel


def rmc_partition_ids(n_pixels: int, partition: int, generator: Optional[torch.Generator] = None,
                      device=None) -> torch.Tensor:
    """Reversed-Monte-Carlo partition assignment (spec: SURVEY.md 8(c)-2; the
    reference fork has no sampler).  Drawn from PyTorch's RNG stream --
    ``torch.randperm(N, generator) % P`` in (b, h, w) pixel order -- so the CUDA
    path consumes exactly the indices a PyTorch restatement sees.  Without a
    generator the draw runs on ``device`` (torch's CUDA RNG: no host round trip);
    a generator is used on its own device."""
    if generator is not None:
        gen_dev = generator.device                    # the generator decides where the draw happens
    else:
        gen_dev = torch.device(device) if device is not None else torch.device("cpu")      # default: on the map's device
    perm = torch.randperm(n_pixels, generator=generator, device=gen_dev)
    ids = (perm % partition).to(torch.int32)
    return ids if device is None else ids.to(device)


def cal_centroid(decoder_ft, label, previous_centroid=None, momentum=0.95, pseudo_label=False, n_class=4, partition=1,
                 threshold: int = None, thd_w: float = 0.0, weighted_ave=False, epoch=0, max_epoch=1000,
                 low_thd=0, high_thd=0.99, stdmin=False, part_id=None, generator=None, group=None, from_logits=False):
    """Per-class (soft-label weighted) feature centroids (reference
    utils/utils_.py:479-565, with the repair of SURVEY.md section 0).

    Same positional/keyword arguments and return triple ``(centroids, ratio,
    stddevs)`` as the reference (``ratio`` is None and ``stddevs`` is [] there
    too, :565).  ``partition > 1`` returns a list of P ``[K,C]`` tensors (what
    trainer/Trainer_MCCL.py:281-326 consumes); the partition of every pixel
    comes from ``part_id`` or is drawn with ``rmc_partition_ids(generator)``.
    Extra keywords (``part_id``, ``generator``, ``group``, ``from_logits``) are additions.

    ``from_logits=True`` takes the segmentor's logits ``[B, K, h, w]`` at the feature map's resolution as ``label`` and
    returns what ``cal_centroid(decoder_ft, softmax(label, 1), pseudo_label=True, ...)`` returns, gradients included
    (into the logits), with the softmax done inside the class-sum and backward kernels.  It needs ``pseudo_label=True``.
    Logits at another resolution: interpolating probabilities does not commute with the softmax, so call ``softmax``
    and this function without ``from_logits``.
    """
    b, c, h, w = decoder_ft.shape
    if from_logits:
        if not pseudo_label:
            raise ValueError("from_logits=True needs pseudo_label=True (logits are soft labels)")
        if tuple(label.shape) != (b, n_class, h, w):
            raise ValueError(f"from_logits=True needs logits [B, K, h, w] = {(b, n_class, h, w)} at the feature map's "
                             f"resolution, got {tuple(label.shape)}")
    lab = label
    if not pseudo_label and (lab.shape[-1] != w or lab.shape[-2] != h):                 # :498-502
        if lab.ndim == 3:
            lab = lab.unsqueeze(1)
        lab = F.interpolate(lab.float(), size=(h, w), mode='nearest').long().squeeze(1)
    if pseudo_label and (lab.shape[-1] != w or lab.shape[-2] != h):                     # :503-505
        if lab.ndim == 3:
            raise ValueError("Soft pseudo-label must have channel dimension K")
        lab = F.interpolate(lab, size=(h, w), mode='bilinear', align_corners=False)

    n_part = int(partition) if (pseudo_label and partition > 1) else 1
    if n_part > 1:
        if part_id is None:
            part_id = rmc_partition_ids(b * h * w, n_part, generator, decoder_ft.device)
        part_id = part_id.to(device=decoder_ft.device, dtype=torch.int32).reshape(-1)
    else:
        part_id = None

    prev = None
    if previous_centroid is not None:                                                   # :552-563
        if isinstance(previous_centroid, torch.Tensor) and n_part == 1 and previous_centroid.shape == (n_class, c):
            prev = previous_centroid
        elif isinstance(previous_centroid, (list, tuple)) and n_part > 1 and len(previous_centroid) == n_part:
            prev = list(previous_centroid)
        else:
            print(f"Warning: Shape/type mismatch for EMA. Prev type: {type(previous_centroid)}")

    thr = float(threshold) if (pseudo_label and threshold is not None) else 0.0
    if pseudo_label:
        cen = SF.centroids(decoder_ft, None, lab, prev if isinstance(prev, torch.Tensor) else None,
                           weighted=bool(weighted_ave), threshold=thr, part_id=part_id, n_partitions=n_part,
                           n_class=n_class, momentum=float(momentum), group=group, from_logits=bool(from_logits))
    else:
        cen = SF.centroids(decoder_ft, lab.reshape(-1).long(), None, prev if isinstance(prev, torch.Tensor) else None,
                           weighted=False, threshold=0.0, part_id=None, n_partitions=1, n_class=n_class,
                           momentum=float(momentum), group=group)
    if n_part > 1:
        out = [cen[p * n_class:(p + 1) * n_class] for p in range(n_part)]
        if isinstance(prev, list):
            out = [momentum * prev[p] + (1 - momentum) * out[p] for p in range(n_part)]
    else:
        out = cen
    return out, None, []
