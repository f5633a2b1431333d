"""torch custom ops (``torch.ops.slcl.*``) over the C ABI of libslcl.so.

Each op allocates its outputs and workspace with torch (caching allocator),
then makes ONE call into the C ABI on the current CUDA stream.  The ops carry
no autograd formulas; the autograd wiring lives in ``slcl.functional``.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional, Tuple

import torch
from torch import Tensor

from . import _lib
from ._lib import MapT, PeerT, ProtoParamsT, check, ptr, require_cuda, stream_ptr

_F32 = torch.float32


class _NoGuard:
    def __enter__(self):
        return None

    def __exit__(self, *a):
        return False


_NOGUARD = _NoGuard()


def _guard(dev):
    """Device guard only when the tensor's device is not the current one."""
    if dev.index is None or torch.cuda.current_device() == dev.index:
        return _NOGUARD
    return torch.cuda.device(dev)


def _ws(nbytes: int, device) -> Tensor:
    return torch.empty(max(int(nbytes), 256), dtype=torch.uint8, device=device)


def _map_nchw(feat: Tensor) -> Tuple[Tensor, MapT]:
    """[B,C,H,W] -> (tensor actually read, strided map).  H and W must collapse
    into one pixel stride; anything else is made contiguous first."""
    if feat.dim() != 4:
        raise ValueError("feature map must be [B, C, H, W]")
    b, c, h, w = feat.shape
    sb, sc, sh, sw = feat.stride()
    if feat.dtype != _F32:
        raise ValueError("slcl kernels compute in fp32; pass a float32 feature map")
    if sw != 1 or (h > 1 and sh != w) or sc < h * w or (b > 1 and sb < c * h * w):
        feat = feat.contiguous()
        sb, sc = c * h * w, h * w
    return feat, MapT(b, c, h * w, sb, sc, 1)


def _map_rows(rows: Tensor) -> Tuple[Tensor, MapT]:
    """[N,C] row-major rows (the layout MPCL.forward receives) as a map with B=1."""
    if rows.dim() != 2:
        raise ValueError("rows must be [N, C]")
    if rows.dtype != _F32:
        raise ValueError("slcl kernels compute in fp32; pass float32 rows")
    rows = rows.contiguous()
    n, c = rows.shape
    return rows, MapT(1, c, n, 0, 1, c)


def _params(n_class: int, temperature: float, base_temperature: float, margin: float, easy_margin: bool,
            normalize: bool) -> ProtoParamsT:
    return ProtoParamsT(int(n_class), float(temperature), float(base_temperature), float(margin),
                        int(bool(easy_margin)), int(bool(normalize)))


def _feat_map(feat: Tensor, rows_layout: bool):
    return _map_rows(feat) if rows_layout else _map_nchw(feat)


# ----------------------------------------------------------------------------
# prototype path
# ----------------------------------------------------------------------------
def _peer(peer_ptrs: int, rank: int, world: int, capacity_words: int, timeout_s: float) -> Optional[PeerT]:
    """slcl_peer_t from the flat (ptrs, rank, world, capacity, timeout) form ops carry (slcl.peer.PeerMailbox.args());
    world <= 1 or a null pointer table = no exchange."""
    if world <= 1 or not peer_ptrs:
        return None
    return PeerT(peer_ptrs, rank, world, capacity_words, timeout_s)


@torch.library.custom_op("slcl::proto_fwd", mutates_args=(), device_types="cuda")
def proto_fwd(feat: Tensor, labels: Optional[Tensor], soft_mask: Optional[Tensor], sel: Optional[Tensor],
              centres: Tensor, rows_layout: bool, n_class: int, temperature: float, base_temperature: float,
              margin: float, easy_margin: bool, normalize: bool, peer_ptrs: int = 0, rank: int = 0, world: int = 1,
              capacity_words: int = 0, timeout_s: float = 0.0) -> Tuple[Tensor, Tensor, Tensor]:
    """-> (scal[4] = {loss, coef, weight sum, row-loss sum}, stash[(K+1), N], cstate[K*C+K]).  With a peer mailbox
    (slcl.peer.PeerMailbox.args()) the finaliser exchanges the loss pair with the other ranks: scal is GLOBAL."""
    dev = require_cuda(feat, labels, soft_mask, sel, centres)
    lib = _lib.load()
    feat_c, m = _feat_map(feat, rows_layout)
    n = m.batch * m.pixels
    if labels is not None:
        labels = labels.contiguous()
        if labels.dtype != torch.int64:
            raise ValueError("labels must be int64")
    if soft_mask is not None:
        soft_mask = soft_mask.to(_F32).contiguous()
    if sel is not None:
        sel = sel.to(_F32).contiguous()
    centres = centres.to(_F32).contiguous()
    scal = torch.empty(4, dtype=_F32, device=dev)
    stash = torch.empty((n_class + 1, n), dtype=_F32, device=dev)
    cstate = torch.empty(n_class * m.channels + n_class, dtype=_F32, device=dev)
    nbytes = lib.slcl_proto_workspace_bytes(n)
    ws = _ws(nbytes, dev)
    p = _params(n_class, temperature, base_temperature, margin, easy_margin, normalize)
    peer = _peer(peer_ptrs, rank, world, capacity_words, timeout_s)
    with _guard(dev):
        st = lib.slcl_proto_fwd_peer(ptr(feat_c), C.byref(m), ptr(labels), ptr(soft_mask), ptr(sel), ptr(centres), C.byref(p),
                                     ptr(stash), ptr(cstate), ptr(scal), C.byref(peer) if peer is not None else None, 0, ptr(ws),
                                     ws.numel(), stream_ptr(dev))
    check(st, "slcl_proto_fwd")
    return scal, stash, cstate


@proto_fwd.register_fake
def _(feat, labels, soft_mask, sel, centres, rows_layout, n_class, temperature, base_temperature, margin, easy_margin,
      normalize, peer_ptrs=0, rank=0, world=1, capacity_words=0, timeout_s=0.0):
    n = feat.shape[0] if rows_layout else feat.shape[0] * feat.shape[2] * feat.shape[3]
    c = feat.shape[1]
    return (feat.new_empty(4), feat.new_empty((n_class + 1, n)), feat.new_empty(n_class * c + n_class))


@torch.library.custom_op("slcl::proto_fwd_target", mutates_args=(), device_types="cuda")
def proto_fwd_target(feat: Tensor, centres: Tensor, sel_threshold: float, n_class: int, temperature: float,
                     base_temperature: float, margin: float, easy_margin: bool, peer_ptrs: int = 0, rank: int = 0,
                     world: int = 1, capacity_words: int = 0,
                     timeout_s: float = 0.0) -> Tuple[Tensor, Tensor, Tensor, Tensor, Tensor]:
    """-> (scal[4], stash, cstate, label[N] int64, sel[N]) : pseudo labels + target loss forward, one read of feat."""
    dev = require_cuda(feat, centres)
    lib = _lib.load()
    feat_c, m = _map_nchw(feat)
    n = m.batch * m.pixels
    centres = centres.to(_F32).contiguous()
    scal = torch.empty(4, dtype=_F32, device=dev)
    stash = torch.empty((n_class + 1, n), dtype=_F32, device=dev)
    cstate = torch.empty(n_class * m.channels + n_class, dtype=_F32, device=dev)
    label = torch.empty(n, dtype=torch.int64, device=dev)
    sel = torch.empty(n, dtype=_F32, device=dev)
    ws = _ws(lib.slcl_proto_workspace_bytes(n), dev)
    p = _params(n_class, temperature, base_temperature, margin, easy_margin, True)
    peer = _peer(peer_ptrs, rank, world, capacity_words, timeout_s)
    with _guard(dev):
        st = lib.slcl_proto_fwd_target_peer(ptr(feat_c), C.byref(m), ptr(centres), C.byref(p), float(sel_threshold), ptr(label),
                                            ptr(sel), ptr(stash), ptr(cstate), ptr(scal),
                                            C.byref(peer) if peer is not None else None, ptr(ws), ws.numel(), stream_ptr(dev))
    check(st, "slcl_proto_fwd_target")
    return scal, stash, cstate, label, sel


@proto_fwd_target.register_fake
def _(feat, centres, sel_threshold, n_class, temperature, base_temperature, margin, easy_margin, peer_ptrs=0, rank=0, world=1,
      capacity_words=0, timeout_s=0.0):
    n = feat.shape[0] * feat.shape[2] * feat.shape[3]
    c = feat.shape[1]
    return (feat.new_empty(4), feat.new_empty((n_class + 1, n)), feat.new_empty(n_class * c + n_class),
            torch.empty(n, dtype=torch.int64, device=feat.device), feat.new_empty(n))


@torch.library.custom_op("slcl::target_step", mutates_args=(), device_types="cuda")
def target_step(feat: Tensor, centres: Tensor, sel_threshold: float, weight_by_sel: bool, n_class: int, temperature: float,
                base_temperature: float, margin: float, easy_margin: bool, previous: Optional[Tensor], momentum: float,
                peer_ptrs: int = 0, rank: int = 0, world: int = 1, capacity_words: int = 0,
                timeout_s: float = 0.0) -> Tuple[Tensor, Tensor, Tensor, Tensor, Tensor, Tensor, Tensor, Tensor]:
    """Fused target step in ONE pass over feat: pseudo labels + target loss forward + per-class sums under those labels.
    -> (scal[4], stash, cstate, label[N] int64, sel[N], sums [K,C+1] f64, centroids [K,C], inv_weight [K]).
    Raises SlclError(unsupported) for shapes the tile kernel does not cover (the caller falls back)."""
    dev = require_cuda(feat, centres, previous)
    lib = _lib.load()
    feat = _nchw_contig(feat)
    b, c, h, w = feat.shape
    n = b * h * w
    centres = centres.to(_F32).contiguous()
    if previous is not None:
        previous = previous.to(_F32).contiguous()
    scal = torch.empty(4, dtype=_F32, device=dev)
    stash = torch.empty((n_class + 1, n), dtype=_F32, device=dev)
    cstate = torch.empty(n_class * c + n_class, dtype=_F32, device=dev)
    label = torch.empty(n, dtype=torch.int64, device=dev)
    sel = torch.empty(n, dtype=_F32, device=dev)
    sums = torch.empty((n_class, c + 1), dtype=torch.float64, device=dev)
    cen = torch.empty((n_class, c), dtype=_F32, device=dev)
    inv_w = torch.empty(n_class, dtype=_F32, device=dev)
    ws = _ws(lib.slcl_target_step_workspace_bytes(c, n_class), dev)
    p = _params(n_class, temperature, base_temperature, margin, easy_margin, True)
    peer = _peer(peer_ptrs, rank, world, capacity_words, timeout_s)
    with _guard(dev):
        st = lib.slcl_target_step(ptr(feat), b, c, h * w, ptr(centres), C.byref(p), float(sel_threshold), int(weight_by_sel),
                                  ptr(label), ptr(sel), ptr(stash), ptr(cstate), ptr(scal), ptr(sums), ptr(previous),
                                  float(momentum), ptr(cen), ptr(inv_w), C.byref(peer) if peer is not None else None, ptr(ws),
                                  ws.numel(), stream_ptr(dev))
    check(st, "slcl_target_step")
    return scal, stash, cstate, label, sel, sums, cen, inv_w


@target_step.register_fake
def _(feat, centres, sel_threshold, weight_by_sel, n_class, temperature, base_temperature, margin, easy_margin, previous,
      momentum, peer_ptrs=0, rank=0, world=1, capacity_words=0, timeout_s=0.0):
    n = feat.shape[0] * feat.shape[2] * feat.shape[3]
    c = feat.shape[1]
    dev = feat.device
    return (feat.new_empty(4), feat.new_empty((n_class + 1, n)), feat.new_empty(n_class * c + n_class),
            torch.empty(n, dtype=torch.int64, device=dev), feat.new_empty(n),
            torch.empty((n_class, c + 1), dtype=torch.float64, device=dev), feat.new_empty((n_class, c)), feat.new_empty(n_class))


def target_step_supported(feat: Tensor, n_class: int) -> bool:
    """Shapes the one-pass tile kernel covers (include/slcl.h, slcl_target_step)."""
    if feat.dim() != 4 or feat.dtype != _F32:
        return False
    b, c, h, w = feat.shape
    return (h * w) % 4 == 0 and c <= 128 and (c <= 64 or n_class <= 5) and 2 <= n_class <= 8


@torch.library.custom_op("slcl::proto_rescale", mutates_args=("scal",), device_types="cuda")
def proto_rescale(scal: Tensor, has_sel: bool) -> None:
    """Recompute scal[0:2] from the (all-reduced) sums scal[2:4], in place."""
    dev = require_cuda(scal)
    with _guard(dev):
        st = _lib.load().slcl_proto_rescale(ptr(scal), int(has_sel), stream_ptr(dev))
    check(st, "slcl_proto_rescale")


@torch.library.custom_op("slcl::proto_rescale_peer", mutates_args=("scal",), device_types="cuda")
def proto_rescale_peer(scal: Tensor, has_sel: bool, peer_ptrs: int, rank: int, world: int, capacity_words: int,
                       timeout_s: float) -> None:
    """Exchange scal[2:4] with the other ranks through NVLink peer mailboxes (slcl.peer.PeerMailbox) and rescale,
    in one kernel; every rank must call it in the same order."""
    dev = require_cuda(scal)
    peer = PeerT(peer_ptrs, rank, world, capacity_words, timeout_s)
    with _guard(dev):
        st = _lib.load().slcl_proto_rescale_peer(ptr(scal), int(has_sel), C.byref(peer), stream_ptr(dev))
    check(st, "slcl_proto_rescale_peer")


@torch.library.custom_op("slcl::peer_allreduce_f64", mutates_args=("buf",), device_types="cuda")
def peer_allreduce_f64(buf: Tensor, peer_ptrs: int, rank: int, world: int, capacity_words: int, timeout_s: float) -> None:
    """In-place sum of a float64 tensor over the ranks through the peer mailboxes (one kernel, no collective)."""
    dev = require_cuda(buf)
    if buf.dtype != torch.float64 or not buf.is_contiguous():
        raise ValueError("buf must be a contiguous float64 tensor")
    peer = PeerT(peer_ptrs, rank, world, capacity_words, timeout_s)
    with _guard(dev):
        st = _lib.load().slcl_peer_allreduce_f64(ptr(buf), buf.numel(), C.byref(peer), stream_ptr(dev))
    check(st, "slcl_peer_allreduce_f64")


@torch.library.custom_op("slcl::peer_allgather", mutates_args=("status",), device_types="cuda")
def peer_allgather(record: Tensor, status: Tensor, peer_ptrs: int, rank: int, world: int, capacity_words: int, timeout_s: float,
                   regions_ptr: int, slot_bytes: int) -> Tensor:
    """All ranks' uint8 records [n] (n % 16 == 0, equal first 16 bytes) -> [world, n] in rank order, over NVLink peer memory
    (slcl.peer.PeerMailbox built with rows_bytes).  ``status`` int32 [1], in/out: non-zero = a peer timed out (bit 0) or sent
    a record of another size (bit 1); the caller turns it into NaN."""
    dev = require_cuda(record, status)
    rec = record.contiguous()
    n = rec.numel()
    if rec.dtype != torch.uint8 or n % 16 or n < 16:
        raise ValueError("record must be uint8 with a multiple of 16 bytes")
    if status.dtype != torch.int32 or status.numel() != 1:
        raise ValueError("status must be int32 [1]")
    if not regions_ptr or slot_bytes <= 0:
        raise ValueError("this mailbox has no row region: build it with rows_bytes > 0")
    if n > slot_bytes:
        raise ValueError(f"record of {n} bytes exceeds the mailbox's row slot of {slot_bytes} bytes (rows_bytes)")
    out = torch.empty((world, n), dtype=torch.uint8, device=dev)
    peer = PeerT(peer_ptrs, rank, world, capacity_words, timeout_s)
    with _guard(dev):
        st = _lib.load().slcl_peer_allgather(ptr(rec), n, ptr(out), ptr(status), C.byref(peer), regions_ptr, slot_bytes,
                                             stream_ptr(dev))
    check(st, "slcl_peer_allgather")
    return out


@peer_allgather.register_fake
def _(record, status, peer_ptrs, rank, world, capacity_words, timeout_s, regions_ptr, slot_bytes):
    return record.new_empty((world, record.numel()))


@torch.library.custom_op("slcl::proto_bwd", mutates_args=(), device_types="cuda")
def proto_bwd(feat: Tensor, stash: Tensor, cstate: Tensor, scal: Tensor, grad_out: Tensor, rows_layout: bool,
              n_class: int, normalize: bool) -> Tensor:
    dev = require_cuda(feat, stash, cstate, scal, grad_out)
    lib = _lib.load()
    feat_c, m = _feat_map(feat, rows_layout)
    dfeat = torch.empty_strided(feat_c.shape, feat_c.stride(), dtype=_F32, device=dev)
    grad_out = grad_out.to(_F32).contiguous()
    p = _params(n_class, 1.0, 1.0, 0.0, False, normalize)
    with _guard(dev):
        st = lib.slcl_proto_bwd(ptr(feat_c), C.byref(m), ptr(stash), ptr(cstate), ptr(scal), ptr(grad_out), C.byref(p),
                                ptr(dfeat), stream_ptr(dev))
    check(st, "slcl_proto_bwd")
    return dfeat


@proto_bwd.register_fake
def _(feat, stash, cstate, scal, grad_out, rows_layout, n_class, normalize):
    return torch.empty_like(feat)


@torch.library.custom_op("slcl::proto_bwd_aux", mutates_args=(), device_types="cuda")
def proto_bwd_aux(feat: Tensor, labels: Optional[Tensor], soft_mask: Optional[Tensor], sel: Optional[Tensor], cstate: Tensor,
                  scal: Tensor, grad_out: Tensor, rows_layout: bool, n_class: int, temperature: float, base_temperature: float,
                  margin: float, easy_margin: bool, normalize: bool, want_dmask: bool, want_dsel: bool) -> Tuple[Tensor, Tensor]:
    """-> (d loss / d soft_mask [N,K], d loss / d pixel_sel_loc [N]); an output that is not wanted comes back empty."""
    dev = require_cuda(feat, labels, soft_mask, sel, cstate, scal, grad_out)
    lib = _lib.load()
    feat_c, m = _feat_map(feat, rows_layout)
    n = m.batch * m.pixels
    if labels is not None:
        labels = labels.contiguous()
    if soft_mask is not None:
        soft_mask = soft_mask.to(_F32).contiguous()
    if sel is not None:
        sel = sel.to(_F32).contiguous()
    if want_dmask and soft_mask is None:
        raise ValueError("d/d mask needs the soft mask")
    if want_dsel and sel is None:
        raise ValueError("d/d pixel_sel_loc needs pixel_sel_loc")
    dmask = torch.empty((n, n_class) if want_dmask else (0, n_class), dtype=_F32, device=dev)
    dsel = torch.empty(n if want_dsel else 0, dtype=_F32, device=dev)
    grad_out = grad_out.to(_F32).contiguous()
    p = _params(n_class, temperature, base_temperature, margin, easy_margin, normalize)
    with _guard(dev):
        st = lib.slcl_proto_bwd_aux(ptr(feat_c), C.byref(m), ptr(labels), ptr(soft_mask), ptr(sel), ptr(cstate), ptr(scal),
                                    ptr(grad_out), C.byref(p), ptr(dmask) if want_dmask else None,
                                    ptr(dsel) if want_dsel else None, stream_ptr(dev))
    check(st, "slcl_proto_bwd_aux")
    return dmask, dsel


@proto_bwd_aux.register_fake
def _(feat, labels, soft_mask, sel, cstate, scal, grad_out, rows_layout, n_class, temperature, base_temperature, margin,
      easy_margin, normalize, want_dmask, want_dsel):
    n = feat.shape[0] if rows_layout else feat.shape[0] * feat.shape[2] * feat.shape[3]
    return feat.new_empty((n if want_dmask else 0, n_class)), feat.new_empty(n if want_dsel else 0)


@torch.library.custom_op("slcl::proto_bwd_centres", mutates_args=(), device_types="cuda")
def proto_bwd_centres(feat: Tensor, stash: Tensor, cstate: Tensor, scal: Tensor, grad_out: Tensor, rows_layout: bool,
                      n_class: int, normalize: bool) -> Tensor:
    dev = require_cuda(feat, stash, cstate, scal, grad_out)
    lib = _lib.load()
    feat_c, m = _feat_map(feat, rows_layout)
    dcen = torch.empty((n_class, m.channels), dtype=_F32, device=dev)
    grad_out = grad_out.to(_F32).contiguous()
    ws = _ws(lib.slcl_proto_bwd_centres_workspace_bytes(m.batch * m.pixels, m.channels, n_class), dev)
    p = _params(n_class, 1.0, 1.0, 0.0, False, normalize)
    with _guard(dev):
        st = lib.slcl_proto_bwd_centres(ptr(feat_c), C.byref(m), ptr(stash), ptr(cstate), ptr(scal), ptr(grad_out),
                                        C.byref(p), ptr(dcen), ptr(ws), ws.numel(), stream_ptr(dev))
    check(st, "slcl_proto_bwd_centres")
    return dcen


@proto_bwd_centres.register_fake
def _(feat, stash, cstate, scal, grad_out, rows_layout, n_class, normalize):
    return feat.new_empty((n_class, feat.shape[1]))


@torch.library.custom_op("slcl::pseudo_label", mutates_args=(), device_types="cuda")
def pseudo_label(feat: Tensor, centres: Tensor, threshold: float) -> Tuple[Tensor, Tensor]:
    dev = require_cuda(feat, centres)
    lib = _lib.load()
    feat_c, m = _map_nchw(feat)
    centres = centres.to(_F32).contiguous()
    k = centres.shape[0]
    n = m.batch * m.pixels
    label = torch.empty(n, dtype=torch.int64, device=dev)
    sel = torch.empty(n, dtype=_F32, device=dev)
    ws = _ws((k * m.channels + k) * 4, dev)
    with _guard(dev):
        st = lib.slcl_pseudo_label(ptr(feat_c), C.byref(m), ptr(centres), k, float(threshold), ptr(label), ptr(sel),
                                   ptr(ws), ws.numel(), stream_ptr(dev))
    check(st, "slcl_pseudo_label")
    return label, sel


@pseudo_label.register_fake
def _(feat, centres, threshold):
    n = feat.shape[0] * feat.shape[2] * feat.shape[3]
    return (torch.empty(n, dtype=torch.int64, device=feat.device), feat.new_empty(n))


# ----------------------------------------------------------------------------
# class sums / centroids
# ----------------------------------------------------------------------------
def _nchw_contig(feat: Tensor) -> Tensor:
    if feat.dim() != 4 or feat.dtype != _F32:
        raise ValueError("feature map must be float32 [B, C, H, W]")
    return feat.contiguous()


@torch.library.custom_op("slcl::class_sums", mutates_args=(), device_types="cuda")
def class_sums(feat: Tensor, labels: Optional[Tensor], probs: Optional[Tensor], weighted: bool, threshold: float,
               part_id: Optional[Tensor], n_partitions: int, n_class: int) -> Tensor:
    """-> sums [P*K, C+1] float64 (weighted feature sums | weight sums)."""
    dev = require_cuda(feat, labels, probs, part_id)
    lib = _lib.load()
    feat = _nchw_contig(feat)
    b, c, h, w = feat.shape
    if labels is not None:
        labels = labels.contiguous()
        if labels.dtype != torch.int64 or labels.numel() != b * h * w:
            raise ValueError("labels must be int64 with B*H*W elements")
    if probs is not None:
        probs = probs.to(_F32).contiguous()
        if probs.shape != (b, n_class, h, w):
            raise ValueError("probs must be [B, K, H, W] at feature resolution")
    if part_id is not None:
        part_id = part_id.contiguous()
        if part_id.dtype != torch.int32 or part_id.numel() != b * h * w:
            raise ValueError("part_id must be int32 with B*H*W elements")
    cols = n_partitions * n_class
    sums = torch.empty((cols, c + 1), dtype=torch.float64, device=dev)
    ws = _ws(lib.slcl_class_sums_workspace_bytes(b, c, h * w, cols), dev)
    with _guard(dev):
        st = lib.slcl_class_sums(ptr(feat), b, c, h * w, ptr(labels), ptr(probs), int(weighted), float(threshold),
                                 ptr(part_id), n_partitions, n_class, ptr(sums), ptr(ws), ws.numel(), stream_ptr(dev))
    check(st, "slcl_class_sums")
    return sums


@class_sums.register_fake
def _(feat, labels, probs, weighted, threshold, part_id, n_partitions, n_class):
    return torch.empty((n_partitions * n_class, feat.shape[1] + 1), dtype=torch.float64, device=feat.device)


@torch.library.custom_op("slcl::class_centres_update", mutates_args=(), device_types="cuda")
def class_centres_update(feat: Tensor, labels: Tensor, old_centres: Tensor, m: float, peer_ptrs: int = 0, rank: int = 0,
                         world: int = 1, capacity_words: int = 0, timeout_s: float = 0.0) -> Tuple[Tensor, Tensor]:
    """update_class_center_iter as two launches: hard class sums, then reduce [+ peer all-reduce] + EMA finalise.
    -> (new centres [K,C], sums [K,C+1] float64 -- the GLOBAL sums when a peer mailbox is given)."""
    dev = require_cuda(feat, labels, old_centres)
    lib = _lib.load()
    feat = _nchw_contig(feat)
    b, c, h, w = feat.shape
    labels = labels.contiguous()
    if labels.dtype != torch.int64 or labels.numel() != b * h * w:
        raise ValueError("labels must be int64 with B*H*W elements")
    old = old_centres.to(_F32).contiguous()
    k = old.shape[0]
    if old.shape != (k, c):
        raise ValueError("class centres must be [K, C]")
    sums = torch.empty((k, c + 1), dtype=torch.float64, device=dev)
    new = torch.empty_like(old)
    ws = _ws(lib.slcl_class_sums_workspace_bytes(b, c, h * w, k), dev)
    peer = _peer(peer_ptrs, rank, world, capacity_words, timeout_s)
    with _guard(dev):
        st = lib.slcl_class_centres_update(ptr(feat), b, c, h * w, ptr(labels), k, ptr(old), float(m), ptr(new), ptr(sums),
                                           C.byref(peer) if peer is not None else None, ptr(ws), ws.numel(), stream_ptr(dev))
    check(st, "slcl_class_centres_update")
    return new, sums


@class_centres_update.register_fake
def _(feat, labels, old_centres, m, peer_ptrs=0, rank=0, world=1, capacity_words=0, timeout_s=0.0):
    return (torch.empty_like(old_centres, dtype=_F32),
            torch.empty((old_centres.shape[0], feat.shape[1] + 1), dtype=torch.float64, device=feat.device))


@torch.library.custom_op("slcl::centroids_fwd", mutates_args=(), device_types="cuda")
def centroids_fwd(feat: Tensor, labels: Optional[Tensor], probs: Optional[Tensor], weighted: bool, threshold: float,
                  part_id: Optional[Tensor], n_partitions: int, n_class: int, previous: Optional[Tensor], momentum: float,
                  peer_ptrs: int = 0, rank: int = 0, world: int = 1, capacity_words: int = 0,
                  timeout_s: float = 0.0) -> Tuple[Tensor, Tensor, Tensor]:
    """cal_centroid forward as two launches: class sums, then reduce [+ peer all-reduce] + centroid finalise.
    -> (centroids [P*K, C], inv_weight [P*K], sums [P*K, C+1] float64)."""
    dev = require_cuda(feat, labels, probs, part_id, previous)
    lib = _lib.load()
    feat = _nchw_contig(feat)
    b, c, h, w = feat.shape
    if labels is not None:
        labels = labels.contiguous()
        if labels.dtype != torch.int64 or labels.numel() != b * h * w:
            raise ValueError("labels must be int64 with B*H*W elements")
    if probs is not None:
        probs = probs.to(_F32).contiguous()
        if probs.shape != (b, n_class, h, w):
            raise ValueError("probs must be [B, K, H, W] at feature resolution")
    if part_id is not None:
        part_id = part_id.contiguous()
        if part_id.dtype != torch.int32 or part_id.numel() != b * h * w:
            raise ValueError("part_id must be int32 with B*H*W elements")
    if previous is not None:
        previous = previous.to(_F32).contiguous()
        if previous.shape != (n_class, c):
            raise ValueError("previous centroid must be [K, C]")
    cols = n_partitions * n_class
    sums = torch.empty((cols, c + 1), dtype=torch.float64, device=dev)
    cen = torch.empty((cols, c), dtype=_F32, device=dev)
    inv_w = torch.empty(cols, dtype=_F32, device=dev)
    ws = _ws(lib.slcl_class_sums_workspace_bytes(b, c, h * w, cols), dev)
    peer = _peer(peer_ptrs, rank, world, capacity_words, timeout_s)
    with _guard(dev):
        st = lib.slcl_centroids_fwd(ptr(feat), b, c, h * w, ptr(labels), ptr(probs), int(weighted), float(threshold),
                                    ptr(part_id), n_partitions, n_class, ptr(previous), float(momentum), ptr(cen), ptr(inv_w),
                                    ptr(sums), C.byref(peer) if peer is not None else None, ptr(ws), ws.numel(),
                                    stream_ptr(dev))
    check(st, "slcl_centroids_fwd")
    return cen, inv_w, sums


@centroids_fwd.register_fake
def _(feat, labels, probs, weighted, threshold, part_id, n_partitions, n_class, previous, momentum, peer_ptrs=0, rank=0,
      world=1, capacity_words=0, timeout_s=0.0):
    rows, c = n_partitions * n_class, feat.shape[1]
    return (torch.empty((rows, c), dtype=_F32, device=feat.device), torch.empty(rows, dtype=_F32, device=feat.device),
            torch.empty((rows, c + 1), dtype=torch.float64, device=feat.device))


@torch.library.custom_op("slcl::ema_finalize", mutates_args=(), device_types="cuda")
def ema_finalize(sums: Tensor, old_centres: Tensor, m: float) -> Tensor:
    dev = require_cuda(sums, old_centres)
    lib = _lib.load()
    old = old_centres.to(_F32).contiguous()
    k, c = old.shape
    if sums.dtype != torch.float64 or sums.shape != (k, c + 1):
        raise ValueError("sums must be float64 [K, C+1]")
    out = torch.empty_like(old)
    with _guard(dev):
        st = lib.slcl_ema_finalize(ptr(sums.contiguous()), ptr(old), float(m), k, c, ptr(out), stream_ptr(dev))
    check(st, "slcl_ema_finalize")
    return out


@ema_finalize.register_fake
def _(sums, old_centres, m):
    return torch.empty_like(old_centres)


@torch.library.custom_op("slcl::centroid_finalize", mutates_args=(), device_types="cuda")
def centroid_finalize(sums: Tensor, previous: Optional[Tensor], momentum: float, n_sets: int,
                      n_class: int) -> Tuple[Tensor, Tensor]:
    dev = require_cuda(sums, previous)
    lib = _lib.load()
    sums = sums.contiguous()
    rows, c1 = sums.shape
    c = c1 - 1
    if sums.dtype != torch.float64 or rows != n_sets * n_class:
        raise ValueError("sums must be float64 [sets*K, C+1]")
    if previous is not None:
        previous = previous.to(_F32).contiguous()
        if previous.shape != (n_class, c):
            raise ValueError("previous centroid must be [K, C]")
    cen = torch.empty((rows, c), dtype=_F32, device=dev)
    inv_w = torch.empty(rows, dtype=_F32, device=dev)
    with _guard(dev):
        st = lib.slcl_centroid_finalize(ptr(sums), ptr(previous), float(momentum), n_sets, n_class, c, ptr(cen),
                                        ptr(inv_w), stream_ptr(dev))
    check(st, "slcl_centroid_finalize")
    return cen, inv_w


@centroid_finalize.register_fake
def _(sums, previous, momentum, n_sets, n_class):
    return (torch.empty((sums.shape[0], sums.shape[1] - 1), dtype=_F32, device=sums.device),
            torch.empty(sums.shape[0], dtype=_F32, device=sums.device))


@torch.library.custom_op("slcl::centroid_bwd", mutates_args=(), device_types="cuda")
def centroid_bwd(feat: Tensor, labels: Optional[Tensor], probs: Optional[Tensor], weighted: bool, threshold: float,
                 part_id: Optional[Tensor], n_partitions: int, n_class: int, grad_centroids: Tensor, sums: Tensor,
                 ema_scale: float, need_dprobs: bool) -> Tuple[Tensor, Tensor]:
    dev = require_cuda(feat, labels, probs, part_id, grad_centroids, sums)
    lib = _lib.load()
    feat = _nchw_contig(feat)
    b, c, h, w = feat.shape
    if labels is not None:
        labels = labels.contiguous()
    if probs is not None:
        probs = probs.to(_F32).contiguous()
    if part_id is not None:
        part_id = part_id.contiguous()
    cols = n_partitions * n_class
    g = grad_centroids.to(_F32).contiguous()
    if g.shape != (cols, c):
        raise ValueError("grad_centroids must be [P*K, C]")
    dfeat = torch.empty_like(feat)
    dprobs = torch.empty_like(probs) if (need_dprobs and probs is not None) else torch.empty(0, dtype=_F32, device=dev)
    ws = _ws(lib.slcl_centroid_bwd_workspace_bytes(c, cols), dev)
    with _guard(dev):
        st = lib.slcl_centroid_bwd(ptr(feat), b, c, h * w, ptr(labels), ptr(probs), int(weighted), float(threshold),
                                   ptr(part_id), n_partitions, n_class, ptr(g), ptr(sums.contiguous()), float(ema_scale),
                                   ptr(dfeat), ptr(dprobs) if dprobs.numel() else None, ptr(ws), ws.numel(),
                                   stream_ptr(dev))
    check(st, "slcl_centroid_bwd")
    return dfeat, dprobs


@centroid_bwd.register_fake
def _(feat, labels, probs, weighted, threshold, part_id, n_partitions, n_class, grad_centroids, sums, ema_scale,
      need_dprobs):
    dp = torch.empty_like(probs) if (need_dprobs and probs is not None) else feat.new_empty(0)
    return torch.empty_like(feat), dp


@torch.library.custom_op("slcl::centroid_loss", mutates_args=(), device_types="cuda")
def centroid_loss(centroid_s: Tensor, centroid_t: Tensor, mode: int, first_row: int, n_rows: int,
                  norm: bool) -> Tuple[Tensor, Tensor, Tensor]:
    """-> (loss[1], dL/ds, dL/dt) for dL/dloss = 1."""
    dev = require_cuda(centroid_s, centroid_t)
    lib = _lib.load()
    s = centroid_s.to(_F32).contiguous()
    t = centroid_t.to(_F32).contiguous()
    if s.dim() != 2 or s.shape != t.shape:
        raise ValueError("centroids must both be [K, C]")
    k, c = s.shape
    loss = torch.empty(1, dtype=_F32, device=dev)
    ds = torch.empty_like(s)
    dt = torch.empty_like(t)
    with _guard(dev):
        st = lib.slcl_centroid_loss(ptr(s), ptr(t), k, c, mode, first_row, n_rows, int(norm), ptr(loss), ptr(ds), ptr(dt),
                                    stream_ptr(dev))
    check(st, "slcl_centroid_loss")
    return loss, ds, dt


@centroid_loss.register_fake
def _(centroid_s, centroid_t, mode, first_row, n_rows, norm):
    return centroid_s.new_empty(1), torch.empty_like(centroid_s), torch.empty_like(centroid_t)


@torch.library.custom_op("slcl::mccl_losses", mutates_args=(), device_types="cuda")
def mccl_losses(centroid_s: Tensor, centroid_t_parts: Tensor, centroid_t_aug: Optional[Tensor], n_partitions: int, split: bool,
                bg: bool, norm: bool, inter_w: float, intra_w: float, cnr_w: float) -> Tuple[Tensor, Tensor, Tensor, Tensor]:
    """All centroid<->centroid terms of one MCCL step in two launches.
    -> (losses[4] = {total, inter, intra, cnr}, d total/d S [K,C], d total/d T [P*K,C], d total/d A [K,C] (empty without A))."""
    dev = require_cuda(centroid_s, centroid_t_parts, centroid_t_aug)
    lib = _lib.load()
    s = centroid_s.to(_F32).contiguous()
    t = centroid_t_parts.to(_F32).contiguous()
    k, c = s.shape
    if t.shape != (n_partitions * k, c):
        raise ValueError("centroid_t_parts must be [P*K, C]")
    a = None
    if centroid_t_aug is not None:
        a = centroid_t_aug.to(_F32).contiguous()
        if a.shape != (k, c):
            raise ValueError("centroid_t_aug must be [K, C]")
    losses = torch.empty(4, dtype=_F32, device=dev)
    ds, dt = torch.empty_like(s), torch.empty_like(t)
    da = torch.empty_like(s) if a is not None else torch.empty(0, dtype=_F32, device=dev)
    ws = _ws(lib.slcl_mccl_losses_workspace_bytes(n_partitions, k, c), dev)
    with _guard(dev):
        st = lib.slcl_mccl_losses(ptr(s), ptr(t), ptr(a), n_partitions, k, c, int(split), int(bg), int(norm), float(inter_w),
                                  float(intra_w), float(cnr_w), ptr(losses), ptr(ds), ptr(dt), ptr(da) if a is not None else None,
                                  ptr(ws), ws.numel(), stream_ptr(dev))
    check(st, "slcl_mccl_losses")
    return losses, ds, dt, da


@mccl_losses.register_fake
def _(centroid_s, centroid_t_parts, centroid_t_aug, n_partitions, split, bg, norm, inter_w, intra_w, cnr_w):
    da = torch.empty_like(centroid_s) if centroid_t_aug is not None else centroid_s.new_empty(0)
    return centroid_s.new_empty(4), torch.empty_like(centroid_s), torch.empty_like(centroid_t_parts), da


# ----------------------------------------------------------------------------
# sampler
# ----------------------------------------------------------------------------
@torch.library.custom_op("slcl::compact_by_class", mutates_args=(), device_types="cuda")
def compact_by_class(labels: Tensor, n_class: int) -> Tuple[Tensor, Tensor, Tensor]:
    """-> (counts[K], offsets[K+1], index[N]) int64; index[offsets[k]:offsets[k+1]] == nonzero(labels == k)."""
    dev = require_cuda(labels)
    lib = _lib.load()
    lab = labels.reshape(-1).contiguous()
    if lab.dtype != torch.int64:
        raise ValueError("labels must be int64")
    n = lab.numel()
    counts = torch.empty(n_class, dtype=torch.int64, device=dev)
    offsets = torch.empty(n_class + 1, dtype=torch.int64, device=dev)
    index = torch.empty(n, dtype=torch.int64, device=dev)
    ws = _ws(lib.slcl_compact_workspace_bytes(n, n_class), dev)
    with _guard(dev):
        st = lib.slcl_compact_by_class(ptr(lab), n, n_class, ptr(counts), ptr(offsets), ptr(index), ptr(ws), ws.numel(),
                                       stream_ptr(dev))
    check(st, "slcl_compact_by_class")
    return counts, offsets, index


@compact_by_class.register_fake
def _(labels, n_class):
    dev = labels.device
    return (torch.empty(n_class, dtype=torch.int64, device=dev), torch.empty(n_class + 1, dtype=torch.int64, device=dev),
            torch.empty(labels.numel(), dtype=torch.int64, device=dev))


@torch.library.custom_op("slcl::sample_balanced", mutates_args=(), device_types="cuda")
def sample_balanced(perm: Tensor, labels: Tensor, n_class: int, per_a: int, per_b: int) -> Tuple[Tensor, Tensor, Tensor, Tensor]:
    """Two-phase class-balanced pick for two quotas from one permutation (slcl_sample_balanced):
    -> (idx_a [K*per_a], filled_a [1], idx_b [K*per_b], filled_b [1]) int64."""
    dev = require_cuda(perm, labels)
    lib = _lib.load()
    pm, lab = perm.reshape(-1).contiguous(), labels.reshape(-1).contiguous()
    if pm.dtype != torch.int64 or lab.dtype != torch.int64 or pm.numel() != lab.numel():
        raise ValueError("perm and labels must be int64 of equal length")
    if per_a < 1 or per_b < 1:
        raise ValueError("both quotas need at least one pick per class")
    n = lab.numel()
    out_a = torch.empty(n_class * per_a, dtype=torch.int64, device=dev)
    out_b = torch.empty(n_class * per_b, dtype=torch.int64, device=dev)
    fill_a = torch.empty(1, dtype=torch.int64, device=dev)
    fill_b = torch.empty(1, dtype=torch.int64, device=dev)
    ws = _ws(lib.slcl_sample_balanced_workspace_bytes(n, n_class), dev)
    with _guard(dev):
        st = lib.slcl_sample_balanced(ptr(pm), ptr(lab), n, int(n_class), int(per_a), ptr(out_a), ptr(fill_a), int(per_b), ptr(out_b),
                                      ptr(fill_b), ptr(ws), ws.numel(), stream_ptr(dev))
    check(st, "slcl_sample_balanced")
    return out_a, fill_a, out_b, fill_b


@sample_balanced.register_fake
def _(perm, labels, n_class, per_a, per_b):
    dev = perm.device
    return (torch.empty(n_class * per_a, dtype=torch.int64, device=dev), torch.empty(1, dtype=torch.int64, device=dev),
            torch.empty(n_class * per_b, dtype=torch.int64, device=dev), torch.empty(1, dtype=torch.int64, device=dev))


@torch.library.custom_op("slcl::self_maps_bounded", mutates_args=(), device_types="cuda")
def self_maps_bounded(id_a: Tensor, id_b: Tensor, n_ids: int) -> Tuple[Tensor, Tensor, Tensor]:
    """(a_selfcol [A], b_selfrow [M], row_of_id [2, n_ids]) int32 for ids in [0, n_ids) (pixel indices), unique within
    each side: two lookup tables instead of the sort of ``self_maps``; the tables come back too (row_of_id[0][id] =
    anchor row holding id or -1, row_of_id[1] likewise for the contrast rows)."""
    dev = require_cuda(id_a, id_b)
    lib = _lib.load()
    ia, ib = id_a.reshape(-1).contiguous(), id_b.reshape(-1).contiguous()
    if ia.dtype != torch.int64 or ib.dtype != torch.int64:
        raise ValueError("ids must be int64")
    selfcol = torch.empty(ia.numel(), dtype=torch.int32, device=dev)
    selfrow = torch.empty(ib.numel(), dtype=torch.int32, device=dev)
    tables = torch.empty((2, int(n_ids)), dtype=torch.int32, device=dev)
    with _guard(dev):
        st = lib.slcl_self_maps(ptr(ia), ia.numel(), ptr(ib), ib.numel(), int(n_ids), ptr(selfcol), ptr(selfrow), ptr(tables),
                                stream_ptr(dev))
    check(st, "slcl_self_maps")
    return selfcol, selfrow, tables


@self_maps_bounded.register_fake
def _(id_a, id_b, n_ids):
    dev = id_a.device
    return (torch.empty(id_a.numel(), dtype=torch.int32, device=dev), torch.empty(id_b.numel(), dtype=torch.int32, device=dev),
            torch.empty((2, n_ids), dtype=torch.int32, device=dev))


@torch.library.custom_op("slcl::scatter_rows_by_map", mutates_args=(), device_types="cuda")
def scatter_rows_by_map(feat: Tensor, normalize: bool, map_a: Tensor, d_a: Tensor, inv_a: Tensor,
                        map_b: Optional[Tensor], d_b: Optional[Tensor], inv_b: Optional[Tensor]) -> Tensor:
    """dfeat (every element written) from row gradients and pixel -> row maps (slcl_scatter_rows_by_map)."""
    dev = require_cuda(feat, map_a, d_a, inv_a)
    lib = _lib.load()
    if not feat.is_contiguous() or feat.dim() != 4 or feat.dtype != _F32:
        raise ValueError("feat must be a contiguous float32 NCHW map")
    b, c, h, w = feat.shape
    n = b * h * w

    def chk(m, d, what):
        if m.dtype != torch.int32 or m.numel() != n or not m.is_contiguous():
            raise ValueError(f"{what}: the pixel -> row map must be contiguous int32 [{n}]")
        if d.dtype != _F32 or d.dim() != 2 or d.shape[1] != c or not d.is_contiguous():
            raise ValueError(f"{what}: row gradients must be contiguous float32 [rows, {c}]")
    chk(map_a, d_a, "set a")
    two = map_b is not None
    if two:
        if d_b is None or inv_b is None:
            raise ValueError("set b needs its map, its row gradients and its inverse norms")
        chk(map_b, d_b, "set b")
    dfeat = torch.empty_like(feat)
    with _guard(dev):
        st = lib.slcl_scatter_rows_by_map(ptr(feat), b, c, h * w, int(normalize), ptr(map_a), ptr(d_a), ptr(inv_a.contiguous()),
                                          ptr(map_b) if two else None, ptr(d_b) if two else None,
                                          ptr(inv_b.contiguous()) if two else None, ptr(dfeat), stream_ptr(dev))
    check(st, "slcl_scatter_rows_by_map")
    return dfeat


@scatter_rows_by_map.register_fake
def _(feat, normalize, map_a, d_a, inv_a, map_b, d_b, inv_b):
    return torch.empty_like(feat)


@torch.library.custom_op("slcl::rows_meta", mutates_args=(), device_types="cuda")
def rows_meta(labels: Tensor, pixel_idx: Tensor) -> Tensor:
    """{label, id = pixel index} int32 pairs of the sampled rows, padded to a multiple of 64 rows with INT_MIN -- what
    ``pad_meta(labels[idx], idx)`` builds, in one launch."""
    dev = require_cuda(labels, pixel_idx)
    lib = _lib.load()
    lab, idx = labels.reshape(-1).contiguous(), pixel_idx.reshape(-1).contiguous()
    if lab.dtype != torch.int64 or idx.dtype != torch.int64:
        raise ValueError("labels and pixel_idx must be int64")
    n = idx.numel()
    meta = torch.empty(((n + 63) // 64 * 64, 2), dtype=torch.int32, device=dev)
    with _guard(dev):
        st = lib.slcl_rows_meta(ptr(lab), lab.numel(), ptr(idx), n, ptr(meta), stream_ptr(dev))
    check(st, "slcl_rows_meta")
    return meta


@rows_meta.register_fake
def _(labels, pixel_idx):
    n = pixel_idx.numel()
    return torch.empty(((n + 63) // 64 * 64, 2), dtype=torch.int32, device=labels.device)


@torch.library.custom_op("slcl::tile_weights", mutates_args=(), device_types="cuda")
def tile_weights(meta: Tensor, n_rows: int, n_tiles: int, zero_if_empty: bool) -> Tuple[Tensor, Tensor]:
    """Row weights fg_r / (foreground rows of r's tile) / (tiles with foreground) from the first ``n_rows`` metadata
    rows of ``rows_meta`` / ``pad_meta`` (label != 0 = foreground), split into ``n_tiles`` equal tiles
    (slcl_tile_weights) -> (weight [n_rows], tile_fg [n_tiles])."""
    dev = require_cuda(meta)
    lib = _lib.load()
    if meta.dtype != torch.int32 or meta.dim() != 2 or meta.shape[1] != 2 or not meta.is_contiguous():
        raise ValueError("meta must be contiguous int32 [rows_padded, 2]")
    if n_tiles < 1 or n_rows < 1 or n_rows % n_tiles or n_rows > meta.shape[0]:
        raise ValueError("n_rows must be a positive multiple of n_tiles within the metadata rows")
    weight = torch.empty(n_rows, dtype=_F32, device=dev)
    tile_fg = torch.empty(n_tiles, dtype=_F32, device=dev)
    with _guard(dev):
        st = lib.slcl_tile_weights(ptr(meta), int(n_tiles), n_rows // n_tiles, int(zero_if_empty), ptr(tile_fg), ptr(weight),
                                   stream_ptr(dev))
    check(st, "slcl_tile_weights")
    return weight, tile_fg


@tile_weights.register_fake
def _(meta, n_rows, n_tiles, zero_if_empty):
    return (torch.empty(n_rows, dtype=_F32, device=meta.device), torch.empty(n_tiles, dtype=_F32, device=meta.device))


@torch.library.custom_op("slcl::gather_unit_rows", mutates_args=(), device_types="cuda")
def gather_unit_rows(feat: Tensor, pixel_idx: Tensor, normalize: bool, want_bf16: bool,
                     want_f32: bool) -> Tuple[Tensor, Tensor, Tensor]:
    """-> (rows_bf16 [R, pad64(C)] (pad columns zero), rows_f32 [R, C], inv_norm [R])."""
    dev = require_cuda(feat, pixel_idx)
    lib = _lib.load()
    feat = _nchw_contig(feat)
    b, c, h, w = feat.shape
    idx = pixel_idx.reshape(-1).contiguous()
    if idx.dtype != torch.int64:
        raise ValueError("pixel_idx must be int64")
    r = idx.numel()
    cp = (c + 63) // 64 * 64
    rows_bf16 = torch.empty((r, cp) if want_bf16 else (0, cp), dtype=torch.bfloat16, device=dev)
    rows_f32 = torch.empty((r, c) if want_f32 else (0, c), dtype=_F32, device=dev)
    inv_norm = torch.empty(r, dtype=_F32, device=dev)
    with _guard(dev):
        st = lib.slcl_gather_unit_rows(ptr(feat), b, c, h * w, ptr(idx), r, int(normalize),
                                       ptr(rows_bf16) if want_bf16 else None, cp, ptr(rows_f32) if want_f32 else None,
                                       ptr(inv_norm), stream_ptr(dev))
    check(st, "slcl_gather_unit_rows")
    return rows_bf16, rows_f32, inv_norm


@gather_unit_rows.register_fake
def _(feat, pixel_idx, normalize, want_bf16, want_f32):
    r, c = pixel_idx.numel(), feat.shape[1]
    cp = (c + 63) // 64 * 64
    return (torch.empty((r if want_bf16 else 0, cp), dtype=torch.bfloat16, device=feat.device),
            torch.empty((r if want_f32 else 0, c), dtype=_F32, device=feat.device), feat.new_empty(r))


@torch.library.custom_op("slcl::p2p_shift", mutates_args=(), device_types="cuda")
def p2p_shift(inv_norm_a: Tensor, inv_norm_b: Tensor, temperature: float) -> Tensor:
    """exp shift of un-normalised rows, shift_i = |a_i| max_j |b_j| / T (one launch instead of five torch ops)."""
    dev = require_cuda(inv_norm_a, inv_norm_b)
    lib = _lib.load()
    ia, ib = inv_norm_a.contiguous(), inv_norm_b.contiguous()
    if ia.dtype != _F32 or ib.dtype != _F32:
        raise ValueError("inv_norm tensors must be float32")
    if ib.numel() > (1 << 20):          # beyond the single-launch kernel's range
        return (1.0 / ia) * ((1.0 / ib).amax() / temperature)
    shift = torch.empty_like(ia)
    with _guard(dev):
        st = lib.slcl_p2p_shift(ptr(ia), ia.numel(), ptr(ib), ib.numel(), float(temperature), ptr(shift), stream_ptr(dev))
    check(st, "slcl_p2p_shift")
    return shift


@p2p_shift.register_fake
def _(inv_norm_a, inv_norm_b, temperature):
    return torch.empty_like(inv_norm_a)


@torch.library.custom_op("slcl::scatter_rows_bwd", mutates_args=("dfeat",), device_types="cuda")
def scatter_rows_bwd(feat: Tensor, pixel_idx: Tensor, normalize: bool, d_rows: Tensor, inv_norm: Tensor,
                     dfeat: Tensor) -> None:
    dev = require_cuda(feat, pixel_idx, d_rows, inv_norm, dfeat)
    lib = _lib.load()
    if not (feat.is_contiguous() and dfeat.is_contiguous() and feat.shape == dfeat.shape):
        raise ValueError("feat and dfeat must be contiguous NCHW of equal shape")
    b, c, h, w = feat.shape
    idx = pixel_idx.reshape(-1).contiguous()
    d_rows = d_rows.to(_F32).contiguous()
    with _guard(dev):
        st = lib.slcl_scatter_rows_bwd(ptr(feat), b, c, h * w, ptr(idx), idx.numel(), int(normalize), ptr(d_rows),
                                       ptr(inv_norm), ptr(dfeat), stream_ptr(dev))
    check(st, "slcl_scatter_rows_bwd")


# ----------------------------------------------------------------------------
# pixel <-> pixel (tensor cores)
# ----------------------------------------------------------------------------
def pad_meta(label: Tensor, ident: Tensor) -> Tensor:
    """{label, id} int32 pairs padded to a multiple of 64 rows with INT_MIN (the kernel's masked sentinel)."""
    n = label.numel()
    out = torch.full(((n + 63) // 64 * 64, 2), -2 ** 31, dtype=torch.int32, device=label.device)
    out[:n, 0] = label.to(torch.int32)
    out[:n, 1] = ident.to(torch.int32)
    return out


def _p2p_check(a: Tensor, b: Tensor, a_meta: Tensor, b_meta: Tensor, shift: Tensor, weight: Tensor):
    if a.dtype != torch.bfloat16 or b.dtype != torch.bfloat16 or a.dim() != 2 or b.dim() != 2 or a.shape[1] != b.shape[1]:
        raise ValueError("anchors / contrast rows must be bf16 [rows, dim_padded] with equal dim_padded")
    if a.shape[1] % 64 or a.shape[1] > 256:
        raise ValueError("dim_padded must be a multiple of 64, at most 256")
    if not (a.is_contiguous() and b.is_contiguous()):
        raise ValueError("rows must be contiguous")
    for m, t in ((a_meta, a), (b_meta, b)):
        if m.dtype != torch.int32 or m.shape != ((t.shape[0] + 63) // 64 * 64, 2) or not m.is_contiguous():
            raise ValueError("meta must be contiguous int32 [pad64(rows), 2] = {label, id} (see pad_meta)")
    if shift.shape != (a.shape[0],) or weight.shape != (a.shape[0],) or shift.dtype != _F32 or weight.dtype != _F32:
        raise ValueError("shift / weight must be float32 [A]")


def self_maps(id_a: Tensor, id_b: Tensor) -> Tuple[Tensor, Tensor]:
    """(a_selfcol [A], b_selfrow [M]) int32 for the analytic p2p mode: the contrast row carrying anchor i's id
    (-1: none) and its inverse.  Ids must be unique within each side.  No host synchronisation (no boolean-mask
    indexing): anchors without a contrast row scatter into a dump slot."""
    m = id_b.numel()
    sorted_b, perm = torch.sort(id_b.reshape(-1).long())
    ia = id_a.reshape(-1).long()
    pos = torch.searchsorted(sorted_b, ia).clamp_(max=m - 1)
    found = sorted_b[pos] == ia
    selfcol = torch.where(found, perm[pos], torch.full_like(pos, -1))
    selfrow = torch.full((m + 1,), -1, dtype=torch.long, device=id_b.device)
    selfrow.index_put_((torch.where(found, selfcol, torch.full_like(selfcol, m)),),
                       torch.arange(ia.numel(), device=ia.device))
    return selfcol.to(torch.int32), selfrow[:m].to(torch.int32).contiguous()


def _selfcol_check(t: Optional[Tensor], n: int, what: str):
    if t is not None and (t.dtype != torch.int32 or t.shape != (n,) or not t.is_contiguous()):
        raise ValueError(f"{what} must be contiguous int32 [{n}]")


@torch.library.custom_op("slcl::p2p_fwd", mutates_args=(), device_types="cuda")
def p2p_fwd(a: Tensor, b: Tensor, a_meta: Tensor, b_meta: Tensor, shift: Tensor, weight: Tensor,
            temperature: float, n_class: int = 0, a_selfcol: Optional[Tensor] = None,
            keep_state: bool = False, n_batch: int = 1) -> Tuple[Tensor, Tensor, Tensor]:
    """-> (loss[1], stats[A,3], state): ``state`` is the opaque uint8 buffer for p2p_bwd (empty unless
    n_class > 0 -- analytic mode, include/slcl.h -- and keep_state)."""
    dev = require_cuda(a, b, a_meta, b_meta, shift, weight)
    lib = _lib.load()
    _p2p_check(a, b, a_meta, b_meta, shift, weight)
    na, dp = a.shape
    m = b.shape[0]
    _selfcol_check(a_selfcol, na, "a_selfcol")
    if n_class == 0 and keep_state:
        raise ValueError("keep_state needs n_class > 0 (analytic mode)")
    stats = torch.empty((na, 3), dtype=_F32, device=dev)
    loss = torch.empty(1, dtype=_F32, device=dev)
    keep = n_class > 0 and keep_state
    state = torch.empty(lib.slcl_p2p_state_bytes(na, dp) if keep else 0, dtype=torch.uint8, device=dev)
    ws = _ws(lib.slcl_p2p_workspace_bytes(na, m, dp), dev)
    with _guard(dev):
        st = lib.slcl_p2p_fwd(ptr(a), ptr(b), na, m, dp, ptr(a_meta), ptr(b_meta), ptr(a_selfcol), int(n_class), int(n_batch),
                              ptr(shift.contiguous()), ptr(weight.contiguous()), float(temperature), ptr(stats), ptr(loss),
                              ptr(state) if keep else None, ptr(ws), ws.numel(), stream_ptr(dev))
    check(st, "slcl_p2p_fwd")
    return loss, stats, state


@p2p_fwd.register_fake
def _(a, b, a_meta, b_meta, shift, weight, temperature, n_class=0, a_selfcol=None, keep_state=False, n_batch=1):
    # the real op returns the opaque backward state (slcl_p2p_state_bytes: a pure function of the shapes, no device
    # needed) when it is kept, an empty tensor otherwise
    n_state = _lib.load().slcl_p2p_state_bytes(a.shape[0], a.shape[1]) if (n_class > 0 and keep_state) else 0
    return (shift.new_empty(1), shift.new_empty((a.shape[0], 3)), torch.empty(n_state, dtype=torch.uint8, device=a.device))


@torch.library.custom_op("slcl::p2p_bwd", mutates_args=(), device_types="cuda")
def p2p_bwd(a: Tensor, b: Tensor, dim: int, a_meta: Tensor, b_meta: Tensor, shift: Tensor, weight: Tensor,
            temperature: float, stats: Tensor, grad_out: Tensor, need_a: bool, need_b: bool, n_class: int = 0,
            a_selfcol: Optional[Tensor] = None, b_selfrow: Optional[Tensor] = None,
            state: Optional[Tensor] = None, n_batch: int = 1) -> Tuple[Tensor, Tensor]:
    """-> (d_a [A, dim], d_b [M, dim]) fp32 (empty when not needed)."""
    dev = require_cuda(a, b, a_meta, b_meta, shift, weight, stats, grad_out)
    lib = _lib.load()
    _p2p_check(a, b, a_meta, b_meta, shift, weight)
    na, dp = a.shape
    m = b.shape[0]
    _selfcol_check(a_selfcol, na, "a_selfcol")
    _selfcol_check(b_selfrow, m, "b_selfrow")
    if state is not None and state.numel() == 0:
        state = None
    if state is not None and (state.dtype != torch.uint8 or state.numel() < lib.slcl_p2p_state_bytes(na, dp)
                              or not state.is_contiguous()):
        raise ValueError("state must be the uint8 buffer returned by p2p_fwd(..., keep_state=True)")
    d_a = torch.empty((na, dim) if need_a else (0, dim), dtype=_F32, device=dev)
    d_b = torch.empty((m, dim) if need_b else (0, dim), dtype=_F32, device=dev)
    ws = _ws(lib.slcl_p2p_workspace_bytes(na, m, dp), dev)
    g = grad_out.to(_F32).reshape(1).contiguous()
    with _guard(dev):
        st = lib.slcl_p2p_bwd(ptr(a), ptr(b), na, m, dp, dim, ptr(a_meta), ptr(b_meta), ptr(a_selfcol), ptr(b_selfrow),
                              int(n_class), int(n_batch), ptr(shift.contiguous()), ptr(weight.contiguous()), float(temperature),
                              ptr(stats.contiguous()), ptr(state), ptr(g),
                              ptr(d_a) if need_a else None, ptr(d_b) if need_b else None, ptr(ws), ws.numel(), stream_ptr(dev))
    check(st, "slcl_p2p_bwd")
    return d_a, d_b


@p2p_bwd.register_fake
def _(a, b, dim, a_meta, b_meta, shift, weight, temperature, stats, grad_out, need_a, need_b, n_class=0, a_selfcol=None,
      b_selfrow=None, state=None, n_batch=1):
    return (shift.new_empty((a.shape[0] if need_a else 0, dim)), shift.new_empty((b.shape[0] if need_b else 0, dim)))


P2P_STATE_FIELDS = ("u", "bsum", "absum", "colshift", "alpha", "beta")


def p2p_state_layout(n_anchor: int, dim_padded: int) -> dict:
    """Byte offsets of the fields of the analytic backward state (slcl_p2p_state_layout) plus its ``total`` size."""
    off = (C.c_int64 * 7)()
    check(_lib.load().slcl_p2p_state_layout(int(n_anchor), int(dim_padded), off), "slcl_p2p_state_layout")
    return dict(zip(P2P_STATE_FIELDS + ("total",), list(off)))


@torch.library.custom_op("slcl::p2p_state_assemble", mutates_args=(), device_types="cuda")
def p2p_state_assemble(alpha: Tensor, beta: Tensor, colshift: Tensor, absum_parts: Tensor, dim_padded: int,
                       n_class: int, n_batch: int = 1) -> Tensor:
    """Backward state for p2p_bwd(need_b only) over the anchors of all ranks (slcl_p2p_state_assemble_batched): per-anchor
    constants [A] in the order the d_b sweep reads them (rank-major; batch-major for ``n_batch`` block-diagonal batches),
    ABsum tables [parts, n_batch * n_class * (dim_padded + 1)] summed in rank order."""
    dev = require_cuda(alpha, beta, colshift, absum_parts)
    lib = _lib.load()
    na = alpha.numel()
    for t in (alpha, beta, colshift, absum_parts):
        if t.dtype != _F32 or not t.is_contiguous():
            raise ValueError("state pieces must be contiguous float32")
    if beta.numel() != na or colshift.numel() != na or absum_parts.dim() != 2 or \
            absum_parts.shape[1] != n_batch * n_class * (dim_padded + 1):
        raise ValueError("alpha / beta / colshift [A] and absum_parts [parts, n_batch * n_class * (dim_padded + 1)]")
    state = torch.empty(lib.slcl_p2p_state_bytes(na, dim_padded), dtype=torch.uint8, device=dev)
    with _guard(dev):
        st = lib.slcl_p2p_state_assemble_batched(ptr(state), na, dim_padded, n_class, int(n_batch), ptr(alpha), ptr(beta),
                                                 ptr(colshift), ptr(absum_parts), absum_parts.shape[0], stream_ptr(dev))
    check(st, "slcl_p2p_state_assemble_batched")
    return state


@p2p_state_assemble.register_fake
def _(alpha, beta, colshift, absum_parts, dim_padded, n_class, n_batch=1):
    return torch.empty(_lib.load().slcl_p2p_state_bytes(alpha.numel(), dim_padded), dtype=torch.uint8, device=alpha.device)


# ----------------------------------------------------------------------------
# segmentation losses / entropy map (SURVEY.md 8(f)-2)
# ----------------------------------------------------------------------------
@torch.library.custom_op("slcl::seg_fwd", mutates_args=(), device_types="cuda")
def seg_fwd(logits: Tensor, labels: Tensor) -> Tuple[Tensor, Tensor]:
    """-> (losses[3] = {ce, dice, jaccard}, stats[B,K,4])"""
    dev = require_cuda(logits, labels)
    lib = _lib.load()
    if logits.dim() != 4 or logits.dtype != _F32:
        raise ValueError("logits must be float32 [B, K, H, W]")
    logits = logits.contiguous()
    b, k, h, w = logits.shape
    labels = labels.reshape(b, -1).long().contiguous()
    if labels.shape[1] != h * w:
        raise ValueError("labels must be [B, H, W] at the resolution of the logits")
    stats = torch.empty((b, k, 4), dtype=_F32, device=dev)
    losses = torch.empty(3, dtype=_F32, device=dev)
    ws = _ws(lib.slcl_seg_workspace_bytes(b, h * w, k), dev)
    with _guard(dev):
        st = lib.slcl_seg_fwd(ptr(logits), ptr(labels), b, k, h * w, ptr(stats), ptr(losses), ptr(ws), ws.numel(),
                              stream_ptr(dev))
    check(st, "slcl_seg_fwd")
    return losses, stats


@seg_fwd.register_fake
def _(logits, labels):
    return logits.new_empty(3), logits.new_empty((logits.shape[0], logits.shape[1], 4))


@torch.library.custom_op("slcl::seg_bwd", mutates_args=(), device_types="cuda")
def seg_bwd(logits: Tensor, labels: Tensor, stats: Tensor, grad_losses: Tensor) -> Tensor:
    dev = require_cuda(logits, labels, stats, grad_losses)
    lib = _lib.load()
    logits = logits.contiguous()
    b, k, h, w = logits.shape
    labels = labels.reshape(b, -1).long().contiguous()
    g = grad_losses.to(_F32).reshape(3).contiguous()
    dlogits = torch.empty_like(logits)
    with _guard(dev):
        st = lib.slcl_seg_bwd(ptr(logits), ptr(labels), b, k, h * w, ptr(stats.contiguous()), ptr(g), ptr(dlogits),
                              stream_ptr(dev))
    check(st, "slcl_seg_bwd")
    return dlogits


@seg_bwd.register_fake
def _(logits, labels, stats, grad_losses):
    return torch.empty_like(logits)


def seg_vec_len(n_class: int) -> int:
    """Length of the data-parallel vector {inter_k, card_k, n_valid, sum ce, sum dice_bk, n_images} (fp64)."""
    return 2 * int(n_class) + 4


def _seg_inputs(logits: Tensor, labels: Tensor):
    if logits.dim() != 4 or logits.dtype != _F32:
        raise ValueError("logits must be float32 [B, K, H, W]")
    logits = logits.contiguous()
    b, k, h, w = logits.shape
    labels = labels.reshape(b, -1).long().contiguous()
    if labels.shape[1] != h * w:
        raise ValueError("labels must be [B, H, W] at the resolution of the logits")
    return logits, labels


@torch.library.custom_op("slcl::seg_fwd_peer", mutates_args=(), device_types="cuda")
def seg_fwd_peer(logits: Tensor, labels: Tensor, peer_ptrs: int, rank: int, world: int, capacity_words: int,
                 timeout_s: float) -> Tuple[Tensor, Tensor, Tensor]:
    """Segmentation losses of the ranks' concatenated batches, exchanged through the peer mailboxes inside the
    finaliser (slcl.peer.PeerMailbox.args()).  -> (GLOBAL losses[3], local stats[B,K,4], GLOBAL vec[2K+4] fp64)."""
    dev = require_cuda(logits, labels)
    lib = _lib.load()
    logits, labels = _seg_inputs(logits, labels)
    b, k, h, w = logits.shape
    if capacity_words < 2 * seg_vec_len(k):
        raise ValueError(f"seg losses over {k} classes exchange {seg_vec_len(k)} doubles: the mailbox needs "
                         f"capacity_words >= {2 * seg_vec_len(k)}, it has {capacity_words}")
    stats = torch.empty((b, k, 4), dtype=_F32, device=dev)
    vec = torch.empty(seg_vec_len(k), dtype=torch.float64, device=dev)
    losses = torch.empty(3, dtype=_F32, device=dev)
    ws = _ws(lib.slcl_seg_workspace_bytes(b, h * w, k), dev)
    peer = PeerT(peer_ptrs, rank, world, capacity_words, timeout_s)
    with _guard(dev):
        st = lib.slcl_seg_fwd_peer(ptr(logits), ptr(labels), b, k, h * w, ptr(stats), ptr(vec), ptr(losses), C.byref(peer),
                                   ptr(ws), ws.numel(), stream_ptr(dev))
    check(st, "slcl_seg_fwd_peer")
    return losses, stats, vec


@seg_fwd_peer.register_fake
def _(logits, labels, peer_ptrs, rank, world, capacity_words, timeout_s):
    b, k = logits.shape[0], logits.shape[1]
    return logits.new_empty(3), logits.new_empty((b, k, 4)), logits.new_empty(seg_vec_len(k), dtype=torch.float64)


@torch.library.custom_op("slcl::seg_fwd_local", mutates_args=(), device_types="cuda")
def seg_fwd_local(logits: Tensor, labels: Tensor) -> Tuple[Tensor, Tensor]:
    """-> (stats[B,K,4], this rank's vec[2K+4] fp64); sum vec over the ranks, then seg_finish."""
    dev = require_cuda(logits, labels)
    lib = _lib.load()
    logits, labels = _seg_inputs(logits, labels)
    b, k, h, w = logits.shape
    stats = torch.empty((b, k, 4), dtype=_F32, device=dev)
    vec = torch.empty(seg_vec_len(k), dtype=torch.float64, device=dev)
    ws = _ws(lib.slcl_seg_workspace_bytes(b, h * w, k), dev)
    with _guard(dev):
        st = lib.slcl_seg_fwd_local(ptr(logits), ptr(labels), b, k, h * w, ptr(stats), ptr(vec), ptr(ws), ws.numel(),
                                    stream_ptr(dev))
    check(st, "slcl_seg_fwd_local")
    return stats, vec


@seg_fwd_local.register_fake
def _(logits, labels):
    b, k = logits.shape[0], logits.shape[1]
    return logits.new_empty((b, k, 4)), logits.new_empty(seg_vec_len(k), dtype=torch.float64)


@torch.library.custom_op("slcl::seg_finish", mutates_args=(), device_types="cuda")
def seg_finish(vec: Tensor, n_class: int) -> Tensor:
    """losses[3] = {ce, dice, jaccard} from a vector summed over the ranks (the peer finaliser's arithmetic)."""
    dev = require_cuda(vec)
    if vec.dtype != torch.float64 or vec.numel() != seg_vec_len(n_class):
        raise ValueError(f"vec must be float64 [{seg_vec_len(n_class)}]")
    v = vec.contiguous()
    losses = torch.empty(3, dtype=_F32, device=dev)
    with _guard(dev):
        st = _lib.load().slcl_seg_finish(ptr(v), int(n_class), ptr(losses), stream_ptr(dev))
    check(st, "slcl_seg_finish")
    return losses


@seg_finish.register_fake
def _(vec, n_class):
    return vec.new_empty(3, dtype=_F32)


@torch.library.custom_op("slcl::seg_bwd_global", mutates_args=(), device_types="cuda")
def seg_bwd_global(logits: Tensor, labels: Tensor, stats: Tensor, vec: Tensor, grad_losses: Tensor) -> Tensor:
    """This rank's dlogits of the global losses: local stats, global vec (seg_fwd_peer / summed seg_fwd_local)."""
    dev = require_cuda(logits, labels, stats, vec, grad_losses)
    lib = _lib.load()
    logits = logits.contiguous()
    b, k, h, w = logits.shape
    if vec.dtype != torch.float64 or vec.numel() != seg_vec_len(k):
        raise ValueError(f"vec must be float64 [{seg_vec_len(k)}]")
    labels = labels.reshape(b, -1).long().contiguous()
    g = grad_losses.to(_F32).reshape(3).contiguous()
    dlogits = torch.empty_like(logits)
    with _guard(dev):
        st = lib.slcl_seg_bwd_global(ptr(logits), ptr(labels), b, k, h * w, ptr(stats.contiguous()), ptr(vec.contiguous()),
                                     ptr(g), ptr(dlogits), stream_ptr(dev))
    check(st, "slcl_seg_bwd_global")
    return dlogits


@seg_bwd_global.register_fake
def _(logits, labels, stats, vec, grad_losses):
    return torch.empty_like(logits)


@torch.library.custom_op("slcl::entropy_map", mutates_args=(), device_types="cuda")
def entropy_map(prob: Tensor) -> Tensor:
    dev = require_cuda(prob)
    lib = _lib.load()
    p = prob.to(_F32).contiguous()
    out = torch.empty_like(p)
    with _guard(dev):
        st = lib.slcl_entropy_map(ptr(p), p.numel(), p.shape[1], ptr(out), None, None, stream_ptr(dev))
    check(st, "slcl_entropy_map")
    return out


@entropy_map.register_fake
def _(prob):
    return torch.empty_like(prob)


@torch.library.custom_op("slcl::entropy_map_bwd", mutates_args=(), device_types="cuda")
def entropy_map_bwd(prob: Tensor, grad_out: Tensor) -> Tensor:
    dev = require_cuda(prob, grad_out)
    lib = _lib.load()
    p = prob.to(_F32).contiguous()
    g = grad_out.to(_F32).contiguous()
    dp = torch.empty_like(p)
    with _guard(dev):
        st = lib.slcl_entropy_map(ptr(p), p.numel(), p.shape[1], None, ptr(g), ptr(dp), stream_ptr(dev))
    check(st, "slcl_entropy_map")
    return dp


@entropy_map_bwd.register_fake
def _(prob, grad_out):
    return torch.empty_like(prob)


# ----------------------------------------------------------------------------
# eager fast path
# ----------------------------------------------------------------------------
class _EagerOps:
    """``dispatch.<op>(...)``: in plain eager mode call the op BODY registered above directly (the same Python function
    the dispatcher would reach, ~20 us of dispatch cheaper per call -- the MCCL loss section makes ~30 such calls per
    step and is host-launch-bound); under torch.compile / fake tensors go through ``torch.ops.slcl`` as usual."""

    def __getattr__(self, name):
        op_def = globals().get(name)
        body = getattr(op_def, "_init_fn", None)
        registered = getattr(torch.ops.slcl, name)
        if body is None:
            return registered

        def call(*args, **kwargs):
            if torch.compiler.is_compiling():
                return registered(*args, **kwargs)
            return body(*args, **kwargs)

        setattr(self, name, call)          # cache: __getattr__ is not consulted again for this name
        return call


dispatch = _EagerOps()
