"""ctypes binding of libslcl.so (the C ABI declared in include/slcl.h).

There is no CPU fallback: if the library is missing, or an op is called with a
non-CUDA tensor, this module raises.  ``SLCL_AUTOBUILD=1`` lets the loader run
``build.py`` (nvcc) once when the .so is absent; otherwise build it explicitly
with ``python soft-labeled-contrastive-learning_b200/build.py``.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("SLCL_LIB_PATH", os.path.join(_HERE, "libslcl.so"))   # override: kernel-tuning variants

SLCL_OK = 0
MAX_CLASSES = 8
MAX_WEIGHT_COLS = 16


class SlclError(RuntimeError):
    pass


class MapT(C.Structure):
    """slcl_map_t"""
    _fields_ = [("batch", C.c_int64), ("channels", C.c_int64), ("pixels", C.c_int64),
                ("stride_b", C.c_int64), ("stride_c", C.c_int64), ("stride_p", C.c_int64)]


class ProtoParamsT(C.Structure):
    """slcl_proto_params_t"""
    _fields_ = [("n_class", C.c_int), ("temperature", C.c_float), ("base_temperature", C.c_float),
                ("margin", C.c_float), ("easy_margin", C.c_int), ("normalize", C.c_int)]


class PeerT(C.Structure):
    """slcl_peer_t"""
    _fields_ = [("mailboxes_dev", C.c_void_p), ("rank", C.c_int), ("world", C.c_int), ("capacity_words", C.c_int64),
                ("timeout_s", C.c_double)]


_P = C.c_void_p
_I64 = C.c_int64
_SZ = C.c_size_t

# name -> (restype, argtypes); mirrors include/slcl.h one to one
SIGNATURES = {
    "slcl_version": (C.c_int, []),
    "slcl_strerror": (C.c_char_p, [C.c_int]),
    "slcl_last_cuda_error": (C.c_char_p, []),
    "slcl_proto_workspace_bytes": (_SZ, [_I64]),
    "slcl_proto_fwd": (C.c_int, [_P, C.POINTER(MapT), _P, _P, _P, _P, C.POINTER(ProtoParamsT), _P, _P, _P, _P, _SZ, _P]),
    "slcl_proto_fwd_peer": (C.c_int, [_P, C.POINTER(MapT), _P, _P, _P, _P, C.POINTER(ProtoParamsT), _P, _P, _P, C.POINTER(PeerT),
                                      C.c_int, _P, _SZ, _P]),
    "slcl_proto_bwd_peer": (C.c_int, [_P, C.POINTER(MapT), _P, _P, _P, _P, C.POINTER(ProtoParamsT), _P, C.POINTER(PeerT), C.c_int,
                                      _P]),
    "slcl_proto_fwd_target_peer": (C.c_int, [_P, C.POINTER(MapT), _P, C.POINTER(ProtoParamsT), C.c_float, _P, _P, _P, _P, _P,
                                             C.POINTER(PeerT), _P, _SZ, _P]),
    "slcl_proto_fwd_target": (C.c_int, [_P, C.POINTER(MapT), _P, C.POINTER(ProtoParamsT), C.c_float, _P, _P, _P, _P, _P, _P, _SZ, _P]),
    "slcl_target_step_workspace_bytes": (_SZ, [_I64, C.c_int]),
    "slcl_target_step": (C.c_int, [_P, _I64, _I64, _I64, _P, C.POINTER(ProtoParamsT), C.c_float, C.c_int, _P, _P, _P, _P, _P, _P, _P,
                                   C.c_float, _P, _P, C.POINTER(PeerT), _P, _SZ, _P]),
    "slcl_proto_rescale": (C.c_int, [_P, C.c_int, _P]),
    "slcl_peer_mailbox_bytes": (_SZ, [C.c_int, _I64]),
    "slcl_proto_rescale_peer": (C.c_int, [_P, C.c_int, C.POINTER(PeerT), _P]),
    "slcl_peer_allreduce_f64": (C.c_int, [_P, _I64, C.POINTER(PeerT), _P]),
    "slcl_class_centres_update": (C.c_int, [_P, _I64, _I64, _I64, _P, C.c_int, _P, C.c_float, _P, _P, C.POINTER(PeerT), _P, _SZ,
                                            _P]),
    "slcl_centroids_fwd": (C.c_int, [_P, _I64, _I64, _I64, _P, _P, C.c_int, C.c_float, _P, C.c_int, C.c_int, _P, C.c_float,
                                     _P, _P, _P, C.POINTER(PeerT), _P, _SZ, _P]),
    "slcl_proto_bwd": (C.c_int, [_P, C.POINTER(MapT), _P, _P, _P, _P, C.POINTER(ProtoParamsT), _P, _P]),
    "slcl_proto_bwd_aux": (C.c_int, [_P, C.POINTER(MapT), _P, _P, _P, _P, _P, _P, C.POINTER(ProtoParamsT), _P, _P, _P]),
    "slcl_proto_bwd_centres_workspace_bytes": (_SZ, [_I64, _I64, C.c_int]),
    "slcl_proto_bwd_centres": (C.c_int, [_P, C.POINTER(MapT), _P, _P, _P, _P, C.POINTER(ProtoParamsT), _P, _P, _SZ, _P]),
    "slcl_pseudo_label": (C.c_int, [_P, C.POINTER(MapT), _P, C.c_int, C.c_float, _P, _P, _P, _SZ, _P]),
    "slcl_class_sums_workspace_bytes": (_SZ, [_I64, _I64, _I64, C.c_int]),
    "slcl_class_sums": (C.c_int, [_P, _I64, _I64, _I64, _P, _P, C.c_int, C.c_float, _P, C.c_int, C.c_int, _P, _P, _SZ, _P]),
    "slcl_ema_finalize": (C.c_int, [_P, _P, C.c_float, C.c_int, _I64, _P, _P]),
    "slcl_centroid_finalize": (C.c_int, [_P, _P, C.c_float, C.c_int, C.c_int, _I64, _P, _P, _P]),
    "slcl_centroid_bwd_workspace_bytes": (_SZ, [_I64, C.c_int]),
    "slcl_centroid_bwd": (C.c_int, [_P, _I64, _I64, _I64, _P, _P, C.c_int, C.c_float, _P, C.c_int, C.c_int, _P, _P,
                                    C.c_float, _P, _P, _P, _SZ, _P]),
    "slcl_centroid_loss": (C.c_int, [_P, _P, C.c_int, _I64, C.c_int, C.c_int, C.c_int, C.c_int, _P, _P, _P, _P]),
    "slcl_mccl_losses_workspace_bytes": (_SZ, [C.c_int, C.c_int, _I64]),
    "slcl_mccl_losses": (C.c_int, [_P, _P, _P, C.c_int, C.c_int, _I64, C.c_int, C.c_int, C.c_int, C.c_float, C.c_float, C.c_float,
                                   _P, _P, _P, _P, _P, _SZ, _P]),
    "slcl_compact_workspace_bytes": (_SZ, [_I64, C.c_int]),
    "slcl_compact_by_class": (C.c_int, [_P, _I64, C.c_int, _P, _P, _P, _P, _SZ, _P]),
    "slcl_sample_balanced_workspace_bytes": (_SZ, [_I64, C.c_int]),
    "slcl_sample_balanced": (C.c_int, [_P, _P, _I64, C.c_int, _I64, _P, _P, _I64, _P, _P, _P, _SZ, _P]),
    "slcl_self_maps": (C.c_int, [_P, _I64, _P, _I64, _I64, _P, _P, _P, _P]),
    "slcl_scatter_rows_by_map": (C.c_int, [_P, _I64, _I64, _I64, C.c_int, _P, _P, _P, _P, _P, _P, _P, _P]),
    "slcl_tile_weights": (C.c_int, [_P, _I64, _I64, C.c_int, _P, _P, _P]),
    "slcl_rows_meta": (C.c_int, [_P, _I64, _P, _I64, _P, _P]),
    "slcl_gather_unit_rows": (C.c_int, [_P, _I64, _I64, _I64, _P, _I64, C.c_int, _P, _I64, _P, _P, _P]),
    "slcl_scatter_rows_bwd": (C.c_int, [_P, _I64, _I64, _I64, _P, _I64, C.c_int, _P, _P, _P, _P]),
    "slcl_p2p_shift": (C.c_int, [_P, _I64, _P, _I64, C.c_float, _P, _P]),
    "slcl_seg_workspace_bytes": (_SZ, [_I64, _I64, C.c_int]),
    "slcl_seg_fwd": (C.c_int, [_P, _P, _I64, C.c_int, _I64, _P, _P, _P, _SZ, _P]),
    "slcl_seg_bwd": (C.c_int, [_P, _P, _I64, C.c_int, _I64, _P, _P, _P, _P]),
    # segmentation losses over the global batch of data-parallel ranks (utils/loss.py:11-103)
    "slcl_seg_fwd_peer": (C.c_int, [_P, _P, _I64, C.c_int, _I64, _P, _P, _P, C.POINTER(PeerT), _P, _SZ, _P]),
    "slcl_seg_fwd_local": (C.c_int, [_P, _P, _I64, C.c_int, _I64, _P, _P, _P, _SZ, _P]),
    "slcl_seg_finish": (C.c_int, [_P, C.c_int, _P, _P]),
    "slcl_seg_bwd_global": (C.c_int, [_P, _P, _I64, C.c_int, _I64, _P, _P, _P, _P, _P]),
    "slcl_entropy_map": (C.c_int, [_P, _I64, C.c_int, _P, _P, _P, _P]),
    "slcl_p2p_workspace_bytes": (_SZ, [_I64, _I64, _I64]),
    "slcl_p2p_state_bytes": (_SZ, [_I64, _I64]),
    "slcl_p2p_fwd": (C.c_int, [_P, _P, _I64, _I64, _I64, _P, _P, _P, C.c_int, C.c_int, _P, _P, C.c_float, _P, _P, _P, _P, _SZ,
                               _P]),
    "slcl_p2p_bwd": (C.c_int, [_P, _P, _I64, _I64, _I64, _I64, _P, _P, _P, _P, C.c_int, C.c_int, _P, _P, C.c_float, _P, _P, _P,
                               _P, _P, _P, _SZ, _P]),
    "slcl_peer_rows_region_bytes": (_SZ, [_I64]),
    "slcl_peer_allgather": (C.c_int, [_P, _I64, _P, _P, C.POINTER(PeerT), _P, _I64, _P]),
    "slcl_p2p_state_layout": (C.c_int, [_I64, _I64, _P]),
    "slcl_p2p_state_assemble": (C.c_int, [_P, _I64, _I64, C.c_int, _P, _P, _P, _P, C.c_int, _P]),
    "slcl_p2p_state_assemble_batched": (C.c_int, [_P, _I64, _I64, C.c_int, C.c_int, _P, _P, _P, _P, C.c_int, _P]),
}

_lib: Optional[C.CDLL] = None


def load() -> C.CDLL:
    """Load libslcl.so (once).  Raises SlclError when it is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH) and os.environ.get("SLCL_AUTOBUILD") == "1":
        import importlib.util
        spec = importlib.util.spec_from_file_location("slcl_build", os.path.join(os.path.dirname(_HERE), "build.py"))
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
        mod.build()
    if not os.path.exists(LIB_PATH):
        raise SlclError(f"{LIB_PATH} not found: build it with "
                        f"`python soft-labeled-contrastive-learning_b200/build.py` (there is no CPU fallback)")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)           # AttributeError if the .so lacks a declared symbol
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(status: int, what: str) -> None:
    if status == SLCL_OK:
        return
    lib = load()
    msg = lib.slcl_strerror(status).decode()
    if status == -4:
        msg += ": " + lib.slcl_last_cuda_error().decode()
    if status == -1:
        raise ValueError(f"{what}: {msg}")
    raise SlclError(f"{what}: {msg}")


def ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    """Device pointer of a tensor (None -> NULL)."""
    if t is None:
        return None
    return t.data_ptr()


_raw_stream = None if os.environ.get("SLCL_STREAM_OBJECT") else getattr(torch._C, "_cuda_getCurrentRawStream", None)
# (the handle without building a Stream object; SLCL_STREAM_OBJECT=1 forces the public-API route)


def stream_ptr(device: torch.device) -> int:
    """cudaStream_t of PyTorch's current stream on ``device``.  ``torch.cuda.current_stream()`` costs ~9 us per call
    (it constructs a Stream object); every op makes one such call and the small-shape paths are host-bound."""
    if _raw_stream is not None:
        idx = device.index
        return _raw_stream(torch.cuda.current_device() if idx is None else idx)
    return torch.cuda.current_stream(device).cuda_stream


def require_cuda(*tensors: Optional[torch.Tensor]) -> torch.device:
    dev = None
    for t in tensors:
        if t is None:
            continue
        if not t.is_cuda:
            raise SlclError("slcl ops run on CUDA tensors only (B200 / sm_100a); there is no CPU path")
        if dev is None:
            dev = t.device
        elif t.device != dev:
            raise ValueError("all tensors of one slcl call must be on the same CUDA device")
    if dev is None:
        raise ValueError("no tensor argument")
    return dev
