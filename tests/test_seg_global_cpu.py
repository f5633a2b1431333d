"""CPU checks of the group= segmentation losses: the new C entry points are declared and bound, refuse bad arguments
before anything is launched, and the Python layer raises its argument errors before any exchange."""
import ctypes as C
import inspect

import pytest
import torch

NEW = ("slcl_seg_fwd_peer", "slcl_seg_fwd_local", "slcl_seg_finish", "slcl_seg_bwd_global")


def _stub_mailbox(world=2, capacity_words=8192):
    """A PeerMailbox as the Python layer sees it (no device memory): the argument checks run before it is used."""
    from slcl.peer import PeerMailbox
    box = PeerMailbox.__new__(PeerMailbox)
    box.world, box.rank, box.capacity_words, box.timeout_s = world, 0, capacity_words, 1.0
    return box


def test_new_entry_points_are_declared_and_bound():
    import os
    import re
    from slcl import _lib
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    txt = re.sub(r"/\*.*?\*/", "", open(os.path.join(root, "include", "slcl.h")).read(), flags=re.S)
    lib = _lib.load()
    for name in NEW:
        assert re.search(r"\b" + name + r"\s*\(", txt), name
        assert name in _lib.SIGNATURES
        assert hasattr(lib, name)
    assert lib.slcl_version() == 115


def test_c_entries_refuse_bad_arguments_without_a_launch():
    from slcl import _lib
    lib = _lib.load()
    ws = lib.slcl_seg_workspace_bytes(2, 64, 4)
    ok = _lib.PeerT(16, 0, 2, 2 * (2 * 4 + 4), 1.0)
    small = _lib.PeerT(16, 0, 2, 2 * (2 * 4 + 4) - 1, 1.0)
    bad_rank = _lib.PeerT(16, 2, 2, 64, 1.0)
    assert lib.slcl_seg_fwd_peer(16, 16, 2, 4, 64, 16, 16, 16, C.byref(small), 16, ws, None) == -1   # capacity < 2 (2K+4)
    assert lib.slcl_seg_fwd_peer(16, 16, 2, 4, 64, 16, 16, 16, C.byref(bad_rank), 16, ws, None) == -1
    assert lib.slcl_seg_fwd_peer(16, 16, 2, 4, 64, 16, 16, 16, None, 16, ws, None) == -1
    assert lib.slcl_seg_fwd_peer(16, 16, 2, 4, 64, 16, None, 16, C.byref(ok), 16, ws, None) == -1     # no vec
    assert lib.slcl_seg_fwd_peer(16, 16, 2, 9, 64, 16, 16, 16, C.byref(ok), 16, ws, None) == -1       # K > 8
    assert lib.slcl_seg_fwd_peer(16, 16, 2, 4, 64, 16, 16, 16, C.byref(ok), 16, ws - 1, None) == -3   # workspace
    assert lib.slcl_seg_fwd_local(16, 16, 2, 4, 64, 16, None, 16, ws, None) == -1
    assert lib.slcl_seg_fwd_local(None, 16, 2, 4, 64, 16, 16, 16, ws, None) == -1
    assert lib.slcl_seg_finish(None, 4, 16, None) == -1
    assert lib.slcl_seg_finish(16, 1, 16, None) == -1
    assert lib.slcl_seg_bwd_global(16, 16, 2, 4, 64, 16, None, 16, 16, None) == -1
    assert lib.slcl_seg_bwd_global(16, 16, 0, 4, 64, 16, 16, 16, 16, None) == -1


def test_positional_signatures_kept_and_group_is_keyword_only():
    from slcl import seg
    for fn, pos in ((seg.seg_losses, ["pred", "label"]), (seg.loss_calc, ["pred", "label", "gpu", "jaccard"]),
                    (seg.jaccard_loss, ["true", "logits", "eps"]), (seg.dice_loss, ["pred", "target"])):
        params = inspect.signature(fn).parameters
        assert [n for n, p in params.items() if p.kind == p.POSITIONAL_OR_KEYWORD] == pos
        assert params["group"].kind == inspect.Parameter.KEYWORD_ONLY and params["group"].default is None


def test_argument_errors_before_any_exchange():
    from slcl import seg
    pred = torch.randn(2, 4, 8, 8)
    lab = torch.zeros(2, 8, 8, dtype=torch.long)
    with pytest.raises(TypeError):
        seg.seg_losses(pred, lab, group="world")
    box = _stub_mailbox()
    with pytest.raises(ValueError, match="label"):
        seg.loss_calc(pred, torch.zeros(2, 9, 9, dtype=torch.long), group=box)
    with pytest.raises(ValueError, match="float32"):
        seg.dice_loss(pred.double(), lab, group=box)
    with pytest.raises(ValueError, match="at most"):
        seg.seg_losses(torch.randn(2, 9, 8, 8), lab, group=box)
    with pytest.raises(ValueError, match="capacity_words"):
        seg.jaccard_loss(lab, pred, group=_stub_mailbox(capacity_words=2 * (2 * 4 + 4) - 2))
    with pytest.raises(NotImplementedError):
        seg.seg_losses(torch.randn(2, 1, 8, 8), lab, group=box)
    with pytest.raises(NotImplementedError):
        seg.jaccard_loss(lab, pred, eps=1e-6, group=box)


def test_world_of_one_resolves_to_the_single_rank_call():
    """A one-rank mailbox, and True without an initialised process group, take the single-rank path (which has no CPU
    fallback, so it raises here rather than exchanging)."""
    from slcl import seg
    from slcl._lib import SlclError
    assert seg._resolve_group(None) is None
    assert seg._resolve_group(_stub_mailbox(world=1)) is None
    assert seg._resolve_group(True) is None
    box = _stub_mailbox(world=2)
    assert seg._resolve_group(box) is box
    with pytest.raises(SlclError):
        seg.seg_losses(torch.randn(2, 4, 8, 8), torch.zeros(2, 8, 8, dtype=torch.long), group=True)
