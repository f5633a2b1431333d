"""CPU checks of slcl.loss.mpscl_step: every argument error is raised before anything is launched or exchanged (the inputs
here are CPU tensors, so a launch could not even start), the C entry points refuse bad arguments before any launch, and
the ops are registered with their schemas."""
import ctypes as C

import pytest
import torch


def inputs(b_s=2, b_t=3, c=8, h=8, w=8, k=4):
    g = torch.Generator().manual_seed(0)
    return dict(ft_s=torch.randn(b_s, c, h, w, generator=g), labels_s=torch.randint(0, k, (b_s, h, w), generator=g),
                ft_t=torch.randn(b_t, c, h, w, generator=g), centres=torch.randn(k, c, generator=g))


def modules(k=4, k_t=None):
    from slcl.loss import MPCL
    return (MPCL(None, num_class=k, temperature=1.0, m=0.4, base_temperature=1.0),
            MPCL(None, num_class=k if k_t is None else k_t, temperature=1.0, m=0.2, base_temperature=1.0))


def call(d, k=4, k_t=None, **kw):
    from slcl.loss import mpscl_step
    src, trg = modules(k if k >= 1 else 4, k_t)
    return mpscl_step(d["ft_s"], d["labels_s"], d["ft_t"], d["centres"], src, trg, num_class=k, **kw)


def _mailbox(capacity_words):
    from slcl.peer import PeerMailbox
    box = PeerMailbox.__new__(PeerMailbox)          # the fields the argument checks read; nothing is mapped
    box.world, box.rank, box.capacity_words, box.timeout_s, box.ptrs_dev = 2, 0, capacity_words, 1.0, 0
    return box


BAD = {
    "ft_s float64": lambda d: d.update(ft_s=d["ft_s"].double()),
    "ft_t float16": lambda d: d.update(ft_t=d["ft_t"].half()),
    "ft_s not contiguous": lambda d: d.update(ft_s=d["ft_s"].transpose(2, 3)),
    "ft_t channels_last": lambda d: d.update(ft_t=d["ft_t"].contiguous(memory_format=torch.channels_last)),
    "ft_t 3-d": lambda d: d.update(ft_t=d["ft_t"][0]),
    "ft_t channels": lambda d: d.update(ft_t=d["ft_t"][:, :4].contiguous()),
    "ft_t resolution": lambda d: d.update(ft_t=torch.randn(3, 8, 4, 8)),
    "labels_s resolution": lambda d: d.update(labels_s=torch.zeros(2, 16, 16, dtype=torch.long)),
    "labels_s batch": lambda d: d.update(labels_s=torch.zeros(3, 8, 8, dtype=torch.long)),
    "centres rows": lambda d: d.update(centres=torch.randn(5, 8)),
    "centres channels": lambda d: d.update(centres=torch.randn(4, 9)),
    "centres transposed": lambda d: d.update(centres=torch.randn(8, 4)),
    "centres require grad": lambda d: d.update(centres=d["centres"].requires_grad_(True)),
}


@pytest.mark.parametrize("case", list(BAD), ids=list(BAD))
def test_bad_inputs_raise_value_error(case):
    d = inputs()
    BAD[case](d)
    with pytest.raises(ValueError):
        call(d)


def test_batch_slices_of_the_concatenated_map_pass_the_checks():
    """dcdr_ft[:B] / dcdr_ft[B:] of a concatenated map are contiguous: they get past every check and only fail where a
    CUDA tensor is required."""
    from slcl._lib import SlclError
    cat = torch.randn(5, 8, 8, 8)
    d = inputs()
    d.update(ft_s=cat[:2], ft_t=cat[2:])
    with pytest.raises(SlclError):
        call(d)


@pytest.mark.parametrize("k", [0, 1, 9])
def test_classes_out_of_range(k):
    d = inputs(k=4)
    d["centres"] = torch.randn(max(k, 1), 8)
    with pytest.raises(ValueError):
        call(d, k=k, k_t=k)


def test_module_classes_must_match():
    with pytest.raises(ValueError, match="mpcl_src"):
        _call_modules(5, 4)
    with pytest.raises(ValueError, match="mpcl_trg"):
        _call_modules(4, 5)


def _call_modules(k_s, k_t):
    from slcl.loss import MPCL, mpscl_step
    d = inputs()
    return mpscl_step(d["ft_s"], d["labels_s"], d["ft_t"], d["centres"], MPCL(None, num_class=k_s),
                      MPCL(None, num_class=k_t), num_class=4)


def test_modules_must_be_mpcl():
    from slcl.loss import mpscl_step
    d = inputs()
    with pytest.raises(TypeError):
        mpscl_step(d["ft_s"], d["labels_s"], d["ft_t"], d["centres"], lambda *a: 0, modules()[1], num_class=4)


def test_mailbox_too_small():
    # K = 4, C = 8: 4 rows of 9 doubles -> 72 words
    with pytest.raises(ValueError, match="capacity_words"):
        call(inputs(), group=_mailbox(71))


def test_no_cpu_path():
    from slcl._lib import SlclError
    with pytest.raises(SlclError):
        call(inputs(), group=_mailbox(72))


def _map(b=2, c=32, hw=64):
    from slcl._lib import MapT
    return MapT(b, c, hw, c * hw, hw, 1)


def _params(k=4, t=0.07, normalize=1):
    from slcl._lib import ProtoParamsT
    return ProtoParamsT(k, t, t, 0.4, 0, normalize)


def test_c_entries_refuse_bad_arguments_without_a_launch():
    from slcl import _lib
    from slcl._lib import PeerT
    lib = _lib.load()
    ws = lib.slcl_mpscl_step_workspace_bytes
    assert ws(C.byref(_map(hw=1 << 16)), C.byref(_map(b=3, hw=1 << 16)), 4) > ws(C.byref(_map(hw=1 << 16)), C.byref(_map(b=1, hw=1 << 16)), 4) > 0
    assert ws(C.byref(_map()), C.byref(_map()), 1) == 0
    assert ws(C.byref(_map()), C.byref(_map()), 9) == 0
    assert ws(None, C.byref(_map()), 4) == 0
    p = 16                                      # any non-null pointer: nothing is dereferenced before the checks fail
    big = 1 << 30

    def fwd(**kw):
        a = dict(feat_s=p, map_s=C.byref(_map()), labels_s=p, feat_t=p, map_t=C.byref(_map(b=3)), old=p, m=0.9,
                 ps=C.byref(_params()), pt=C.byref(_params()), th=0.25, centres=p, cstate=p, stash_s=p, stash_t=p, label_t=p,
                 sel_t=p, scal_s=p, scal_t=p, peer=None, workspace=p, workspace_bytes=big, stream=None)
        a.update(kw)
        return lib.slcl_mpscl_step_fwd(*a.values())
    assert fwd(feat_s=None) == -1
    assert fwd(feat_t=None) == -1
    assert fwd(labels_s=None) == -1
    assert fwd(old=None) == -1
    assert fwd(scal_t=None) == -1
    assert fwd(map_t=C.byref(_map(c=16))) == -1                        # channel counts differ
    assert fwd(map_t=C.byref(_map(hw=60))) == -1                       # resolutions differ
    assert fwd(map_s=C.byref(_lib.MapT(2, 32, 64, 32 * 64, 1, 32))) == -1      # not dense NCHW
    assert fwd(ps=C.byref(_params(k=1)), pt=C.byref(_params(k=1))) == -1
    assert fwd(ps=C.byref(_params(k=9)), pt=C.byref(_params(k=9))) == -1
    assert fwd(pt=C.byref(_params(k=5))) == -1                          # the two losses' K differ
    assert fwd(pt=C.byref(_params(t=0.0))) == -1
    assert fwd(ps=C.byref(_params(normalize=0))) == -1
    peer = PeerT(p, 0, 2, 2 * 4 * 33 - 1, 1.0)
    assert fwd(peer=C.byref(peer)) == -1                                # mailbox smaller than 2 K (C+1) words
    assert fwd(workspace_bytes=16) == -3                                # SLCL_ERR_WORKSPACE, before any launch

    def local(**kw):
        a = dict(feat_s=p, map_s=C.byref(_map()), labels_s=p, feat_t=p, map_t=C.byref(_map()), centres=p,
                 ps=C.byref(_params()), pt=C.byref(_params()), th=0.25, cstate=p, stash_s=p, stash_t=p, label_t=p, sel_t=p,
                 pairs=p, workspace=p, workspace_bytes=big, stream=None)
        a.update(kw)
        return lib.slcl_mpscl_step_fwd_local(*a.values())
    assert local(pairs=None) == -1
    assert local(centres=None) == -1
    assert local(map_t=C.byref(_map(c=64))) == -1
    assert local(workspace_bytes=16) == -3
    assert lib.slcl_mpscl_step_finish(None, p, p, None) == -1
    assert lib.slcl_mpscl_step_finish(p, p, None, None) == -1

    def bwd(**kw):
        a = dict(feat_s=p, map_s=C.byref(_map()), feat_t=p, map_t=C.byref(_map()), stash_s=p, stash_t=p, cstate=p,
                 scal_s=p, scal_t=p, grad_s=p, grad_t=p, ps=C.byref(_params()), pt=C.byref(_params()), dfeat_s=p,
                 dfeat_t=p, stream=None)
        a.update(kw)
        return lib.slcl_mpscl_step_bwd(*a.values())
    assert bwd(grad_s=None, grad_t=None) == -1                          # nothing to differentiate
    assert bwd(dfeat_s=None) == -1
    assert bwd(grad_s=None, stash_t=None) == -1
    assert bwd(cstate=None) == -1
    assert bwd(map_t=C.byref(_map(c=16))) == -1
    assert bwd(ps=C.byref(_params(k=9)), pt=C.byref(_params(k=9))) == -1


def test_header_and_ctypes_table_agree_on_the_new_entries():
    import os
    import re
    from slcl import _lib
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    txt = re.sub(r"/\*.*?\*/", "", open(os.path.join(root, "include", "slcl.h")).read(), flags=re.S)
    for name in ("slcl_mpscl_step_workspace_bytes", "slcl_mpscl_step_fwd", "slcl_mpscl_step_fwd_local",
                 "slcl_mpscl_step_finish", "slcl_mpscl_step_bwd"):
        m = re.search(r"\b" + name + r"\s*\(([^;{]*?)\)\s*;", txt, flags=re.S)
        assert m, name
        assert len(m.group(1).split(",")) == len(_lib.SIGNATURES[name][1]), name


def test_ops_are_registered():
    import slcl.ops  # noqa: F401
    names = {n: [a.name for a in getattr(torch.ops.slcl, n).default._schema.arguments]
             for n in ("mpscl_step_fwd", "mpscl_step_fwd_local", "mpscl_step_finish", "mpscl_step_bwd")}
    assert names["mpscl_step_fwd"][:7] == ["feat_s", "labels_s", "feat_t", "old_centres", "m", "sel_threshold", "n_class"]
    assert names["mpscl_step_fwd"][-5:] == ["peer_ptrs", "rank", "world", "capacity_words", "timeout_s"]
    assert names["mpscl_step_fwd_local"][:5] == ["feat_s", "labels_s", "feat_t", "centres", "sel_threshold"]
    assert names["mpscl_step_finish"] == ["pairs"]
    assert names["mpscl_step_bwd"] == ["feat_s", "feat_t", "stash_s", "stash_t", "cstate", "scal", "grad_s", "grad_t",
                                       "n_class"]


def test_fake_kernels_give_the_output_shapes():
    from torch._subclasses.fake_tensor import FakeTensorMode
    import slcl.ops  # noqa: F401
    op = torch.ops.slcl
    with FakeTensorMode():
        fs, ft = torch.empty(2, 8, 4, 4, device="cuda"), torch.empty(3, 8, 4, 4, device="cuda")
        lab = torch.empty(32, dtype=torch.int64, device="cuda")
        cen = torch.empty(4, 8, device="cuda")
        scal, c2, cstate, st_s, st_t, label, sel = op.mpscl_step_fwd(fs, lab, ft, cen, 0.9, 0.25, 4, 1.0, 1.0, 0.4, False,
                                                                     1.0, 1.0, 0.2, False)
        assert scal.shape == (8,) and c2.shape == (4, 8) and cstate.shape == (36,)
        assert st_s.shape == (5, 32) and st_t.shape == (5, 48) and label.shape == (48,) and label.dtype == torch.int64
        pairs = op.mpscl_step_fwd_local(fs, lab, ft, cen, 0.25, 4, 1.0, 1.0, 0.4, False, 1.0, 1.0, 0.2, False)[0]
        assert pairs.shape == (4,) and op.mpscl_step_finish(pairs).shape == (8,)
        d_s, d_t = op.mpscl_step_bwd(fs, ft, st_s, st_t, cstate, scal, None, torch.empty(1, device="cuda"), 4)
        assert d_s.numel() == 0 and d_t.shape == ft.shape
