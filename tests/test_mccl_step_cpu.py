"""CPU checks of slcl.loss.mccl_step: every argument error is raised before anything is launched or exchanged (the inputs
here are CPU tensors, so a launch could not even start), the C entry points refuse bad arguments before any launch, and
the ops are registered."""
import pytest
import torch


def inputs(b=2, c=8, h=8, w=8, k=4, aug=True):
    g = torch.Generator().manual_seed(0)
    d = dict(ft_s=torch.randn(b, c, h, w, generator=g), labels_s=torch.randint(0, k, (b, h, w), generator=g),
             ft_t=torch.randn(b, c, h, w, generator=g), pred_t=torch.randn(b, k, h, w, generator=g))
    if aug:
        d.update(ft_t_aug=torch.randn(b, c, h, w, generator=g), pred_t_aug=torch.randn(b, k, h, w, generator=g))
    return d


def call(d, **kw):
    from slcl.loss import mccl_step
    d = dict(d)
    return mccl_step(d.pop("ft_s"), d.pop("labels_s"), d.pop("ft_t"), d.pop("pred_t"), d.pop("ft_t_aug", None),
                     d.pop("pred_t_aug", None), **kw)


def _mailbox(capacity_words):
    from slcl.peer import PeerMailbox
    box = PeerMailbox.__new__(PeerMailbox)          # the fields the argument checks read; nothing is mapped
    box.world, box.rank, box.capacity_words, box.timeout_s, box.ptrs_dev = 2, 0, capacity_words, 1.0, 0
    return box


BAD = {
    "ft_t float64": lambda d: d.update(ft_t=d["ft_t"].double()),
    "ft_s not contiguous": lambda d: d.update(ft_s=d["ft_s"].transpose(2, 3)),
    "ft_t channels_last": lambda d: d.update(ft_t=d["ft_t"].contiguous(memory_format=torch.channels_last)),
    "ft_t 3-d": lambda d: d.update(ft_t=d["ft_t"][0]),
    "ft_t channels": lambda d: d.update(ft_t=d["ft_t"][:, :4].contiguous()),
    "ft_t_aug channels": lambda d: d.update(ft_t_aug=torch.randn(2, 16, 8, 8)),
    "ft_t resolution": lambda d: d.update(ft_t=torch.randn(2, 8, 4, 8), pred_t=torch.randn(2, 4, 4, 8)),
    "labels_s resolution": lambda d: d.update(labels_s=torch.zeros(2, 16, 16, dtype=torch.long)),
    "pred_t resolution": lambda d: d.update(pred_t=torch.randn(2, 4, 16, 16)),
    "pred_t classes": lambda d: d.update(pred_t=torch.randn(2, 5, 8, 8)),
    "pred_t_aug resolution": lambda d: d.update(pred_t_aug=torch.randn(2, 4, 4, 4)),
    "pred_t float64": lambda d: d.update(pred_t=d["pred_t"].double()),
    "aug map without pred": lambda d: d.pop("pred_t_aug"),
}


@pytest.mark.parametrize("case", list(BAD), ids=list(BAD))
def test_bad_maps_raise_value_error(case):
    d = inputs()
    BAD[case](d)
    with pytest.raises(ValueError):
        call(d, partition=2)


def test_batch_slices_of_the_concatenated_map_pass_the_checks():
    """dcdr_ft[:B] / dcdr_ft[B:] of the trainer's concatenated map are contiguous: they get past every check and only
    fail where a CUDA tensor is required."""
    from slcl._lib import SlclError
    cat = torch.randn(4, 8, 8, 8)
    d = inputs()
    d.update(ft_s=cat[:2], ft_t=cat[2:])
    with pytest.raises(SlclError):
        call(d, partition=2)


@pytest.mark.parametrize("k,parts", [(1, 1), (9, 1), (0, 1), (4, 5), (8, 3), (2, 0)])
def test_classes_and_partitions_out_of_range(k, parts):
    d = inputs(k=max(k, 1))
    with pytest.raises(ValueError):
        call(d, n_class=k, partition=parts)


def test_previous_centroid_and_part_id_shapes():
    with pytest.raises(ValueError):
        call(inputs(), previous_centroid_s=torch.zeros(3, 8))
    with pytest.raises(ValueError):
        call(inputs(), partition=2, part_id=torch.zeros(17, dtype=torch.int32))


def test_mailbox_too_small():
    # K = 4, P = 2, aug: 16 rows of C + 1 = 9 doubles -> 288 words
    with pytest.raises(ValueError, match="capacity_words"):
        call(inputs(), partition=2, group=_mailbox(287))
    with pytest.raises(ValueError, match="capacity_words"):
        call(inputs(aug=False), partition=2, group=_mailbox(12 * 9 * 2 - 2))


def test_no_cpu_path():
    from slcl._lib import SlclError
    with pytest.raises(SlclError):
        call(inputs(), partition=2, part_id=torch.zeros(128, dtype=torch.int32))


def test_c_entries_refuse_bad_arguments_without_a_launch():
    from slcl import _lib
    lib = _lib.load()
    ws = lib.slcl_mccl_step_workspace_bytes
    assert ws(2, 2, 2, 32, 64, 2, 4) > 0
    assert ws(2, 2, 0, 32, 64, 2, 4) < ws(2, 2, 2, 32, 64, 2, 4)
    for bad in [(0, 2, 2, 32, 64, 2, 4), (2, 0, 2, 32, 64, 2, 4), (2, 2, -1, 32, 64, 2, 4), (2, 2, 2, 0, 64, 2, 4),
                (2, 2, 2, 32, 0, 2, 4), (2, 2, 2, 32, 64, 0, 4), (2, 2, 2, 32, 64, 2, 1), (2, 2, 2, 32, 64, 1, 9),
                (2, 2, 2, 32, 64, 3, 8)]:
        assert ws(*bad) == 0, bad
    assert lib.slcl_mccl_step_finish_workspace_bytes(1, 32, 2, 4) > 0
    assert lib.slcl_mccl_step_finish_workspace_bytes(1, 32, 3, 8) == 0
    p = 16                                      # any non-null pointer: nothing is dereferenced before the checks fail

    def fwd(**kw):
        a = dict(feat_s=p, labels_s=p, batch_s=2, feat_t=p, pred_t=p, part_id=p, batch_t=2, feat_a=p, pred_a=p, batch_a=2,
                 channels=32, pixels=64, n_partitions=2, n_class=4, flags=1, threshold=0.0, previous_s=None, momentum=0.9,
                 split=0, bg=0, norm=1, inter_w=1.0, intra_w=1.0, cnr_w=4e-5, sums=p, centroids=p, losses=p,
                 d_centroids=p, peer=None, workspace=p, workspace_bytes=1 << 30, stream=None)
        a.update(kw)
        return lib.slcl_mccl_step_fwd(*a.values())
    assert fwd(feat_s=None) == -1
    assert fwd(labels_s=None) == -1
    assert fwd(pred_t=None) == -1
    assert fwd(part_id=None) == -1                          # P > 1 without partition ids
    assert fwd(pred_a=None) == -1                           # aug map without its labels
    assert fwd(batch_a=0) == -1                             # aug pointers with no batch
    assert fwd(n_class=9) == -1
    assert fwd(n_partitions=3, n_class=8) == -1
    assert fwd(flags=4) == -1                               # unknown flag bit
    assert fwd(losses=None) == -1
    assert fwd(workspace_bytes=16) == -3                    # SLCL_ERR_WORKSPACE, before any launch

    def bwd(**kw):
        a = dict(feat_t=p, pred_t=p, part_id=p, batch_t=2, feat_a=p, pred_a=p, batch_a=2, channels=32, pixels=64,
                 n_partitions=2, n_class=4, flags=1, threshold=0.0, sums=p, d_centroids=p, grad_out=p, dfeat_t=p,
                 dpred_t=p, dfeat_a=p, dpred_a=p, workspace=p, workspace_bytes=1 << 30, stream=None)
        a.update(kw)
        return lib.slcl_mccl_step_bwd(*a.values())
    assert bwd(grad_out=None) == -1
    assert bwd(dfeat_a=None) == -1
    assert bwd(flags=0) == -1                               # dpred without soft weights
    assert bwd(part_id=None) == -1
    assert bwd(workspace_bytes=16) == -3


def test_header_and_ctypes_table_agree_on_the_new_entries():
    import os
    import re
    from slcl import _lib
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    txt = re.sub(r"/\*.*?\*/", "", open(os.path.join(root, "include", "slcl.h")).read(), flags=re.S)
    for name in ("slcl_mccl_step_workspace_bytes", "slcl_mccl_step_finish_workspace_bytes", "slcl_mccl_step_fwd",
                 "slcl_mccl_step_fwd_local", "slcl_mccl_step_finish", "slcl_mccl_step_bwd"):
        m = re.search(r"\b" + name + r"\s*\(([^;{]*?)\)\s*;", txt, flags=re.S)
        assert m, name
        assert len(m.group(1).split(",")) == len(_lib.SIGNATURES[name][1]), name


def test_ops_are_registered():
    import slcl.ops  # noqa: F401
    names = {n: [a.name for a in getattr(torch.ops.slcl, n).default._schema.arguments]
             for n in ("mccl_step_fwd", "mccl_step_fwd_local", "mccl_step_finish", "mccl_step_bwd")}
    assert names["mccl_step_fwd"][:8] == ["feat_s", "labels_s", "feat_t", "pred_t", "part_id", "feat_a", "pred_a",
                                          "previous_s"]
    assert names["mccl_step_bwd"][-3:] == ["d_centroids", "grad_out", "need_dpred"]
