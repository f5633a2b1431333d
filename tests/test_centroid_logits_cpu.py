"""CPU checks of cal_centroid(from_logits=True): argument errors are raised before anything reaches the device, the C
entry points refuse a bad flags word before any launch, and the three ops carry the new trailing argument."""
import pytest
import torch


def test_from_logits_needs_pseudo_label():
    from slcl.utils_ import cal_centroid
    ft = torch.randn(2, 8, 4, 4)
    z = torch.randn(2, 4, 4, 4)
    with pytest.raises(ValueError, match="pseudo_label"):
        cal_centroid(ft, z, pseudo_label=False, n_class=4, from_logits=True)


@pytest.mark.parametrize("shape", [(2, 4, 8, 8), (2, 4, 4, 5), (2, 3, 4, 4), (1, 4, 4, 4), (2, 4, 4)])
def test_from_logits_needs_logits_at_feature_resolution(shape):
    """Bilinear interpolation of probabilities does not commute with a softmax: other resolutions are refused."""
    from slcl.utils_ import cal_centroid
    ft = torch.randn(2, 8, 4, 4)
    with pytest.raises(ValueError, match="resolution"):
        cal_centroid(ft, torch.randn(*shape), pseudo_label=True, n_class=4, weighted_ave=True, from_logits=True)


def test_c_entries_refuse_bad_flags_without_a_launch():
    from slcl import _lib
    lib = _lib.load()
    big = 1 << 24
    # SLCL_SOFT_LOGITS (2) with hard labels
    assert lib.slcl_class_sums(16, 1, 4, 16, 16, None, 2, 0.0, None, 1, 4, 16, 16, big, None) == -1
    assert lib.slcl_centroids_fwd(16, 1, 4, 16, 16, None, 2, 0.0, None, 1, 4, None, 0.9, 16, 16, 16, None, 16, big,
                                  None) == -1
    assert lib.slcl_centroid_bwd(16, 1, 4, 16, 16, None, 3, 0.0, None, 1, 4, 16, 16, 1.0, 16, None, 16, big, None) == -1
    # a bit above SLCL_SOFT_WEIGHTED | SLCL_SOFT_LOGITS
    for flags in (4, 5, 7, 1 << 30):
        assert lib.slcl_class_sums(16, 1, 4, 16, None, 16, flags, 0.0, None, 1, 4, 16, 16, big, None) == -1
        assert lib.slcl_centroids_fwd(16, 1, 4, 16, None, 16, flags, 0.0, None, 1, 4, None, 0.9, 16, 16, 16, None, 16, big,
                                      None) == -1
        assert lib.slcl_centroid_bwd(16, 1, 4, 16, None, 16, flags, 0.0, None, 1, 4, 16, 16, 1.0, 16, 16, 16, big,
                                     None) == -1
    # d(logits) asked for without the weighted bit: the arg-max weights have no gradient
    assert lib.slcl_centroid_bwd(16, 1, 4, 16, None, 16, 2, 0.0, None, 1, 4, 16, 16, 1.0, 16, 16, 16, big, None) == -1
    assert lib.slcl_centroid_bwd(16, 1, 4, 16, None, 16, 0, 0.0, None, 1, 4, 16, 16, 1.0, 16, 16, 16, big, None) == -1


@pytest.mark.parametrize("op", ["class_sums", "centroids_fwd", "centroid_bwd"])
def test_ops_take_a_trailing_from_logits(op):
    import slcl.ops  # noqa: F401  (registers torch.ops.slcl.*)
    args = getattr(torch.ops.slcl, op).default._schema.arguments
    assert args[-1].name == "from_logits"
    assert str(args[-1].type) == "bool" and args[-1].default_value is False
    assert [a.name for a in args[:5]] == ["feat", "labels", "probs", "weighted", "threshold"]
