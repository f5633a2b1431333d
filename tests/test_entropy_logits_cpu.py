"""CPU checks of prob_2_entropy(from_logits=True): argument errors are raised before anything reaches the device, the C
entry point refuses bad arguments before any launch, and the two ops are registered."""
import pytest
import torch


@pytest.mark.parametrize("z", [torch.randn(2, 4, 8), torch.randn(1, 2, 4, 8, 8), torch.randn(2, 4, 8, 8).double(),
                               torch.randn(2, 4, 8, 8).half(), torch.randn(2, 1, 8, 8), torch.randn(2, 9, 8, 8)],
                         ids=["3d", "5d", "float64", "float16", "k1", "k9"])
def test_from_logits_refuses_bad_logits(z):
    from slcl.seg import prob_2_entropy
    with pytest.raises(ValueError):
        prob_2_entropy(z, from_logits=True)
    with pytest.raises(ValueError):
        prob_2_entropy(z.requires_grad_(True), from_logits=True)


def test_from_logits_has_no_cpu_path():
    from slcl._lib import SlclError
    from slcl.seg import prob_2_entropy
    with pytest.raises(SlclError):
        prob_2_entropy(torch.randn(2, 4, 8, 8), from_logits=True)


def test_c_entry_refuses_bad_arguments_without_a_launch():
    from slcl import _lib
    lib = _lib.load()
    f = lib.slcl_entropy_map_logits
    assert f(None, 2, 4, 64, 16, None, None, None) == -1                 # no logits
    assert f(16, 0, 4, 64, 16, None, None, None) == -1                   # batch <= 0
    assert f(16, -1, 4, 64, 16, None, None, None) == -1
    assert f(16, 2, 4, 0, 16, None, None, None) == -1                    # pixels <= 0
    assert f(16, 2, 4, -5, 16, None, None, None) == -1
    for k in (-1, 0, 1, 9, 64):                                          # K outside [2, 8]
        assert f(16, 2, k, 64, 16, 16, 16, None) == -1
    assert f(16, 2, 4, 64, None, None, None, None) == -1                 # no output
    assert f(16, 2, 4, 64, None, 16, None, None) == -1                   # grad_out alone is no output
    assert f(16, 2, 4, 64, None, None, 16, None) == -1                   # dlogits without grad_out
    assert f(16, 2, 4, 64, 16, None, 16, None) == -1


def test_ops_are_registered():
    import slcl.ops  # noqa: F401  (registers torch.ops.slcl.*)
    fwd = torch.ops.slcl.entropy_map_logits.default._schema
    bwd = torch.ops.slcl.entropy_map_logits_bwd.default._schema
    assert [a.name for a in fwd.arguments] == ["logits"]
    assert [a.name for a in bwd.arguments] == ["logits", "grad_out"]
