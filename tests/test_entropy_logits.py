"""prob_2_entropy(z, from_logits=True): the entropy map of softmax(z, 1) from the segmentor's logits, the softmax fused
into the map's forward and backward kernels (Trainer_MPSCL.py:171-172 without the F.softmax).

Pinned to the reference's golden outputs, to an fp64 restatement (softmax in fp64, then the oracle's prob_2_entropy) on
both load paths of the kernel, and to the two-op chain softmax + prob_2_entropy it replaces.
"""
import os

import numpy as np
import pytest
import torch

from oracle import cases
from oracle import slcl_oracle as O

pytestmark = pytest.mark.gpu

RTOL = 1e-4


@pytest.fixture(autouse=True, scope="module")
def _register_ops():
    import slcl.ops  # noqa: F401


def dev():
    return torch.device("cuda:0")


def close(a, b, rtol=RTOL, atol=1e-6):
    torch.testing.assert_close(torch.as_tensor(a).detach().double().cpu(), torch.as_tensor(b).detach().double().cpu(),
                               rtol=rtol, atol=atol)


def grad_close(a, b, rtol=RTOL, floor=0.1):
    """rtol per element with an absolute floor of floor * rtol * max|b| (as test_gpu_parity.grad_close)."""
    b = torch.as_tensor(b).double()
    close(a, b, rtol=rtol, atol=rtol * (float(b.abs().max()) + 1e-30) * floor)


def fused(z, w):
    """(map, dL/dz) of the fused op for L = sum(map * w)."""
    z = z.detach().clone().requires_grad_(True)
    from slcl import seg
    e = seg.prob_2_entropy(z, from_logits=True)
    (e * w).sum().backward()
    return e.detach(), z.grad


def fp64(z, w):
    z = z.detach().double().requires_grad_(True)
    e = O.prob_2_entropy(torch.softmax(z, 1))
    (e * w.double()).sum().backward()
    return e.detach(), z.grad


def chain(z, w):
    from slcl import seg
    z = z.detach().clone().requires_grad_(True)
    e = seg.prob_2_entropy(torch.softmax(z, 1))
    (e * w).sum().backward()
    return e.detach(), z.grad


def draw(b, k, h, w, seed, scale=3.0):
    gen = torch.Generator(device=dev()).manual_seed(seed)
    z = scale * torch.randn(b, k, h, w, device=dev(), generator=gen)
    wt = 2 * torch.rand(b, k, h, w, device=dev(), generator=gen) - 1
    return z, wt


def check_fp64(z, wt):
    e, dz = fused(z, wt)
    e_ref, dz_ref = fp64(z, wt)
    close(e, e_ref, rtol=0.0, atol=1e-6)
    close(dz, dz_ref, rtol=1e-5, atol=1e-5 * float(dz_ref.abs().max()))


def test_vs_reference_golden():
    from slcl import seg
    gold = dict(np.load(os.path.join(cases.GOLDEN_DIR, "reference_seg_outputs.npz")))
    logits, _ = cases.seg_case()
    z = logits.to(dev()).requires_grad_(True)
    ent = seg.prob_2_entropy(z, from_logits=True)
    (ent * torch.linspace(0.5, 1.5, ent.numel(), device=dev()).view_as(ent)).sum().backward()
    close(ent, gold["seg_entropy_map"], atol=1e-7)
    grad_close(z.grad, gold["seg_entropy_dlogits"])


@pytest.mark.parametrize("shape", [(2, 4, 224, 224), (2, 8, 16, 16), (3, 5, 33, 33), (1, 2, 7, 5)],
                         ids=["vec4_cfg", "vec4_k8", "scalar_33", "scalar_tiny"])
def test_vs_fp64_shapes(shape):
    check_fp64(*draw(*shape, seed=sum(shape)))


@pytest.mark.parametrize("hw", [(32, 32), (9, 7)], ids=["vec4", "scalar"])
@pytest.mark.parametrize("k", [2, 3, 4, 5, 6, 7, 8])
def test_vs_fp64_every_k(k, hw):
    check_fp64(*draw(2, k, *hw, seed=100 * k + hw[0]))


def misaligned(t):
    """A contiguous copy of t one float past a 16-byte boundary."""
    buf = torch.empty(t.numel() + 1, device=t.device)
    v = buf[1:].view(t.shape)
    v.copy_(t)
    assert v.is_contiguous() and v.data_ptr() % 16 == 4
    return v


def spy_entropy_calls(monkeypatch):
    """Arguments of every slcl_entropy_map_logits call from here on."""
    from slcl import _lib
    lib = _lib.load()
    real = lib.slcl_entropy_map_logits
    calls = []

    def spy(*args):
        calls.append(args)
        return real(*args)
    monkeypatch.setattr(lib, "slcl_entropy_map_logits", spy)
    return calls


def entropy_kernels(fn):
    """Names of the entropy_logits_kernel launches fn makes."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return [ev.name for ev in prof.events()
            if ev.device_type == torch.autograd.DeviceType.CUDA and "entropy_logits_kernel" in ev.name]


def test_misaligned_view_takes_the_scalar_path(monkeypatch):
    """Contiguous logits one float past a 16-byte boundary (HW % 4 == 0 still) reach the kernel as they are, and the
    kernel takes the scalar loads (VEC = 1); the result equals the fp64 restatement and the aligned (vec4) run."""
    from slcl import seg
    b, k, h, w = 2, 4, 16, 16
    z0, wt = draw(b, k, h, w, seed=7)
    e0, dz0 = fused(z0, wt)
    zl = misaligned(z0).detach().requires_grad_(True)       # a leaf on the misaligned storage itself
    assert zl.data_ptr() % 16 == 4
    calls = spy_entropy_calls(monkeypatch)
    res = {}

    def run():
        res["e"] = seg.prob_2_entropy(zl, from_logits=True)
        (res["e"] * wt).sum().backward()
    names = entropy_kernels(run)
    assert [c[0] for c in calls] == [zl.data_ptr()] * 2            # forward and backward saw the misaligned pointer
    assert len(names) == 2 and all(f"entropy_logits_kernel<{k}, 1, " in n for n in names), names
    e, dz = res["e"].detach(), zl.grad
    e_ref, dz_ref = fp64(z0, wt)
    close(e, e_ref, rtol=0.0, atol=1e-6)
    close(dz, dz_ref, rtol=1e-5, atol=1e-5 * float(dz_ref.abs().max()))
    close(e, e0, rtol=1e-6, atol=1e-7)
    close(dz, dz0, rtol=1e-6, atol=1e-6 * float(dz0.abs().max()))
    assert all(f"entropy_logits_kernel<{k}, 4, " in n for n in entropy_kernels(lambda: fused(z0, wt)))


def test_misaligned_grad_out_takes_the_scalar_path(monkeypatch):
    """Aligned logits with a misaligned upstream gradient: the backward takes the scalar loads too."""
    op = torch.ops.slcl
    z, wt = draw(2, 4, 16, 16, seed=8)
    want = op.entropy_map_logits_bwd(z, wt)
    g = misaligned(wt)
    calls = spy_entropy_calls(monkeypatch)
    res = {}
    names = entropy_kernels(lambda: res.setdefault("dz", op.entropy_map_logits_bwd(z, g)))
    assert len(calls) == 1 and calls[0][5] == g.data_ptr()
    assert len(names) == 1 and "entropy_logits_kernel<4, 1, true>" in names[0], names
    close(res["dz"], want, rtol=1e-6, atol=1e-6 * float(want.abs().max()))


def test_channels_last_logits():
    z, wt = draw(2, 5, 24, 24, seed=11)
    zc = z.to(memory_format=torch.channels_last)
    assert not zc.is_contiguous()
    check_fp64(zc, wt)
    e, dz = fused(zc, wt)
    e0, dz0 = fused(z, wt)
    assert torch.equal(e, e0) and torch.equal(dz, dz0)


@pytest.mark.parametrize("k", [2, 4, 8])
def test_saturated_softmax(k):
    """Logits of scale 50: most pixels have one probability at 1 and the others at or near 0 (underflowed in fp32)."""
    z, wt = draw(2, k, 64, 64, seed=50 + k, scale=50.0)
    p = torch.softmax(z, 1)
    assert int((p == 0).sum()) > 0 and int((p == 1).sum()) > 0
    check_fp64(z, wt)
    e, dz = fused(z, wt)
    assert bool(torch.isfinite(e).all()) and bool(torch.isfinite(dz).all())


@pytest.mark.parametrize("shape", [(2, 4, 224, 224), (3, 5, 33, 33)], ids=["vec4", "scalar"])
def test_vs_softmax_then_prob_2_entropy(shape):
    z, wt = draw(*shape, seed=3 + sum(shape))
    e, dz = fused(z, wt)
    e_ref, dz_ref = chain(z, wt)
    close(e, e_ref, rtol=1e-5, atol=1e-6)
    close(dz, dz_ref, rtol=1e-5, atol=1e-5 * float(dz_ref.abs().max()))


def test_c_entry_writes_map_and_gradient_in_one_launch():
    """out and (grad_out, dlogits) together: the backward kernel also writes the map."""
    from slcl import _lib
    lib = _lib.load()
    z, wt = draw(2, 4, 16, 20, seed=21)
    e_ref, dz_ref = fused(z, wt)
    out, dz = torch.empty_like(z), torch.empty_like(z)
    st = lib.slcl_entropy_map_logits(z.data_ptr(), 2, 4, 16 * 20, out.data_ptr(), wt.data_ptr(), dz.data_ptr(),
                                     torch.cuda.current_stream().cuda_stream)
    assert st == 0
    torch.cuda.synchronize()
    assert torch.equal(out, e_ref) and torch.equal(dz, dz_ref)


def test_forward_only_is_one_launch_and_saves_nothing():
    from torch.profiler import ProfilerActivity, profile
    from slcl import seg
    z, _ = draw(2, 4, 32, 32, seed=31)
    zg = z.clone().requires_grad_(True)
    with torch.no_grad():
        want = seg.prob_2_entropy(zg, from_logits=True)
    torch.cuda.synchronize()
    for inp, no_grad in ((zg, True), (z, False)):
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            with torch.set_grad_enabled(not no_grad):
                e = seg.prob_2_entropy(inp, from_logits=True)
            torch.cuda.synchronize()
        kernels = [ev for ev in prof.events() if ev.device_type == torch.autograd.DeviceType.CUDA]
        assert len(kernels) == 1 and "entropy_logits_kernel" in kernels[0].name, [ev.name for ev in kernels]
        assert e.grad_fn is None and not e.requires_grad
        assert torch.equal(e, want)


def test_no_host_sync():
    from slcl import seg
    z, wt = draw(2, 4, 32, 32, seed=41)
    e_ref, dz_ref = fused(z, wt)
    zz = z.clone().requires_grad_(True)
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        e = seg.prob_2_entropy(zz, from_logits=True)
        (e * wt).sum().backward()
        with torch.no_grad():
            e2 = seg.prob_2_entropy(zz, from_logits=True)
    finally:
        torch.cuda.set_sync_debug_mode(0)
    torch.cuda.synchronize()
    assert torch.equal(e.detach(), e_ref) and torch.equal(e2, e_ref) and torch.equal(zz.grad, dz_ref)


def test_cuda_graph_replay_equals_eager():
    from slcl import seg
    z, wt = draw(2, 4, 64, 64, seed=51)
    e_ref, dz_ref = fused(z, wt)
    zz = z.clone().requires_grad_(True)

    def step():
        e = seg.prob_2_entropy(zz, from_logits=True)
        (e * wt).sum().backward()
        return e.detach()
    side = torch.cuda.Stream(dev())
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        step()
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    zz.grad = None
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        static_e = step()
    static_e.zero_()
    for _ in range(2):
        zz.grad.zero_()
        graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(static_e, e_ref) and torch.equal(zz.grad, dz_ref)
