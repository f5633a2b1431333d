"""Oracle pinned against the REAL reference on randomised inputs.

``tests/test_oracle_golden.py`` checks the restatement (oracle/slcl_oracle.py) against committed outputs of the
reference on the KAT inputs; this file goes further -- several seeds, shapes the fixtures do not contain, hard / soft /
thresholded labels, empty classes, out-of-range labels, both margin modes -- losses AND gradients.  Nothing here
touches the product or a GPU.

Every case compares the restatement with the reference outputs stored in tests/golden/reference_live_cases.npz (its
``provenance`` entry says where they came from).  Where a checkout of the original project is present (``oracle/_ref``
or ``SLCL_REFERENCE_ROOT``, see oracle/ref_loader.py) the reference's own callables are also run side by side, and

    SLCL_RECORD_LIVE_CASES=1 python -m pytest tests/test_oracle_live_reference.py

rewrites the stored file from those live outputs.
"""
import os
import re

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import cases, ref_loader
from oracle import slcl_oracle as O

RTOL = 1e-6
STORED = os.path.join(cases.GOLDEN_DIR, "reference_live_cases.npz")
RECORD = os.environ.get("SLCL_RECORD_LIVE_CASES") == "1"
_recorded = {}


@pytest.fixture(scope="module")
def ref():
    """The original project's callables, or None without a checkout (then only the stored outputs are compared)."""
    if RECORD and not ref_loader.available():
        pytest.fail("SLCL_RECORD_LIVE_CASES=1 needs a checkout of the original project (oracle/_ref or SLCL_REFERENCE_ROOT)")
    return ref_loader.load() if ref_loader.available() else None


@pytest.fixture(scope="module")
def stored():
    yield {} if RECORD else dict(np.load(STORED))
    if RECORD:
        np.savez_compressed(STORED, provenance=np.array(
            "outputs of the original project's own callables (oracle/ref_loader.py) on the inputs of "
            "tests/test_oracle_live_reference.py, recorded with SLCL_RECORD_LIVE_CASES=1"), **_recorded)


@pytest.fixture
def check(request, ref, stored):
    """check(live, got, **tol): `got` maps output names to the restatement's tensors.  Each is compared with the stored
    reference output of this case and, with a checkout of the original present, with ``live(ref)`` -- the same names
    computed by the reference's own callables.  tol: per-name dict(rtol=, atol=) overriding RTOL / 1e-7."""
    case = re.sub(r"\W+", "_", request.node.name).strip("_")

    def _check(live, got, **tol):
        want = live(ref) if ref is not None else None
        for name, value in got.items():
            kw = tol.get(name, {})
            if want is not None:
                same(value, want[name], **kw)
            if RECORD:
                _recorded[f"{case}__{name}"] = want[name].detach().cpu().numpy()
            else:
                same(value, torch.from_numpy(stored[f"{case}__{name}"]), **kw)
    return _check


def g(seed):
    return torch.Generator().manual_seed(seed)


def same(a, b, rtol=RTOL, atol=1e-7):
    # equal_nan: where the reference divides 0 by 0 (e.g. SupConLoss on an all-background crop, utils/loss.py:382-384)
    # the restatement must produce the same NaN
    torch.testing.assert_close(a.detach().float(), b.detach().float(), rtol=rtol, atol=atol, equal_nan=True)


@pytest.mark.parametrize("seed,b,c,h,w,k,m,easy,tag", [
    (11, 2, 16, 9, 7, 4, 0.4, False, "source"),       # odd map, labels at another resolution (nearest resize)
    (12, 1, 64, 16, 16, 5, 0.2, False, "target"),
    (13, 3, 8, 5, 11, 3, 0.5, True, "source"),        # easy margin
    (14, 2, 32, 12, 12, 8, 1.2, False, "target"),     # large margin: the cos <= th branch is taken often
])
def test_prototype_loss_and_gradient(check, seed, b, c, h, w, k, m, easy, tag):
    gen = g(seed)
    feas = torch.randn(b, c, h, w, generator=gen)
    centres = torch.randn(k, c, generator=gen)
    if tag == "source":
        labels = torch.randint(0, k + 1, (b, 2 * h + 1, 3 * w), generator=gen)      # k is out of range: all-zero one-hot row
        sel = None
    else:
        labels = torch.randint(0, k, (b * h * w,), generator=gen)
        sel = (torch.rand(b * h * w, generator=gen) > 0.4).float()

    def live(ref):
        fr = feas.clone().requires_grad_(True)
        with ref_loader.host_tensors():
            crit = ref.MPCL("cpu", num_class=k, temperature=0.1, m=m, base_temperature=1.0, easy_margin=easy)
            loss = ref.mpcl_loss_calc(fr, labels, centres, crit, pixel_sel_loc=sel, tag=tag)
        loss.backward()
        return {"loss": loss, "dfeas": fr.grad}
    fo = feas.clone().requires_grad_(True)
    got = O.mpcl_loss_calc(fo, labels, centres, O.MarginSpec(k, 0.1, m, 1.0, easy), pixel_sel_loc=sel, tag=tag)
    got.backward()
    check(live, {"loss": got, "dfeas": fo.grad}, dfeas=dict(atol=1e-9))


@pytest.mark.parametrize("seed", [21, 22, 23])
def test_soft_mask_forward(check, seed):
    gen = g(seed)
    n, c, k = 150, 24, 5
    unit = F.normalize(torch.randn(n, c, generator=gen), dim=1).unsqueeze(1)
    cen = F.normalize(torch.randn(k, c, generator=gen), dim=1).t().contiguous()
    mask = torch.softmax(2 * torch.randn(n, k, generator=gen), 1)

    def live(ref):
        with ref_loader.host_tensors():
            return {"loss": ref.MPCL("cpu", num_class=k, temperature=0.07, m=0.5, base_temperature=0.07)(unit, None, cen,
                                                                                                       mask=mask)}
    check(live, {"loss": O.mpcl_forward(O.MarginSpec(k, 0.07, 0.5, 0.07), unit, None, cen, mask=mask)})


@pytest.mark.parametrize("seed", [24, 25])
def test_soft_mask_and_pixel_sel_loc_gradients(check, seed):
    """The reference takes `mask` and `pixel_sel_loc` as tensors (utils/loss.py:516-517, :558-565): its autograd gives
    their gradients, and the restatement -- which the GPU test of slcl_proto_bwd_aux is checked against -- must agree."""
    gen = g(seed)
    n, c, k = 120, 16, 4
    unit = F.normalize(torch.randn(n, c, generator=gen), dim=1).unsqueeze(1)
    cen = F.normalize(torch.randn(k, c, generator=gen), dim=1).t().contiguous()
    mask = torch.softmax(2 * torch.randn(n, k, generator=gen), 1)
    sel = torch.rand(n, generator=gen)

    def live(ref):
        mr, sr = mask.clone().requires_grad_(True), sel.clone().requires_grad_(True)
        with ref_loader.host_tensors():
            loss = ref.MPCL("cpu", num_class=k, temperature=0.1, m=0.4, base_temperature=1.0)(unit, None, cen,
                                                                                             pixel_sel_loc=sr, mask=mr)
            loss.backward()
        return {"loss": loss, "dmask": mr.grad, "dsel": sr.grad}
    mo, so = mask.clone().requires_grad_(True), sel.clone().requires_grad_(True)
    got = O.mpcl_forward(O.MarginSpec(k, 0.1, 0.4, 1.0), unit, None, cen, pixel_sel_loc=so, mask=mo)
    got.backward()
    check(live, {"loss": got, "dmask": mo.grad, "dsel": so.grad}, dmask=dict(atol=1e-9), dsel=dict(atol=1e-9))


def test_more_than_one_view_fails_in_the_reference_too(ref):
    """MPCL with n_views > 1: mask.repeat(anchor_count, contrast_count) (utils/loss.py:548) makes a [V N, V K] mask
    against [V N, K] logits -- a RuntimeError in the reference (recorded here as the expected message); the restatement
    fails the same way, and the product raises the same type up front."""
    gen = g(26)
    feats = F.normalize(torch.randn(6, 2, 8, generator=gen), dim=2)
    cen = F.normalize(torch.randn(8, 4, generator=gen), dim=0)
    labels = torch.randint(0, 4, (6,), generator=gen)
    with pytest.raises(RuntimeError, match="must match the size of tensor b"):
        O.mpcl_forward(O.MarginSpec(4, 0.07, 0.5, 0.07), feats, labels, cen)
    if ref is not None:
        with ref_loader.host_tensors():
            with pytest.raises(RuntimeError, match="must match the size of tensor b"):
                ref.MPCL("cpu", num_class=4)(feats, labels, cen)


@pytest.mark.parametrize("seed,k,drop", [(31, 4, None), (32, 4, 2), (33, 5, 0)])
def test_ema_class_centres_with_empty_class(check, seed, k, drop):
    gen = g(seed)
    feas = torch.randn(3, 12, 10, 6, generator=gen)
    labels = torch.randint(0, k, (3, 10, 6), generator=gen)
    if drop is not None:
        labels[labels == drop] = (drop + 1) % k          # class `drop` is empty: its centre must stay
    centres = torch.randn(k, 12, generator=gen)

    def live(ref):
        with ref_loader.host_tensors():
            return {"centres": ref.update_class_center_iter(feas, labels, centres, m=0.8, num_class=k)}
    got = O.update_class_center_iter(feas, labels, centres, m=0.8, num_class=k)
    check(live, {"centres": got})
    if drop is not None:
        same(got[drop], 0.8 * centres[drop] + 0.2 * centres[drop])


@pytest.mark.parametrize("seed,th", [(41, 0.25), (42, 0.0), (43, 0.6)])
def test_pseudo_labels_bit_exact(check, seed, th):
    gen = g(seed)
    feas = torch.randn(2, 20, 13, 9, generator=gen)
    centres = torch.randn(5, 20, generator=gen)

    def live(ref):
        with ref_loader.host_tensors():
            lab_r, sel_r = ref.generate_pseudo_label(feas, centres, th)
        return {"label": lab_r.reshape(-1), "sel": sel_r.reshape(-1).float()}
    lab_o, sel_o = O.generate_pseudo_label(feas, centres, th)
    exact = dict(rtol=0, atol=0)
    check(live, {"label": lab_o, "sel": sel_o}, label=exact, sel=exact)


@pytest.mark.parametrize("seed,kw", [
    (51, dict(pseudo_label=False)),
    (52, dict(pseudo_label=True, weighted_ave=True)),
    (53, dict(pseudo_label=True, weighted_ave=False)),
    (54, dict(pseudo_label=True, weighted_ave=True, threshold=0.6)),
    (55, dict(pseudo_label=True, weighted_ave=False, threshold=0.5)),
])
def test_centroids_forward_and_gradients(check, seed, kw):
    gen = g(seed)
    b, c, h, w, k = 2, 10, 8, 12, 4
    feat = torch.randn(b, c, h, w, generator=gen)
    prev = torch.randn(k, c, generator=gen)
    if kw["pseudo_label"]:
        label = torch.softmax(3 * torch.randn(b, k, h, w, generator=gen), 1)
    else:
        label = torch.randint(0, k, (b, 2 * h, 2 * w), generator=gen)           # resized with 'nearest' inside
    with_dlab = kw["pseudo_label"] and kw["weighted_ave"]

    def run(fn):
        f = feat.clone().requires_grad_(True)
        lab = label.clone().requires_grad_(True) if kw["pseudo_label"] else label
        cen, ratio, std = fn(f, lab, previous_centroid=prev, momentum=0.9, n_class=k, **kw)
        assert ratio is None and list(std) == []
        (cen * torch.arange(1, k * c + 1).view(k, c).float()).sum().backward()
        out = {"cen": cen, "dfeat": f.grad}
        if with_dlab:
            out["dlabel"] = lab.grad
        return out
    check(lambda ref: run(ref.cal_centroid_repaired), run(O.cal_centroid), dfeat=dict(atol=1e-8), dlabel=dict(atol=1e-8))


@pytest.mark.parametrize("seed,bg,split", [(61, False, False), (62, True, False), (63, False, True), (64, True, True)])
def test_centroid_contrastive_loss(check, seed, bg, split):
    gen = g(seed)
    cs, ct = torch.randn(4, 32, generator=gen) * 3, torch.randn(4, 32, generator=gen) * 3
    check(lambda ref: {"loss": ref.ContrastiveLoss(tau=seed, n_class=4)(cs, ct, bg=bg, split=split)},   # tau is ignored
          {"loss": O.contrastive_loss(cs, ct, bg=bg, split=split)})


@pytest.mark.parametrize("seed,labelled", [(71, True), (72, False), (73, True)])
def test_pixel_to_pixel_family(check, seed, labelled):
    gen = g(seed)
    f5 = F.normalize(torch.randn(1, 2, 12, 64, 64, generator=gen), dim=2)
    lab = torch.randint(0, 4, (1, 2, 64, 64), generator=gen) if labelled else None
    if seed == 73:
        lab[:, :, :32, :32] = 0                                # one all-background 32 x 32 block: skipped by BlockConLoss
    small, small_lab = f5[..., :10, :10].contiguous(), None if lab is None else lab[..., :10, :10].contiguous()

    def live(ref):
        fr = small.clone().requires_grad_(True)
        loss = ref.SupConLoss(temperature=0.5)(fr, small_lab)
        loss.backward()
        return {"supcon": loss, "dsmall": fr.grad,
                "supcon_dup": ref.SupConLoss_dup(temperature=0.5)(small, small_lab),           # utils/losses.py copy
                "local": ref.LocalConLoss(0.7, 4)(f5, lab), "block": ref.BlockConLoss(0.7, 32)(f5, lab)}
    fo = small.clone().requires_grad_(True)
    got = O.supcon_loss(fo, small_lab, temperature=0.5)
    got.backward()
    loose = dict(rtol=1e-5)
    check(live, {"supcon": got, "dsmall": fo.grad, "supcon_dup": O.supcon_loss(small, small_lab, 0.5),
                 "local": O.local_con_loss(f5, lab, 0.7, 4), "block": O.block_con_loss(f5, lab, 0.7, 32)},
          supcon=loose, dsmall=dict(rtol=1e-4, atol=1e-7), supcon_dup=loose, local=loose, block=loose)


def test_pixel_to_pixel_all_background_returns_zero(check):
    f5 = F.normalize(torch.randn(1, 2, 8, 32, 32, generator=g(81)), dim=2)
    lab = torch.zeros(1, 2, 32, 32, dtype=torch.long)
    got = {"local": O.local_con_loss(f5, lab, 0.7, 4), "block": O.block_con_loss(f5, lab, 0.7, 32)}
    assert float(got["local"]) == 0.0 == float(got["block"])
    check(lambda ref: {"local": ref.LocalConLoss(0.7, 4)(f5, lab), "block": ref.BlockConLoss(0.7, 32)(f5, lab)}, got,
          local=dict(rtol=0, atol=0), block=dict(rtol=0, atol=0))


@pytest.mark.parametrize("seed", [91, 92])
def test_segmentation_losses_and_entropy(check, seed):
    gen = g(seed)
    pred = torch.randn(2, 4, 17, 9, generator=gen)
    lab = torch.randint(0, 4, (2, 17, 9), generator=gen)
    prob = torch.softmax(pred, 1)

    def live(ref):
        with ref_loader.host_tensors():
            out = {"ce": ref.loss_calc(pred, lab, jaccard=False), "ce_jac": ref.loss_calc(pred, lab, jaccard=True),
                   "dice": ref.dice_loss(pred, lab)}
        out["entropy"] = ref.prob_2_entropy(prob)
        return out
    check(live, {"ce": O.loss_calc(pred, lab, jaccard=False), "ce_jac": O.loss_calc(pred, lab, jaccard=True),
                 "dice": O.dice_loss(pred, lab), "entropy": O.prob_2_entropy(prob)})


@pytest.mark.parametrize("seed,t", [(101, 0.5), (102, 0.1)])
def test_iscl_loss_and_gradient(check, seed, t):
    """InterpolatedSupervisedContrastiveLoss (utils/losses.py:6-81): two label sets mixed per sample over one Gram matrix."""
    gen = g(seed)
    n, c = 48, 20
    feats = torch.randn(n, c, generator=gen)
    l1 = torch.randint(0, 4, (n,), generator=gen)
    l2 = torch.randint(0, 4, (n,), generator=gen)
    lam = torch.rand(n, generator=gen)
    dom = torch.where(lam >= 0.5, l1, l2)

    def live(ref):
        fr = feats.clone().requires_grad_(True)
        loss = ref.ISCL(t)(fr, l1, l2, dom, lam)
        loss.backward()
        return {"loss": loss, "dfeat": fr.grad}
    fo = feats.clone().requires_grad_(True)
    got = O.iscl_loss(fo, l1, l2, dom, lam, t)
    got.backward()
    check(live, {"loss": got, "dfeat": fo.grad}, loss=dict(rtol=1e-5), dfeat=dict(rtol=1e-4, atol=1e-7))
