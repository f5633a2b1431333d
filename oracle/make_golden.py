"""Generate tests/golden/reference_outputs.npz and reference_seg_outputs.npz by running the REAL reference functions
(TEST INFRASTRUCTURE; needs a checkout of the original project, see oracle/ref_loader.py):

    python -m oracle.make_golden

Each fixture stores the outputs (loss, gradients, labels, centres) of the
reference's own code on the seeded inputs of oracle/cases.py.  The committed
fixtures are what the oracle restatement and the CUDA path are compared with
wherever the original project is absent.  (tests/golden/reference_live_cases.npz
is recorded by tests/test_oracle_live_reference.py itself; see its docstring.)
"""
from __future__ import annotations

import os
import shutil

import numpy as np
import torch

from . import cases, ref_loader


def _np(t):
    return t.detach().cpu().numpy()


def main() -> None:
    torch.manual_seed(0)
    torch.set_num_threads(1)      # fixed reduction order for the fixtures
    ref = ref_loader.load()
    os.makedirs(cases.GOLDEN_DIR, exist_ok=True)
    dst = os.path.join(cases.GOLDEN_DIR, "class_center_ct_f0.npy")
    if not os.path.exists(dst):
        shutil.copyfile(ref.class_center_file, dst)       # data fixture (a-9), 640 B
    cc = cases.shipped_centres()
    out = {}

    with ref_loader.host_tensors():
        # ---- KAT 1: source prototype loss --------------------------------
        feas, labels = cases.kat1()
        f = feas.clone().requires_grad_(True)
        c = cc.clone().requires_grad_(True)
        loss = ref.mpcl_loss_calc(f, labels, c, ref.MPCL('cpu', num_class=4, temperature=.1, base_temperature=1, m=.4),
                                  tag='source')
        loss.backward()
        out.update(kat1_loss=_np(loss), kat1_dfeas=_np(f.grad), kat1_dcentres=_np(c.grad))

        # ---- KAT 2: pseudo labels + target loss --------------------------
        ft = cases.kat2()
        hard, sel = ref.generate_pseudo_label(ft, cc, .25)
        f = ft.clone().requires_grad_(True)
        loss = ref.mpcl_loss_calc(f, hard, cc, ref.MPCL('cpu', num_class=4, temperature=.1, base_temperature=1, m=.2),
                                  pixel_sel_loc=sel, tag='target')
        loss.backward()
        out.update(kat2_label=_np(hard), kat2_sel=_np(sel), kat2_loss=_np(loss), kat2_dfeas=_np(f.grad))

        # ---- KAT 3: EMA class centres -------------------------------------
        out.update(kat3_centres=_np(ref.update_class_center_iter(feas, labels, cc, m=.9)))
        lab_empty = labels.clone()
        lab_empty[lab_empty == 2] = 1                      # class 2 empty -> row keeps old centre
        out.update(kat3_empty_centres=_np(ref.update_class_center_iter(feas, lab_empty, cc, m=.9)))

        # ---- KAT 4: centroid contrastive loss -----------------------------
        cs, ct = cases.kat4()
        for name, kw in (("plain", {}), ("split", {"split": True}), ("bg", {"bg": True})):
            a = cs.clone().requires_grad_(True)
            b = ct.clone().requires_grad_(True)
            loss = ref.ContrastiveLoss(tau=5)(a, b, **kw)
            loss.backward()
            out.update({f"kat4_{name}_loss": _np(loss), f"kat4_{name}_ds": _np(a.grad), f"kat4_{name}_dt": _np(b.grad)})
        out.update(kat4_tau01_loss=_np(ref.ContrastiveLoss(tau=.1)(cs, ct)))

        # ---- KAT 5: hard centroids + EMA ----------------------------------
        c1, _, _ = ref.cal_centroid(feas, labels, momentum=.9)
        f = ft.clone().requires_grad_(True)
        c2, _, _ = ref.cal_centroid(f, labels, previous_centroid=c1.detach(), momentum=.9)
        (c2 * c2).sum().backward()
        out.update(kat5_c1=_np(c1), kat5_c2=_np(c2), kat5_dft=_np(f.grad))

        # ---- soft centroids (repaired reference) ---------------------------
        sft, probs = cases.soft_case()
        for name, kw in (("wtd", dict(weighted_ave=True)),
                         ("wtd_thd", dict(weighted_ave=True, threshold=0.6)),
                         ("hardpl_thd", dict(weighted_ave=False, threshold=0.6)),
                         ("wtd_ema", dict(weighted_ave=True, previous_centroid=cc, momentum=.9))):
            f = sft.clone().requires_grad_(True)
            p = probs.clone().requires_grad_(True)
            cen, _, _ = ref.cal_centroid_repaired(f, p, pseudo_label=True, **kw)
            src_c, _ = cases.kat4()
            loss = ref.ContrastiveLoss()(src_c, cen) + (cen * cen).sum()
            loss.backward()
            out.update({f"soft_{name}_cen": _np(cen), f"soft_{name}_loss": _np(loss), f"soft_{name}_dft": _np(f.grad),
                        f"soft_{name}_dp": _np(p.grad) if p.grad is not None else np.zeros(0, np.float32)})

        # ---- KAT 6 / 7: pixel <-> pixel ------------------------------------
        torch.backends.cudnn.allow_tf32 = False
        f5, lab = cases.kat6()
        f = f5.clone().requires_grad_(True)
        loss = ref.SupConLoss(.7)(f, lab)
        loss.backward()
        out.update(kat6_loss=_np(loss), kat6_dfeat=_np(f.grad))
        f = f5.clone().requires_grad_(True)
        loss = ref.SupConLoss(.7)(f)
        loss.backward()
        out.update(kat6_unlab_loss=_np(loss), kat6_unlab_dfeat=_np(f.grad))
        out.update(kat6_dup_loss=_np(ref.SupConLoss_dup(.7)(f5, lab)))
        f7, lab7 = cases.kat7()
        out.update(kat7_local=_np(ref.LocalConLoss(.7, 4)(f7, lab7)), kat7_block=_np(ref.BlockConLoss(.7, 32)(f7, lab7)))
        out.update(kat7_local_unlab=_np(ref.LocalConLoss(.7, 4)(f7)))

        # ---- KAT 8: soft positive mask --------------------------------------
        unit = torch.nn.functional.normalize(feas, p=2, dim=1).permute(0, 2, 3, 1).reshape(-1, 32)
        unit = unit.clone().requires_grad_(True)
        cen = torch.nn.functional.normalize(cc, p=2, dim=1).t()
        loss = ref.MPCL('cpu', num_class=4, temperature=.1, base_temperature=1, m=.4).forward(
            unit.unsqueeze(1), None, cen, mask=cases.kat8_mask())
        loss.backward()
        out.update(kat8_loss=_np(loss), kat8_dunit=_np(unit.grad))

        # ---- KAT 9: cfg1-like geometry, label down-sampling 256 -> 33 -------
        f9, lab9, cc9 = cases.kat9()
        f = f9.clone().requires_grad_(True)
        loss = ref.mpcl_loss_calc(f, lab9, cc9, ref.MPCL('cpu', num_class=5, temperature=.1, base_temperature=1, m=.4),
                                  tag='source')
        loss.backward()
        out.update(kat9_loss=_np(loss), kat9_dfeas_abs_sum=_np(f.grad.abs().sum()),
                   kat9_dfeas_head=_np(f.grad[:, :4, :3, :3]))

        # ---- ragged / out-of-range / selection case (K=5) --------------------
        rf, rl, rc, rsel = cases.ragged_case()
        f = rf.clone().requires_grad_(True)
        c = rc.clone().requires_grad_(True)
        loss = ref.mpcl_loss_calc(f, rl.view(-1), c, ref.MPCL('cpu', num_class=5, temperature=.07, base_temperature=.07, m=.5),
                                  pixel_sel_loc=rsel, tag='target')
        loss.backward()
        out.update(ragged_loss=_np(loss), ragged_dfeas=_np(f.grad), ragged_dcentres=_np(c.grad))
        hard, sel = ref.generate_pseudo_label(rf, rc, .1)
        out.update(ragged_label=_np(hard), ragged_sel=_np(sel))
        out.update(ragged_ema=_np(ref.update_class_center_iter(rf, rl, rc, m=.8, num_class=5)))
        f = rf.clone().requires_grad_(True)
        loss = ref.mpcl_loss_calc(f, rl, rc, ref.MPCL('cpu', num_class=5, temperature=.1, base_temperature=1, m=.4,
                                                      easy_margin=True), tag='source')
        loss.backward()
        out.update(ragged_easy_loss=_np(loss), ragged_easy_dfeas=_np(f.grad))

    seg = {}
    with ref_loader.host_tensors():
        logits, labels = cases.seg_case()
        for name, fn in (("ce", lambda z: ref.loss_calc(z, labels, 0, False)),
                         ("ce_jac", lambda z: ref.loss_calc(z, labels, 0, True)),
                         ("jac", lambda z: ref.jaccard_loss(labels, z)),
                         ("dice", lambda z: ref.dice_loss(z, labels)),
                         ("mpscl_seg", lambda z: ref.loss_calc(z, labels, 0, False) + ref.dice_loss(z, labels))):
            z = logits.clone().requires_grad_(True)
            val = fn(z)
            val.backward()
            seg[f"seg_{name}_loss"] = _np(val)
            seg[f"seg_{name}_dlogits"] = _np(z.grad)
        z = logits.clone().requires_grad_(True)
        ent = ref.prob_2_entropy(torch.softmax(z, dim=1))
        (ent * torch.linspace(0.5, 1.5, ent.numel()).view_as(ent)).sum().backward()
        seg["seg_entropy_map"] = _np(ent)
        seg["seg_entropy_dlogits"] = _np(z.grad)
    feats, l1, l2, dom, lam = cases.iscl_case()
    f = feats.clone().requires_grad_(True)
    val = ref.ISCL(0.5)(f, l1, l2, dom, lam)
    val.backward()
    seg["iscl_loss"] = _np(val)
    seg["iscl_dfeat"] = _np(f.grad)
    seg_path = os.path.join(cases.GOLDEN_DIR, "reference_seg_outputs.npz")
    np.savez_compressed(seg_path, **seg)
    print(f"wrote {seg_path}: {len(seg)} arrays")
    for k in sorted(seg):
        if seg[k].size == 1:
            print(f"  {k} = {float(seg[k]):.10g}")

    path = os.path.join(cases.GOLDEN_DIR, "reference_outputs.npz")
    np.savez_compressed(path, **out)
    print(f"wrote {path}: {len(out)} arrays, {os.path.getsize(path)} bytes")
    for k in sorted(out):
        if out[k].size == 1:
            print(f"  {k} = {float(out[k]):.10g}")


if __name__ == "__main__":
    main()
