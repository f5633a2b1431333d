"""Import the *real* reference loss functions (TEST INFRASTRUCTURE).

The reference is a checkout of the original Soft-Labeled-Contrastive-Learning
project at ``oracle/_ref`` (git-ignored: it is not part of this repository) or
wherever ``SLCL_REFERENCE_ROOT`` points.  This loader is used by
``oracle/make_golden.py`` (to produce the committed fixtures under
``tests/golden/``) and by CPU tests that are skipped when the reference tree is
absent.  Recipe: SURVEY.md appendix B -- stub the four
missing third-party modules that ``utils/utils_.py`` imports but the hot path
never uses, and keep tensors on the host by making ``Tensor.cuda`` the
identity while the reference functions run.
"""
from __future__ import annotations

import contextlib
import inspect
import os
import sys
import types

import torch

REFERENCE_ROOT = os.environ.get("SLCL_REFERENCE_ROOT", os.path.join(os.path.dirname(os.path.abspath(__file__)), "_ref"))


def available() -> bool:
    return os.path.isfile(os.path.join(REFERENCE_ROOT, "utils", "loss.py"))


@contextlib.contextmanager
def host_tensors():
    """While active, ``Tensor.cuda()`` returns the tensor unchanged (CPU oracle)."""
    saved = torch.Tensor.cuda
    torch.Tensor.cuda = lambda self, *a, **k: self
    try:
        yield
    finally:
        torch.Tensor.cuda = saved


_cache = {}


def load():
    """Returns a namespace with the reference callables of the hot path, plus
    ``cal_centroid_repaired`` (utils/utils_.py:479-565 with the missing list
    initialisation inserted before the class loop at :516)."""
    if "ns" in _cache:
        return _cache["ns"]
    if not available():
        raise RuntimeError(f"reference tree not found at {REFERENCE_ROOT}")
    for name in ("nibabel", "skimage", "skimage.measure", "SimpleITK", "easydict"):
        sys.modules.setdefault(name, types.ModuleType(name))
    sys.modules["skimage"].measure = sys.modules["skimage.measure"]
    sys.modules["easydict"].EasyDict = dict
    # the reference's top-level package is called ``utils``; import it under an
    # isolated sys.path entry and drop it again so it cannot shadow anything.
    sys.path.insert(0, REFERENCE_ROOT)
    try:
        for stale in [m for m in sys.modules if m == "utils" or m.startswith("utils.")]:
            del sys.modules[stale]
        import utils.loss as ref_loss            # noqa: E402
        import utils.losses as ref_losses        # noqa: E402
        import utils.utils_ as ref_utils         # noqa: E402
    finally:
        sys.path.remove(REFERENCE_ROOT)

    src = inspect.getsource(ref_utils.cal_centroid)
    marker = "            for k_cls in range(n_class):\n                if weighted_ave:"
    assert marker in src, "reference cal_centroid changed; repair recipe no longer applies"
    fixed = src.replace(marker, "            current_partition_centroids_list_inner = []\n" + marker, 1)
    fixed = fixed.replace("def cal_centroid(", "def cal_centroid_repaired(", 1)
    scope = dict(vars(ref_utils))
    exec(compile(fixed, "<cal_centroid_repaired>", "exec"), scope)

    ns = types.SimpleNamespace(
        MPCL=ref_loss.MPCL, mpcl_loss_calc=ref_loss.mpcl_loss_calc,
        ContrastiveLoss=ref_loss.ContrastiveLoss, SupConLoss=ref_loss.SupConLoss,
        LocalConLoss=ref_loss.LocalConLoss, BlockConLoss=ref_loss.BlockConLoss,
        SupConLoss_dup=ref_losses.SupConLoss, ISCL=ref_losses.InterpolatedSupervisedContrastiveLoss,
        cal_centroid=ref_utils.cal_centroid, cal_centroid_repaired=scope["cal_centroid_repaired"],
        loss_calc=ref_loss.loss_calc, dice_loss=ref_loss.dice_loss, jaccard_loss=ref_loss.jaccard_loss,
        prob_2_entropy=ref_utils.prob_2_entropy,
        update_class_center_iter=ref_utils.update_class_center_iter,
        generate_pseudo_label=ref_utils.generate_pseudo_label,
        class_center_file=os.path.join(REFERENCE_ROOT, "class_center_ct_f0.npy"),
    )
    _cache["ns"] = ns
    return ns
