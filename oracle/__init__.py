"""CPU oracle for the SLCL loss hot path.

TEST INFRASTRUCTURE ONLY.  Nothing under ``oracle/`` is part of the product:
only ``tests/``, ``__graft_entry__.smoke()`` and the ``cpu_baseline`` /
``--impl reference`` legs of ``bench.py`` may import it, and only as the
checker (or as the timed CPU baseline), never as the thing shipped.  The
product package (``soft-labeled-contrastive-learning_b200/slcl``) never imports
this module and raises if its CUDA library is missing.

Pinning status (see DESIGN.md "Oracle"):
  * prototype path, EMA class centres, pseudo labels, hard centroids,
    ContrastiveLoss, SupCon/LocalCon/BlockCon: PINNED -- the restatement in
    ``slcl_oracle.py`` is checked against outputs of the reference's own
    functions (``tests/golden/reference_*outputs.npz``, made by ``oracle/make_golden.py``
    which imports a checkout of the original project, see ``ref_loader.py``) and against
    the nine known-answer values of SURVEY.md section 8(c);
    ``tests/test_oracle_live_reference.py`` checks it on randomised inputs
    (losses and gradients, 33 cases; seg losses and ISCL included) against the
    stored ``tests/golden/reference_live_cases.npz`` and, where a checkout of
    the original is present, against the reference's callables run live.
  * soft-label centroid path: pinned against the reference function with the
    one-line repair described in SURVEY.md section 0 (the shipped function
    raises NameError).
  * reversed-Monte-Carlo partition sampler, class-balanced anchor sampler and
    the rectangular (anchors x contrast set) pixel-to-pixel loss: PARITY
    UNPINNED -- the reference fork contains no implementation of them; the
    oracle *defines* them (spec in SURVEY.md section 8(c)) and the square
    special case of the rectangular loss is pinned against ``SupConLoss``.
"""
