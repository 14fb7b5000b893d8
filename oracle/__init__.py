"""CPU oracle for the Fast AutoAugment per-batch augmentation hot path.

TEST INFRASTRUCTURE ONLY.  Nothing under ``oracle/`` is part of the shipped
product: only ``tests/``, ``__graft_entry__.smoke()`` and the ``cpu_baseline`` /
``--impl reference`` legs of ``bench.py`` may import it, and there only as the
checker (or as the timed CPU baseline), never as the thing that is measured as
"ours" or shipped.  The product path (``fast_autoaugment_b200``) never imports
this package and fails loudly when its CUDA library is missing.

Two layers, both restating ``/root/reference`` (kakaobrain/fast-autoaugment @
2424224) for the path named by BASELINE.json:

* ``oracle.pil_path``  - the reference's own call sequence into Pillow /
  torchvision / the three global RNGs (``augmentations.py``, ``data.py``
  ``Augmentation`` + ``CutoutDefault``, ``aug_mixup.py``), restated table-driven.
  Same third-party C library as the reference, so it is also the honest CPU
  baseline ("port").
* ``oracle.np_model``  - a NumPy restatement of the *arithmetic inside* Pillow
  and torchvision for those calls (16.16 fixed-point nearest gather, fp32 blend,
  histogram LUTs, 3x3 SMOOTH, rectangle fill ...).  This is the specification
  the CUDA kernels are written against.

Pinning: the reference has no tests and no golden vectors of its own
(SURVEY.md section 4), and its arithmetic lives in an un-vendored, un-pinned
Pillow.  The oracle is therefore pinned against *outputs of the reference
itself run in the build container* (Pillow 12.2.0, torchvision 0.26.0, numpy
2.3.5, CPython 3.12): ``tests/golden/make_golden.py`` imports
``/root/reference`` and writes the fixtures under ``tests/golden/``; the
``-m "not gpu"`` tests check both oracle layers against those fixtures; no
test needs the reference itself.
"""
