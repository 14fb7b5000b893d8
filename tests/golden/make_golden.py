#!/usr/bin/env python
"""Generate the golden fixtures from the LIVE reference.

Run in the build container only (needs ``/root/reference``; it does not exist on
the GPU box).  Imports the reference in place, read-only, with two import shims
(``theconf`` is not installed; ``torch._six`` no longer exists - SURVEY.md 8c),
runs the reference's own ``apply_augment`` / ``Augmentation`` / ``CutoutDefault``
/ ``mixup`` and the exact ``transform_train`` of ``data.py:39-44,92,112`` on
seeded synthetic inputs, and writes

    tests/golden/golden_ops.npz      per-op outputs (19 ops x levels x 3 input kinds, 32x32 + 24x40)
    tests/golden/golden_chain.npz    policy outputs + full CIFAR chain fp32 + mixup
    tests/golden/golden_hashes.json  sha256 digests (incl. the SURVEY.md 8c table at 32 and 224, the inputs of
                                     golden_chain.npz, whole-policy outputs and the Lighting chain)

Environment that produced the committed files: Pillow 12.2.0, numpy 2.3.5,
torch 2.11.0, torchvision 0.26.0, CPython 3.12.3.
"""
import collections.abc
import hashlib
import json
import os
import random
import sys
import types

import numpy as np
import PIL
import PIL.Image
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
REF = "/root/reference"
sys.path.insert(0, os.path.dirname(HERE))
from helpers import GOLDEN_POLICY_BATCHES, LIVE_POLICY_RUNS, live_input, make_chain_inputs, sha_policy, synth_batch  # noqa: E402


def import_reference():
    # shim 1: theconf (data.py:16)
    tc = types.ModuleType("theconf")

    class _C:
        _d = {}

        @classmethod
        def get(cls):
            return cls._d
    tc.Config = _C
    tc.ConfigArgumentParser = object
    sys.modules["theconf"] = tc
    # shim 2: torch._six (networks/efficientnet_pytorch/condconv.py:4)
    six = types.ModuleType("torch._six")
    six.container_abcs = collections.abc
    sys.modules["torch._six"] = six
    sys.path.insert(0, REF)
    from FastAutoAugment import augmentations, archive, aug_mixup, data
    return augmentations, archive, aug_mixup, data


def sha(a) -> str:
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def synth(shape, kind, rng):
    """The three input families of SURVEY.md 8(d)."""
    h, w = shape
    if kind == 0:      # uniform noise
        return rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
    if kind == 1:      # low-contrast ramp + noise
        lo = int(rng.integers(0, 200))
        hi = int(rng.integers(lo + 1, 256))
        ramp = np.linspace(lo, hi, w)[None, :, None] + rng.normal(0, 8, (h, w, 3))
        return np.clip(ramp, 0, 255).astype(np.uint8)
    return np.broadcast_to(rng.integers(0, 256, 3, dtype=np.uint8), (h, w, 3)).copy()   # constant


ALL_OPS = ["ShearX", "ShearY", "TranslateX", "TranslateY", "Rotate", "AutoContrast", "Invert",
           "Equalize", "Solarize", "Posterize", "Contrast", "Color", "Brightness", "Sharpness",
           "Cutout", "CutoutAbs", "Posterize2", "TranslateXAbs", "TranslateYAbs"]
LEVELS = [0.0, 0.13, 0.5, 0.7, 1.0]


def main():
    aug, archive, aug_mixup, data = import_reference()
    hashes = {"env": {"pillow": PIL.__version__, "numpy": np.__version__, "torch": torch.__version__}}

    # ---- (1) SURVEY 8c table: rng(1234) noise, seed 0, level 0.7 (Posterize 0.3)
    table = {}
    for s in (32, 224):
        img = np.random.default_rng(1234).integers(0, 256, (s, s, 3), dtype=np.uint8)
        table["input_%d" % s] = sha(img)
        for name in ALL_OPS:
            random.seed(0)
            np.random.seed(0)
            lvl = 0.3 if name == "Posterize" else 0.7
            out = aug.apply_augment(PIL.Image.fromarray(img), name, lvl)
            table["%s_%d" % (name, s)] = sha(np.asarray(out))
    hashes["survey_table"] = table

    # ---- (2) per-op outputs, small images, explicit arrays
    rng = np.random.default_rng(20260921)
    ops = {}
    for shape in ((32, 32), (24, 40)):
        tag = "%dx%d" % shape
        meta, outs, ins = [], [], []
        for kind in (0, 1, 2):
            img = synth(shape, kind, rng)
            ins.append(img)
            for name in ALL_OPS:
                for li, lvl in enumerate(LEVELS):
                    seed = 1000 + li          # alternates the mirror draw across levels
                    random.seed(seed)
                    np.random.seed(seed)
                    out = np.asarray(aug.apply_augment(PIL.Image.fromarray(img), name, lvl))
                    meta.append(json.dumps([name, lvl, seed, kind]))
                    outs.append(out)
        ops["in_" + tag] = np.stack(ins)
        ops["out_" + tag] = np.stack(outs)
        ops["meta_" + tag] = np.array(meta)
    np.savez_compressed(os.path.join(HERE, "golden_ops.npz"), **ops)

    # ---- (3) policy-level: chained digests over seeds 0..63 (SURVEY 8c) + arrays
    chained = {}
    for pol in ("fa_reduced_cifar10", "fa_resnet50_rimagenet"):
        policies = getattr(archive, pol)()
        A = data.Augmentation(policies)
        for s in (32, 224):
            img = np.random.default_rng(1234).integers(0, 256, (s, s, 3), dtype=np.uint8)
            hsh = hashlib.sha256()
            for seed in range(64):
                random.seed(seed)
                np.random.seed(seed)
                hsh.update(np.asarray(A(PIL.Image.fromarray(img))).tobytes())
            chained["%s_%d" % (pol, s)] = hsh.hexdigest()
    hashes["chained_seeds_0_63"] = chained

    # ---- (4) policy outputs on mixed inputs, batch-sequential RNG (num_workers=0 order)
    # (the inputs are regenerated by the tests from their seeds, helpers.make_chain_inputs, and pinned by digest)
    chain = {}
    inputs = make_chain_inputs()
    hashes["chain_inputs"] = {k: sha(a) for k, a in inputs.items()}
    for pol, shape, n in GOLDEN_POLICY_BATCHES:
        policies = getattr(archive, pol)()
        batch = inputs["policy_%s_in" % pol]
        A = data.Augmentation(policies)
        random.seed(5)
        np.random.seed(5)
        torch.manual_seed(5)
        out = np.stack([np.asarray(A(PIL.Image.fromarray(a))) for a in batch])
        chain["policy_%s_out" % pol] = out

    # ---- (5) the exact CIFAR transform_train (data.py:39-44 + :92 + :112), fp32
    from torchvision.transforms import transforms as T
    policies = archive.fa_reduced_cifar10()
    tt = T.Compose([T.RandomCrop(32, padding=4), T.RandomHorizontalFlip(), T.ToTensor(),
                    T.Normalize(data._CIFAR_MEAN, data._CIFAR_STD)])
    tt.transforms.insert(0, data.Augmentation(policies))
    tt.transforms.append(data.CutoutDefault(16))
    batch = inputs["cifar_chain_in"]
    random.seed(11)
    np.random.seed(11)
    torch.manual_seed(11)
    out = torch.stack([tt(PIL.Image.fromarray(a)) for a in batch]).numpy()
    chain["cifar_chain_out_f32"] = out
    hashes["cifar_chain_sha"] = sha(out)

    # ---- (6) mixup (aug_mixup.py:13-23)
    torch.manual_seed(3)
    np.random.seed(3)
    x = torch.from_numpy(out[:16].copy())
    y = torch.arange(16)
    mixed, t1, t2, lam = aug_mixup.mixup(x, y, 0.2)      # (its input is cifar_chain_out_f32[:16])
    hashes["mixup_out"] = sha(mixed.numpy())
    chain["mixup_t2"] = t2.numpy()
    chain["mixup_lam"] = np.array([lam], dtype=np.float64)

    # ---- (7) whole policies on fresh inputs, image by image (the reference's Augmentation loop, data.py:257-264);
    #      16-hex-digit digests keep the fixture small, a mismatch still names the image
    live = {"policies": {}, "outputs": {}}
    rng = np.random.default_rng(5)
    for pol, s, n in LIVE_POLICY_RUNS:
        ref_pol = getattr(archive, pol)()
        live["policies"][pol] = sha_policy(ref_pol)
        digests = []
        for i in range(n):
            img = live_input(rng, s, i)
            random.seed(i)
            np.random.seed(i)
            policy = random.choice(ref_pol)
            im = PIL.Image.fromarray(img)
            for name, pr, level in policy:
                if random.random() > pr:
                    continue
                im = aug.apply_augment(im, name, level)
            digests.append(sha(np.asarray(im))[:16])
        live["outputs"]["%s_%d" % (pol, s)] = digests
    hashes["live_reference"] = live

    # ---- (8) ToTensor -> Lighting(0.1, PCA) -> Normalize of the ImageNet train chain (data.py:70-72), fp32, per image
    lighting = T.Compose([T.ToTensor(), aug.Lighting(0.1, data._IMAGENET_PCA["eigval"], data._IMAGENET_PCA["eigvec"]),
                          T.Normalize(mean=[0.485, 0.456, 0.406], std=[0.229, 0.224, 0.225])])
    batch = synth_batch(40, (64, 72), seed=4)
    torch.manual_seed(5)
    hashes["lighting_chain"] = [sha(lighting(PIL.Image.fromarray(a)).numpy())[:16] for a in batch]

    np.savez_compressed(os.path.join(HERE, "golden_chain.npz"), **chain)
    with open(os.path.join(HERE, "golden_hashes.json"), "w") as f:
        json.dump(hashes, f, indent=1, sort_keys=True)
    print("wrote golden fixtures:", {k: os.path.getsize(os.path.join(HERE, k))
                                     for k in os.listdir(HERE) if k.startswith("golden_")})


if __name__ == "__main__":
    main()
