"""GPU parity of the lean octet paths (csrc/faa_fast.cuh, the 8-pixel streaming loops) against the oracle.

These paths only run for the common launch geometry (W % 8 == 0, float output of the image's own size, no
crop) and, for the gathers / Color / Cutout, only in the light streaming kernel - so every case here is run
twice: forced through the two-kernel split (FAA_SPLIT_MIN=0) and forced through the cluster kernel alone
(FAA_SPLIT_MIN huge).  Each image of a launch gets its own sub-policy, odd images are mirrored.
fp32 output must be bit-exact (exact ToTensor+Normalize table of the oracle's uint8 result); fp16 / bf16 must
equal that fp32 value rounded once.
"""
import hashlib
import json
import os
import random

import numpy as np
import PIL.Image
import pytest
import torch

from helpers import ALL_OPS, GOLDEN, TABLE_STATS, exact_norm_table, fma_shortcut_rounds_like_the_table, seed_all, synth_batch

from fast_autoaugment_b200 import _lib
from fast_autoaugment_b200.engine import IMAGENET_MEAN, IMAGENET_STD, CIFAR_MEAN, CIFAR_STD, CompiledPolicy, TailSpec, augment_batch
from oracle import pil_path

pytestmark = pytest.mark.gpu
_SAMPLE, _BOX = _lib.SAMPLE_DTYPE, _lib.BOX_DTYPE

GEO = ["ShearX", "ShearY", "TranslateX", "TranslateY", "Rotate", "TranslateXAbs", "TranslateYAbs"]
LUTS = ["Invert", "Solarize", "Posterize", "Brightness", "Posterize2"]


def _policies():
    rng = random.Random(11)
    levels = (0.0, 0.07, 0.31, 0.5, 0.75, 0.93, 1.0)
    pols = [[(name, 1.0, lv), (name, 0.0, lv)] for name in ALL_OPS for lv in levels]          # single ops
    pols += [[(name, 0.0, lv), (name, 1.0, lv)] for name in ALL_OPS for lv in (0.2, 0.8)]     # ... in slot 1
    # the fp32 blends over a sweep of alphas (rounding of alpha * (px - deg) decides bytes: a fused multiply-add is wrong
    # for some alphas, e.g. level 0.9 -> alpha 1.72)
    pols += [[(name, 1.0, k / 40.0), (name, 0.0, 0.5)] for name in ("Sharpness", "Color", "Brightness", "Contrast") for k in range(41)]
    pols += [[("Sharpness", 1.0, 0.9), (b, 1.0, 0.37)] for b in ALL_OPS] + [[(a, 1.0, 0.37), ("Sharpness", 1.0, 0.9)] for a in ALL_OPS]
    for g in GEO:                                                                              # gather + LUT partner, both orders
        for l in LUTS:
            pols.append([(g, 1.0, rng.random()), (l, 1.0, rng.random())])
            pols.append([(l, 1.0, rng.random()), (g, 1.0, rng.random())])
    for a in ("Color", "Cutout", "CutoutAbs"):                                                 # partners the lean paths do NOT take
        for g in ("ShearX", "Rotate", "TranslateY"):
            pols.append([(a, 1.0, rng.random()), (g, 1.0, rng.random())])
            pols.append([(g, 1.0, rng.random()), (a, 1.0, rng.random())])
    pols += [[(a, 1.0, rng.random()), (b, 1.0, rng.random())] for a in ALL_OPS for b in ALL_OPS]   # every ordered pair
    pols += [[("Color", 1.0, rng.random()), (l, 1.0, rng.random())] for l in LUTS]
    pols += [[("Cutout", 1.0, rng.random()), ("Color", 1.0, rng.random())], [("Color", 1.0, 0.3), ("Color", 1.0, 0.9)],
             [("Invert", 1.0, 0.3), ("Solarize", 1.0, 0.4)], [("AutoContrast", 1.0, 0.3), ("ShearX", 1.0, 0.9)],
             [("TranslateX", 1.0, 0.9), ("Equalize", 1.0, 0.9)], [("Sharpness", 1.0, 0.9), ("TranslateY", 1.0, 0.1)]]
    return pols


@pytest.mark.parametrize("split_min", ["0", "1000000000000"])
@pytest.mark.parametrize("shape,norm", [((48, 64), "imagenet"), ((224, 224), "imagenet"), ((56, 104), "cifar"), ((380, 376), "imagenet"),
                                        ((224, 224), "float16"), ((56, 104), "bfloat16")])
def test_octet_paths_match_oracle(shape, norm, split_min, monkeypatch):
    """norm "float16" / "bfloat16": Normalize stats for which the fma shortcut does not round like the exact table in that
    dtype, so its launches run the TAB=true light / mid (split) or cluster kernels"""
    monkeypatch.setenv("FAA_SPLIT_MIN", split_min)
    H, W = shape
    policies = _policies()
    n = len(policies)
    pol = CompiledPolicy(policies)
    batch = synth_batch(n, shape, seed=H * 3 + W)
    mean, std = {"imagenet": (IMAGENET_MEAN, IMAGENET_STD), "cifar": (CIFAR_MEAN, CIFAR_STD)}.get(norm) or TABLE_STATS[norm]
    if norm in TABLE_STATS:
        assert not fma_shortcut_rounds_like_the_table(mean, std, getattr(torch, norm))
    seed_all(4)
    want_u8 = np.stack([np.asarray(pil_path.PolicyTransform([policies[i]])(PIL.Image.fromarray(a)))
                        for i, a in enumerate(batch)])
    seed_all(4)
    ss, bb = [], []
    for i in range(n):
        s, b = CompiledPolicy([policies[i]]).sample_parity(1, H, W)
        s["sub"] = i
        s["flip"] = i & 1
        ss.append(s)
        bb.append(b)
    samples, boxes = np.concatenate(ss), np.concatenate(bb)
    for i in range(1, n, 2):
        want_u8[i] = want_u8[i][:, ::-1]
    tab = torch.from_numpy(exact_norm_table(mean, std))
    xc = torch.from_numpy(np.ascontiguousarray(want_u8)).permute(0, 3, 1, 2).long()
    want = torch.stack([tab[c][xc[:, c]] for c in range(3)], 1)
    x = torch.from_numpy(batch).cuda()
    for dt in (torch.float32, torch.float16, torch.bfloat16):
        tail = TailSpec(None, 0, True, mean, std, 0, dt)
        got = augment_batch(pol, x, tail, samples, boxes).cpu()
        bad = [(i, policies[i]) for i in range(n) if not torch.equal(got[i], want[i].to(dt))]
        assert not bad, (shape, dt, split_min, len(bad), bad[:6])
    # uint8 HWC output (the Mixup exchange format) through the same lean paths: the augmented bytes themselves
    got = augment_batch(pol, x, TailSpec(None, 0, True, mean, std, 0, torch.uint8), samples, boxes).cpu().numpy()
    bad = [(i, policies[i]) for i in range(n) if not np.array_equal(got[i], want_u8[i])]
    assert not bad, (shape, "uint8", split_min, len(bad), bad[:6])
    # CutoutDefault post-pass on top of the octet paths
    tail = TailSpec(None, 0, True, mean, std, 16, torch.float32)
    for i in range(n):
        samples[i]["zero_box"] = (max(0, i % H - 8), min(H, i % H + 8), max(0, (3 * i) % W - 8), min(W, (3 * i) % W + 8))
    got = augment_batch(pol, x, tail, samples, boxes).cpu()
    for i in range(n):
        zb = samples[i]["zero_box"]
        w = want[i].clone()
        w[:, zb[0]:zb[1], zb[2]:zb[3]] = 0
        assert torch.equal(got[i], w), (i, policies[i])


@pytest.mark.parametrize("B,shape,replicas,dtype,cutout,split_min", [(64, (32, 32), 5, torch.float32, 16, "1000000000000"),
                                                                     (96, (224, 224), 3, torch.float16, 0, "0"),
                                                                     (40, (56, 104), 4, torch.uint8, 0, "1000000000000")])
def test_tta_replicas_equal_single_launches(B, shape, replicas, dtype, cutout, split_min, monkeypatch):
    """search.py:87-125 batching (row N4): ONE launch evaluates `num_policy` replicas of a validation batch; replica r must
    equal the plain launch that draws the decisions of samples first_index + r*B + i (both schedules: cluster kernel
    alone and the split kernels)"""
    from fast_autoaugment_b200 import archive
    from fast_autoaugment_b200.engine import augment_tta, make_rng
    monkeypatch.setenv("FAA_SPLIT_MIN", split_min)
    H, W = shape
    pol = CompiledPolicy(archive.fa_reduced_cifar10() if H == 32 else archive.fa_resnet50_rimagenet())
    tail = TailSpec.cifar(cutout, dtype) if H == 32 else (TailSpec.raw_u8() if dtype == torch.uint8 else TailSpec.imagenet(cutout, dtype))
    x = torch.from_numpy(synth_batch(B, shape, seed=31)).cuda()
    got = augment_tta(pol, x, tail, replicas, seed=9, first_index=1000)
    assert got.shape[0] == replicas and got.shape[1] == B
    ref_pol = CompiledPolicy(pol.policies)
    for r in range(replicas):
        want = augment_batch(ref_pol, x, tail, rng=make_rng(9, 1000 + r * B, tail))
        assert torch.equal(got[r], want), r
    assert not torch.equal(got[0], got[1])


@pytest.mark.parametrize("shape,kind,dtype", [((32, 32), "cifar", torch.float32), ((224, 224), "imagenet", torch.float16),
                                              ((56, 104), "imagenet_cutout", torch.float32)])
def test_mixup_of_augmented_u8_equals_the_fused_launch(shape, kind, dtype):
    """BASELINE config 4 route (augment once to uint8, exchange, faa_mix_u8) == the fused two-source launch == the
    reference formula data*lam + data[perm]*(1-lam) on the normalised fp32 tensors (aug_mixup.py:21)"""
    from fast_autoaugment_b200 import archive
    from fast_autoaugment_b200.distributed import global_pairing, mixup_global
    from fast_autoaugment_b200.engine import make_rng
    H, W = shape
    n = 96
    pol = CompiledPolicy(archive.fa_reduced_cifar10() if kind == "cifar" else archive.fa_resnet50_rimagenet())
    tail = TailSpec.cifar(16, dtype) if kind == "cifar" else TailSpec.imagenet(16 if kind.endswith("cutout") else 0, dtype)
    x = torch.from_numpy(synth_batch(n, shape, seed=12)).cuda()
    y = torch.arange(n).cuda()
    data, t1, t2, lam = mixup_global(pol, x, y, tail, 0.2, seed=3, step=2)
    perm, lam2 = global_pairing(n, 0.2, seed=3, step=2)
    assert lam == lam2 and torch.equal(t2.cpu(), perm) and torch.equal(t1, y)
    fused = augment_batch(CompiledPolicy(pol.policies), x, tail, rng=make_rng(3, 2 * n, tail), partner=perm, lam=lam)
    assert torch.equal(data, fused)
    if dtype == torch.float32:
        plain = augment_batch(CompiledPolicy(pol.policies), x, tail, rng=make_rng(3, 2 * n, tail))
        ref = plain * np.float32(lam) + plain[perm.cuda()] * np.float32(1 - lam)
        assert torch.equal(data, ref)


def test_color_jitter_matches_torchvision():
    """row N2: ColorJitter(0.4, 0.4, 0.4) of the ImageNet train chain (reference data.py:65-69) - torchvision on PIL
    images under the same torch seed is the oracle; bit-exact uint8"""
    from torchvision import transforms
    from fast_autoaugment_b200.data import ColorJitter
    for shape in ((32, 32), (56, 104), (224, 224)):
        n = 24
        batch = synth_batch(n, shape, seed=shape[0])
        tv = transforms.ColorJitter(brightness=0.4, contrast=0.4, saturation=0.4)
        torch.manual_seed(17)
        want = np.stack([np.asarray(tv(PIL.Image.fromarray(a))) for a in batch])
        torch.manual_seed(17)
        cj = ColorJitter(0.4, 0.4, 0.4)
        recs = cj.sample_parity(n)
        x = torch.from_numpy(batch).cuda()
        got = cj.jitter_batch(x, recs).cpu().numpy()
        bad = [i for i in range(n) if not np.array_equal(got[i], want[i])]
        assert not bad, (shape, bad, recs[bad[:3]])
        inplace = x.clone()
        cj.jitter_batch(inplace, recs, out=inplace)
        assert torch.equal(inplace.cpu(), torch.from_numpy(want))


def test_lighting_folded_into_the_normalisation_matches_the_reference_chain():
    """row N2: ToTensor -> Lighting(0.1, PCA) -> Normalize (reference data.py:70-72, augmentations.py:197-215) as
    per-image normalisation tables; the oracle is the reference's own chain, recorded image by image by
    tests/golden/make_golden.py (torch.manual_seed(5), the same inputs)"""
    from fast_autoaugment_b200.data import Lighting
    with open(os.path.join(GOLDEN, "golden_hashes.json")) as f:
        want = json.load(f)["lighting_chain"]
    n, shape = 40, (64, 72)
    batch = synth_batch(n, shape, seed=4)
    assert len(want) == n
    torch.manual_seed(5)
    rgb = Lighting(0.1).sample_rgb(n)
    pol = CompiledPolicy([[("Invert", 0.0, 0.0), ("Invert", 0.0, 0.0)]])
    z = np.zeros(n, dtype=_SAMPLE)
    zb = np.zeros((n, 2), dtype=_BOX)
    x = torch.from_numpy(batch).cuda()
    for split in ("0", "1000000000000"):
        os.environ["FAA_SPLIT_MIN"] = split
        got = augment_batch(pol, x, TailSpec(None, 0, False, IMAGENET_MEAN, IMAGENET_STD, 0, torch.float32), z, zb, lighting_rgb=rgb).cpu()
        bad = [i for i in range(n) if hashlib.sha256(got[i].numpy().tobytes()).hexdigest()[:16] != want[i]]
        assert got.dtype == torch.float32 and got.shape == (n, 3) + shape and not bad, (split, bad)
        for dt in (torch.float16, torch.bfloat16):          # the per-image tables, then ONE rounding at the store
            half = augment_batch(pol, x, TailSpec(None, 0, False, IMAGENET_MEAN, IMAGENET_STD, 0, dt), z, zb, lighting_rgb=rgb).cpu()
            assert half.dtype == dt and torch.equal(half, got.to(dt)), (split, dt)
    os.environ.pop("FAA_SPLIT_MIN", None)
    # with a policy in front and a flip behind it: equals the un-lit launch re-normalised image by image
    pol2 = CompiledPolicy([[("Rotate", 1.0, 0.3), ("Color", 1.0, 0.6)], [("AutoContrast", 1.0, 0.3), ("Sharpness", 1.0, 0.8)]])
    seed_all(2)
    s2, b2 = pol2.sample_parity(n, *shape, TailSpec.imagenet(0, torch.float32))
    u8 = augment_batch(pol2, x, TailSpec(None, 0, True, IMAGENET_MEAN, IMAGENET_STD, 0, torch.uint8), s2, b2).cpu()
    lit = augment_batch(pol2, x, TailSpec.imagenet(0, torch.float32), s2, b2, lighting_rgb=rgb).cpu()
    m, sd = torch.tensor(IMAGENET_MEAN).view(3, 1, 1), torch.tensor(IMAGENET_STD).view(3, 1, 1)
    for i in range(n):
        t = u8[i].permute(2, 0, 1).float().div(255)
        t = t.add(rgb[i].view(3, 1, 1).expand_as(t))
        assert torch.equal(lit[i], (t - m) / sd), i
    for dt in (torch.float16, torch.bfloat16):
        half = augment_batch(pol2, x, TailSpec.imagenet(0, dt), s2, b2, lighting_rgb=rgb).cpu()
        bad = [i for i in range(n) if not torch.equal(half[i], lit[i].to(dt))]
        assert not bad, (dt, bad)


@pytest.mark.gpu
@pytest.mark.parametrize("shape,pol_name", [((32, 32), "fa_reduced_cifar10"), ((224, 224), "fa_resnet50_rimagenet")])
def test_run_many_and_self_resolving_launches_equal_single_calls(shape, pol_name):
    """faa_augment_many == a loop of faa_augment; launches too small to split resolve inside the pixel kernel and must
    equal launches driven by the device sampler's records (the resolve-kernel route) bit for bit"""
    from fast_autoaugment_b200 import archive
    from fast_autoaugment_b200.distributed import philox_records
    from fast_autoaugment_b200.engine import FusedAugmenter
    H, W = shape
    B = 96
    pol = CompiledPolicy(getattr(archive, pol_name)())
    tail = TailSpec.cifar(16, torch.float16) if H == 32 else TailSpec.imagenet(0, torch.float16)
    xs = [torch.from_numpy(synth_batch(B, shape, seed=10 + i)).cuda() for i in range(5)]
    f = FusedAugmenter(pol, tail, H, W, 77)
    outs = [f.empty_out(B) for _ in range(5)]
    plan = f.plan_many(xs, outs)
    f.run_many(plan, 1000, stride=B)
    torch.cuda.synchronize()
    many = [o.clone() for o in outs]
    single = [f(xs[k], f.empty_out(B), 1000 + k * B).clone() for k in range(5)]
    torch.cuda.synchronize()
    for a, b in zip(many, single):
        assert torch.equal(a, b)
    for k in range(5):
        d_s, d_b = philox_records(pol, B, H, W, tail, 77, 1000 + k * B, "cuda")
        samples = d_s.cpu().numpy().reshape(-1).view(_lib.SAMPLE_DTYPE)
        boxes = d_b.cpu().numpy().reshape(-1).view(_lib.BOX_DTYPE).reshape(B, pol.n_op)
        assert torch.equal(many[k], augment_batch(pol, xs[k], tail, samples, boxes))
