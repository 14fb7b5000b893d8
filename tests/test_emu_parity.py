"""Kernel arithmetic (faa_core.cuh, compiled for the host by tests/emu) vs the oracle.

These tests execute, on the CPU, the same per-pixel source the sm_100a kernels execute -
policy compilation comes from the real C-ABI library (host functions, no GPU needed), the
pixel evaluation from tests/emu - and demand bit-exact agreement with the oracle
(oracle.pil_path = the reference's calls into Pillow) on every op, policy and chain.
"""
import json
import random

import numpy as np
import PIL.Image
import pytest
import torch

from helpers import ALL_OPS, emu_augment, exact_norm_table, golden_chain, seed_all, synth_batch

from fast_autoaugment_b200 import archive
from fast_autoaugment_b200.engine import CIFAR_MEAN, CIFAR_STD, IMAGENET_MEAN, IMAGENET_STD, CompiledPolicy, TailSpec
from oracle import np_model, pil_path


def _policy_oracle(policies, batch):
    """oracle: PolicyTransform image by image (consumes the global RNGs)."""
    t = pil_path.PolicyTransform(policies)
    return np.stack([np.asarray(t(PIL.Image.fromarray(a))) for a in batch])


@pytest.mark.parametrize("name", ALL_OPS)
@pytest.mark.parametrize("shape", [(32, 32), (24, 40), (5, 3), (1, 7), (33, 31)])
def test_single_op_all_levels(emu, name, shape):
    """each of the 19 ops, 9 levels, both mirror signs / several boxes, 3 input families,
    incl. non-square, odd and degenerate sizes; generic and aligned-fast kernel paths"""
    batch = synth_batch(6, shape, seed=hash(name) % 1000 + shape[0])
    for level in (0.0, 0.05, 0.13, 0.31, 0.5, 0.62, 0.7, 0.93, 1.0):
        policies = [[(name, 1.0, level)]]
        pol = CompiledPolicy(policies)
        for seed in (1, 2):
            seed_all(seed)
            want = _policy_oracle(policies, batch)
            seed_all(seed)
            samples, boxes = pol.sample_parity(len(batch), shape[0], shape[1])
            for generic in (False, True):
                got = emu_augment(emu, pol, batch, samples, boxes, force_generic=generic)
                assert np.array_equal(got, want), (name, shape, level, seed, generic)


@pytest.mark.parametrize("pol_name,shape,n", [
    ("fa_reduced_cifar10", (32, 32), 600), ("fa_reduced_svhn", (32, 32), 300),
    ("fa_resnet50_rimagenet", (56, 56), 200), ("fa_resnet50_rimagenet", (224, 224), 24),
    ("arsaug_policy", (24, 40), 200), ("autoaug_policy", (32, 32), 400),
    ("autoaug_paper_cifar10", (32, 32), 300), ("fa_reduced_cifar10", (95, 95), 40)])
def test_archive_policies_match_oracle(emu, pol_name, shape, n):
    policies = getattr(archive, pol_name)()
    pol = CompiledPolicy(policies)
    batch = synth_batch(n, shape, seed=len(pol_name) + shape[0])
    seed_all(123)
    want = _policy_oracle(policies, batch)
    seed_all(123)
    samples, boxes = pol.sample_parity(n, shape[0], shape[1])
    got = emu_augment(emu, pol, batch, samples, boxes)
    bad = [i for i in range(n) if not np.array_equal(got[i], want[i])]
    assert not bad, (pol_name, bad[:5], [policies[samples[i]["sub"]] for i in bad[:5]])
    got2 = emu_augment(emu, pol, batch, samples, boxes, force_generic=True)
    assert np.array_equal(got2, want)


def test_all_op_pairs(emu):
    """every ordered pair of the 19 ops as a 2-op sub-policy with both gates open: covers
    stats-after-geometry, Sharpness-after-Sharpness, Contrast-after-Equalize ..."""
    rng = random.Random(7)
    policies = [[(a, 1.0, rng.random()), (b, 1.0, rng.random())] for a in ALL_OPS for b in ALL_OPS]
    pol = CompiledPolicy(policies)
    shape = (20, 24)
    batch = synth_batch(len(policies), shape, seed=5)
    # force sub-policy i onto image i (the sampler's other draws still come from the RNGs)
    seed_all(9)
    want = []
    for i, a in enumerate(batch):          # a one-sub-policy Augmentation per image
        want.append(np.asarray(pil_path.PolicyTransform([policies[i]])(PIL.Image.fromarray(a))))
    want = np.stack(want)
    seed_all(9)
    samples_all, boxes_all = [], []
    for i in range(len(policies)):
        sub_pol = CompiledPolicy([policies[i]])
        s, b = sub_pol.sample_parity(1, shape[0], shape[1])
        s["sub"] = i
        samples_all.append(s)
        boxes_all.append(b)
    samples = np.concatenate(samples_all)
    boxes = np.concatenate(boxes_all)
    got = emu_augment(emu, pol, batch, samples, boxes)
    bad = [policies[i] for i in range(len(policies)) if not np.array_equal(got[i], want[i])]
    assert not bad, bad[:8]


def test_cifar_chain_fp32_matches_golden_and_oracle(emu):
    """Augmentation -> RandomCrop(32,4) -> HFlip -> ToTensor -> Normalize -> CutoutDefault(16):
    the exact transform_train of reference data.py:39-44,92,112, fp32, max abs diff 0."""
    g = golden_chain()
    batch, want = g["cifar_chain_in"], g["cifar_chain_out_f32"]
    policies = archive.fa_reduced_cifar10()
    pol = CompiledPolicy(policies)
    tail = TailSpec.cifar(cutout=16, out_dtype=torch.float32)
    seed_all(11)
    samples, boxes = pol.sample_parity(len(batch), 32, 32, tail)
    got = emu_augment(emu, pol, batch, samples, boxes, tail, exact_norm_table(CIFAR_MEAN, CIFAR_STD))
    assert np.array_equal(got, want)          # -0.0 == 0.0 inside the zero box
    # and against the oracle chain on fresh data
    batch2 = synth_batch(200, (32, 32), seed=31)
    seed_all(4)
    want2 = pil_path.run_chain_on_batch(pil_path.cifar_train_chain(policies, 16), batch2).numpy()
    seed_all(4)
    samples, boxes = pol.sample_parity(len(batch2), 32, 32, tail)
    got2 = emu_augment(emu, pol, batch2, samples, boxes, tail, exact_norm_table(CIFAR_MEAN, CIFAR_STD))
    assert np.array_equal(got2, want2)


def test_fixed_shape_chain_with_flip_and_cutout(emu):
    policies = archive.fa_resnet50_rimagenet()
    pol = CompiledPolicy(policies)
    batch = synth_batch(48, (64, 64), seed=8)
    tail = TailSpec(None, 0, True, IMAGENET_MEAN, IMAGENET_STD, 16, torch.float32)
    seed_all(21)
    want = pil_path.run_chain_on_batch(pil_path.fixed_shape_chain(policies, IMAGENET_MEAN, IMAGENET_STD, True, 16),
                                       batch).numpy()
    seed_all(21)
    samples, boxes = pol.sample_parity(len(batch), 64, 64, tail)
    for generic in (False, True):
        got = emu_augment(emu, pol, batch, samples, boxes, tail, exact_norm_table(IMAGENET_MEAN, IMAGENET_STD),
                          force_generic=generic)
        assert np.array_equal(got, want)


def test_three_op_policy_chained_windows(emu):
    """search.py --num-op > 2: ops beyond the fused pair run as chained launches"""
    rng = random.Random(3)
    names = ["Rotate", "Equalize", "Sharpness", "Cutout", "Color", "TranslateY", "AutoContrast", "Contrast"]
    policies = [[(rng.choice(names), rng.random(), rng.random()) for _ in range(3)] for _ in range(40)]
    policies += [[(rng.choice(ALL_OPS), 1.0, rng.random()) for _ in range(3)] for _ in range(40)]
    pol = CompiledPolicy(policies)
    batch = synth_batch(160, (32, 32), seed=77)
    seed_all(2)
    want = _policy_oracle(policies, batch)
    seed_all(2)
    samples, boxes = pol.sample_parity(len(batch), 32, 32)
    got = emu_augment(emu, pol, batch, samples, boxes)
    assert np.array_equal(got, want)


def test_fused_mixup_matches_reference_formula(emu):
    """out = aug(x_i)*lam + aug(x_perm[i])*(1-lam) in fp32 (aug_mixup.py:21) == augment, then mix"""
    policies = archive.fa_reduced_cifar10()
    pol = CompiledPolicy(policies)
    tail = TailSpec.cifar(cutout=16, out_dtype=torch.float32)
    batch = synth_batch(32, (32, 32), seed=12)
    norm = exact_norm_table(CIFAR_MEAN, CIFAR_STD)
    seed_all(6)
    samples, boxes = pol.sample_parity(len(batch), 32, 32, tail)
    plain = emu_augment(emu, pol, batch, samples, boxes, tail, norm)
    seed_all(6)
    want_plain = pil_path.run_chain_on_batch(pil_path.cifar_train_chain(policies, 16), batch)
    assert np.array_equal(plain, want_plain.numpy())
    want, _, _, lam = pil_path.mixup_pairs(want_plain, torch.arange(len(batch)), 0.2)
    seed_all(6)
    pil_path.run_chain_on_batch(pil_path.cifar_train_chain(policies, 16), batch)   # advance RNGs identically
    perm = torch.randperm(len(batch))
    lam2 = np.random.beta(0.2, 0.2)
    lam2 = max(lam2, 1.0 - lam2)
    assert lam2 == lam
    got = emu_augment(emu, pol, batch, samples, boxes, tail, norm, partner=perm.numpy(), lam=lam)
    assert np.array_equal(got, want.numpy())


def test_translate_accumulator_break(emu):
    """TranslateX/Y at level 0.75 on 380 px: v*W = 85.50000000000001, Pillow's accumulated
    offset snaps to the next integer part-way through the row -> two different shifts"""
    policies = [[("TranslateX", 1.0, 0.75)], [("TranslateY", 1.0, 0.75)], [("TranslateX", 1.0, 0.25)]]
    pol = CompiledPolicy(policies)
    recs = [pol.compiled_op(380, 380, s, 0, sg) for s in range(3) for sg in (0, 1)]
    assert any(r[0] == 2 and (r[3] < 380 or r[4] < 380) for r in recs)       # a break index is present
    batch = synth_batch(24, (380, 380), seed=1)
    seed_all(3)
    want = _policy_oracle(policies, batch)
    seed_all(3)
    samples, boxes = pol.sample_parity(len(batch), 380, 380)
    assert np.array_equal(emu_augment(emu, pol, batch, samples, boxes), want)


@pytest.mark.parametrize("shape,n,pol_name,cutout", [((224, 224), 512, "fa_resnet50_rimagenet", 0),
                                                      ((380, 380), 256, "fa_resnet50_rimagenet", 16),
                                                      ((32, 32), 512, "fa_reduced_cifar10", 16)])
def test_full_size_configs_every_image_against_the_oracle(emu, shape, n, pol_name, cutout):
    """BASELINE.json configs 2, 3, 5 at FULL size, every image: kernel arithmetic (host build) == the reference's PIL /
    torchvision chain in fp32.  tests/test_gpu_parity.py::test_full_size_configs demands GPU == this host build for every
    image of the same batches, samples and seeds - together: the GPU equals the oracle on the whole batch, not on a sample."""
    H, W = shape
    policies = getattr(archive, pol_name)()
    pol = CompiledPolicy(policies)
    mean, std = (CIFAR_MEAN, CIFAR_STD) if H == 32 else (IMAGENET_MEAN, IMAGENET_STD)
    tail = TailSpec((32, 32), 4, True, mean, std, cutout, torch.float32) if H == 32 else \
        TailSpec(None, 0, True, mean, std, cutout, torch.float32)
    batch = synth_batch(n, shape, seed=H)                      # (the GPU test's batch, seed and sampler call)
    seed_all(77)
    samples, boxes = pol.sample_parity(n, H, W, tail)
    got = emu_augment(emu, pol, batch, samples, boxes, tail, exact_norm_table(mean, std))
    seed_all(77)
    chain = pil_path.cifar_train_chain(policies, cutout) if H == 32 else \
        pil_path.fixed_shape_chain(policies, mean, std, True, cutout)
    want = pil_path.run_chain_on_batch(chain, batch).numpy()
    bad = [i for i in range(n) if not np.array_equal(got[i], want[i])]
    assert not bad, (shape, len(bad), bad[:5], [policies[samples[i]["sub"]] for i in bad[:5]])
