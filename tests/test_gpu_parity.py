"""GPU parity tests: the sm_100a kernels, called through the C ABI, against the oracle.

Bit-exact for every uint8 result and for the fp32 chain; fp16/bf16 outputs must equal the
fp32 oracle rounded to that dtype.  Full-size cases (BASELINE.json configs) are checked
through the host emulation of the same source, through size-independent properties, and
against the oracle on a sample of the batch.
"""
import random

import numpy as np
import PIL.Image
import pytest
import torch

from helpers import ALL_OPS, emu_augment, exact_norm_table, golden_chain, seed_all, synth_batch

from fast_autoaugment_b200 import _lib, archive
from fast_autoaugment_b200.engine import (CIFAR_MEAN, CIFAR_STD, IMAGENET_MEAN, IMAGENET_STD, CompiledPolicy,
                                          TailSpec, augment_batch, make_rng)
from oracle import pil_path

pytestmark = pytest.mark.gpu


def dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def oracle_policy(policies, batch):
    t = pil_path.PolicyTransform(policies)
    return np.stack([np.asarray(t(PIL.Image.fromarray(a))) for a in batch])


def test_library_reports_device():
    assert _lib.device_count() >= 1


@pytest.mark.parametrize("shape", [(32, 32), (24, 40), (5, 3), (33, 31), (64, 64)])
def test_every_op_every_level(shape):
    """19 ops x 9 levels x 2 seeds as one launch per seed: image i gets sub-policy i"""
    levels = (0.0, 0.05, 0.13, 0.31, 0.5, 0.62, 0.7, 0.93, 1.0)
    policies = [[(name, 1.0, lv)] for name in ALL_OPS for lv in levels]
    pol = CompiledPolicy(policies)
    batch = synth_batch(len(policies), shape, seed=shape[0] * 7 + shape[1])
    for seed in (1, 2):
        seed_all(seed)
        want = np.stack([np.asarray(pil_path.PolicyTransform([policies[i]])(PIL.Image.fromarray(a)))
                         for i, a in enumerate(batch)])
        seed_all(seed)
        ss, bb = [], []
        for i in range(len(policies)):
            s, b = CompiledPolicy([policies[i]]).sample_parity(1, shape[0], shape[1])
            s["sub"] = i
            ss.append(s)
            bb.append(b)
        got = augment_batch(pol, dev(batch), TailSpec.raw_u8(), np.concatenate(ss), np.concatenate(bb)).cpu().numpy()
        bad = [policies[i] for i in range(len(policies)) if not np.array_equal(got[i], want[i])]
        assert not bad, (shape, seed, bad[:6])


def test_all_op_pairs():
    rng = random.Random(7)
    policies = [[(a, 1.0, rng.random()), (b, 1.0, rng.random())] for a in ALL_OPS for b in ALL_OPS]
    pol = CompiledPolicy(policies)
    shape = (20, 24)
    batch = synth_batch(len(policies), shape, seed=5)
    seed_all(9)
    want = np.stack([np.asarray(pil_path.PolicyTransform([policies[i]])(PIL.Image.fromarray(a)))
                     for i, a in enumerate(batch)])
    seed_all(9)
    ss, bb = [], []
    for i in range(len(policies)):
        s, b = CompiledPolicy([policies[i]]).sample_parity(1, shape[0], shape[1])
        s["sub"] = i
        ss.append(s)
        bb.append(b)
    got = augment_batch(pol, dev(batch), TailSpec.raw_u8(), np.concatenate(ss), np.concatenate(bb)).cpu().numpy()
    bad = [policies[i] for i in range(len(policies)) if not np.array_equal(got[i], want[i])]
    assert not bad, bad[:8]


@pytest.mark.parametrize("pol_name,shape,n", [
    ("fa_reduced_cifar10", (32, 32), 1024), ("fa_reduced_svhn", (32, 32), 512),
    ("fa_resnet50_rimagenet", (56, 56), 256), ("fa_resnet50_rimagenet", (224, 224), 128),
    ("fa_resnet50_rimagenet", (380, 380), 32), ("arsaug_policy", (24, 40), 256),
    ("autoaug_policy", (32, 32), 512), ("autoaug_paper_cifar10", (32, 32), 512),
    ("fa_reduced_cifar10", (95, 95), 64), ("fa_reduced_cifar10", (128, 96), 64)])
def test_archive_policies(pol_name, shape, n):
    """the reference's policy archives at CIFAR / ImageNet / EfficientNet-B4 sizes (cluster
    sizes 1, 2, 4, 8), three input families incl. constant-colour histogram worst case"""
    policies = getattr(archive, pol_name)()
    pol = CompiledPolicy(policies)
    batch = synth_batch(n, shape, seed=len(pol_name) + shape[0])
    seed_all(123)
    want = oracle_policy(policies, batch)
    seed_all(123)
    samples, boxes = pol.sample_parity(n, shape[0], shape[1])
    got = augment_batch(pol, dev(batch), TailSpec.raw_u8(), samples, boxes).cpu().numpy()
    bad = [i for i in range(n) if not np.array_equal(got[i], want[i])]
    assert not bad, (pol_name, shape, bad[:5], [policies[samples[i]["sub"]] for i in bad[:5]])


def test_golden_policy_outputs():
    """committed outputs of the live reference (tests/golden/make_golden.py)"""
    g = golden_chain()
    for pol_name in ("fa_reduced_cifar10", "autoaug_policy", "fa_reduced_svhn", "arsaug_policy",
                     "fa_resnet50_rimagenet"):
        batch, want = g["policy_%s_in" % pol_name], g["policy_%s_out" % pol_name]
        pol = CompiledPolicy(getattr(archive, pol_name)())
        seed_all(5)
        samples, boxes = pol.sample_parity(len(batch), batch.shape[1], batch.shape[2])
        got = augment_batch(pol, dev(batch), TailSpec.raw_u8(), samples, boxes).cpu().numpy()
        assert np.array_equal(got, want), pol_name


def test_golden_cifar_chain_all_dtypes():
    """transform_train of reference data.py:39-44,92,112: fp32 bit-exact; fp16/bf16 equal the
    fp32 result rounded to that dtype (uint8-level parity is implied, SURVEY.md 8c-12)"""
    g = golden_chain()
    batch, want = g["cifar_chain_in"], torch.from_numpy(g["cifar_chain_out_f32"])
    pol = CompiledPolicy(archive.fa_reduced_cifar10())
    for dt in (torch.float32, torch.float16, torch.bfloat16):
        tail = TailSpec.cifar(cutout=16, out_dtype=dt)
        seed_all(11)
        samples, boxes = pol.sample_parity(len(batch), 32, 32, tail)
        got = augment_batch(pol, dev(batch), tail, samples, boxes).cpu()
        assert torch.equal(got, want.to(dt)), dt


def test_fixed_shape_chain_imagenet_norm():
    policies = archive.fa_resnet50_rimagenet()
    pol = CompiledPolicy(policies)
    batch = synth_batch(96, (64, 64), seed=8)
    for cutout in (0, 16):
        tail = TailSpec(None, 0, True, IMAGENET_MEAN, IMAGENET_STD, cutout, torch.float32)
        seed_all(21)
        want = pil_path.run_chain_on_batch(
            pil_path.fixed_shape_chain(policies, IMAGENET_MEAN, IMAGENET_STD, True, cutout), batch)
        seed_all(21)
        samples, boxes = pol.sample_parity(len(batch), 64, 64, tail)
        got = augment_batch(pol, dev(batch), tail, samples, boxes).cpu()
        assert torch.equal(got, want)
        tail16 = TailSpec(None, 0, True, IMAGENET_MEAN, IMAGENET_STD, cutout, torch.float16)
        got16 = augment_batch(pol, dev(batch), tail16, samples, boxes).cpu()
        assert torch.equal(got16, want.half())


def test_three_op_policy_chained_launches():
    rng = random.Random(3)
    policies = [[(rng.choice(ALL_OPS), rng.random(), rng.random()) for _ in range(3)] for _ in range(60)]
    policies += [[(rng.choice(ALL_OPS), 1.0, rng.random()) for _ in range(3)] for _ in range(60)]
    pol = CompiledPolicy(policies)
    batch = synth_batch(256, (32, 32), seed=77)
    seed_all(2)
    want = oracle_policy(policies, batch)
    seed_all(2)
    samples, boxes = pol.sample_parity(len(batch), 32, 32)
    got = augment_batch(pol, dev(batch), TailSpec.raw_u8(), samples, boxes).cpu().numpy()
    assert np.array_equal(got, want)


def test_mixup_fused_and_standalone():
    """aug_mixup.py:13-23: fused (recomputes the partner) and standalone kernels, fp32 exact"""
    from fast_autoaugment_b200.aug_mixup import mixup, mixup_resolved
    policies = archive.fa_reduced_cifar10()
    pol = CompiledPolicy(policies)
    tail = TailSpec.cifar(cutout=16, out_dtype=torch.float32)
    batch = synth_batch(64, (32, 32), seed=12)
    seed_all(6)
    want_plain = pil_path.run_chain_on_batch(pil_path.cifar_train_chain(policies, 16), batch)
    want, t1, t2, lam = pil_path.mixup_pairs(want_plain, torch.arange(len(batch)), 0.2)
    seed_all(6)
    samples, boxes = pol.sample_parity(len(batch), 32, 32, tail)
    plain = augment_batch(pol, dev(batch), tail, samples, boxes)
    assert torch.equal(plain.cpu(), want_plain)
    # drop-in mixup(): same draws, same tuple
    got, g1, g2, glam = mixup(plain, torch.arange(len(batch)).cuda(), 0.2)
    assert glam == lam and torch.equal(g2.cpu(), t2) and torch.equal(got.cpu(), want)
    # fused: partner recomputed inside the augmentation kernel
    seed_all(6)
    pil_path.run_chain_on_batch(pil_path.cifar_train_chain(policies, 16), batch)
    perm = torch.randperm(len(batch))
    fused = augment_batch(pol, dev(batch), tail, samples, boxes, partner=perm, lam=lam)
    assert torch.equal(fused.cpu(), want)
    # half-precision standalone mixup = fp32 math on the half inputs, rounded once
    h = plain.half()
    mh = mixup_resolved(h, perm, lam)
    ref = (h.float() * np.float32(lam) + h.float()[perm.cuda()] * np.float32(1 - lam)).half()
    assert torch.equal(mh, ref)


def test_philox_records_match_host_model_and_drive_the_same_pixels(emu):
    """device sampler == its host emulation; fused-Philox launch == launch from those records"""
    import ctypes as C
    policies = archive.fa_reduced_cifar10()
    pol = CompiledPolicy(policies)
    tail = TailSpec.cifar(cutout=16, out_dtype=torch.float16)
    B, H, W = 2048, 32, 32
    rng = make_rng(1234, 5000, tail)
    t = tail.c_struct(H, W)
    d_s = torch.zeros(B * 16, dtype=torch.uint8, device="cuda")
    d_b = torch.zeros(B * pol.n_op * 8, dtype=torch.uint8, device="cuda")
    _lib.check(_lib.lib.faa_sample_philox(pol.handle, B, H, W, C.byref(t), C.byref(rng), d_s.data_ptr(),
                                          d_b.data_ptr(), C.c_void_p(torch.cuda.current_stream().cuda_stream)))
    torch.cuda.synchronize()
    s_dev = d_s.cpu().numpy().view(_lib.SAMPLE_DTYPE)
    b_dev = d_b.cpu().numpy().view(_lib.BOX_DTYPE).reshape(B, pol.n_op)
    table = np.ascontiguousarray(pol.compiled_table(H, W))
    s_host = np.zeros(B, dtype=_lib.SAMPLE_DTYPE)
    b_host = np.zeros((B, pol.n_op), dtype=_lib.BOX_DTYPE)
    probs = np.ascontiguousarray(pol.probs)
    emu.faa_emu_philox(table.ctypes.data, probs.ctypes.data, pol.n_sub, pol.n_op, C.byref(rng), B, H, W, 32, 32,
                       s_host.ctypes.data, b_host.ctypes.data)
    assert s_dev.tobytes() == s_host.tobytes()
    assert b_dev.tobytes() == b_host.tobytes()
    batch = dev(synth_batch(B, (H, W), seed=3))
    a = augment_batch(pol, batch, tail, rng=rng)
    b = augment_batch(pol, batch, tail, s_dev, b_dev)
    assert torch.equal(a, b)
    # distribution sanity: gates fire with the policy's probabilities, flips ~ 1/2, crops uniform
    exp_gate = pol.probs[s_dev["sub"], 0].mean()
    assert abs(((s_dev["gate"] & 1) > 0).mean() - exp_gate) < 0.04
    assert abs(s_dev["flip"].mean() - 0.5) < 0.04
    assert set(np.unique(s_dev["crop_dy"])) == set(range(-4, 5))
    assert len(np.unique(s_dev["sub"])) > 400


@pytest.mark.parametrize("shape,n,pol_name,cutout", [((224, 224), 512, "fa_resnet50_rimagenet", 0),
                                                      ((380, 380), 256, "fa_resnet50_rimagenet", 16),
                                                      ((32, 32), 512, "fa_reduced_cifar10", 16)])
def test_full_size_configs(emu, shape, n, pol_name, cutout):
    """BASELINE.json configs 2, 3, 5 at full size: (a) the whole batch against the host
    emulation of the same source, (b) a sample of it against the oracle, (c) properties:
    prob-0 policy == plain normalise, determinism, shard-composability."""
    H, W = shape
    policies = getattr(archive, pol_name)()
    pol = CompiledPolicy(policies)
    mean, std = (CIFAR_MEAN, CIFAR_STD) if H == 32 else (IMAGENET_MEAN, IMAGENET_STD)
    tail = TailSpec((32, 32), 4, True, mean, std, cutout, torch.float32) if H == 32 else \
        TailSpec(None, 0, True, mean, std, cutout, torch.float32)
    batch = synth_batch(n, shape, seed=H)
    seed_all(77)
    samples, boxes = pol.sample_parity(n, H, W, tail)
    x = dev(batch)
    got = augment_batch(pol, x, tail, samples, boxes)
    # (a) emulation of the same source, every image
    want_emu = emu_augment(emu, pol, batch, samples, boxes, tail, exact_norm_table(mean, std))
    assert np.array_equal(got.cpu().numpy(), want_emu)
    # (b) oracle on the first 48 images (same RNG order => same decisions)
    k = 48
    seed_all(77)
    chain = pil_path.cifar_train_chain(policies, cutout) if H == 32 else \
        pil_path.fixed_shape_chain(policies, mean, std, True, cutout)
    want = pil_path.run_chain_on_batch(chain, batch[:k])
    assert torch.equal(got[:k].cpu(), want)
    # (c) properties
    assert torch.equal(got, augment_batch(pol, x, tail, samples, boxes))               # deterministic
    halves = torch.cat([augment_batch(pol, x[: n // 2], tail, samples[: n // 2], boxes[: n // 2]),
                        augment_batch(pol, x[n // 2:], tail, samples[n // 2:], boxes[n // 2:])])
    assert torch.equal(got, halves)                                                     # shards compose
    off = CompiledPolicy([[(o[0], 0.0, o[2]) for o in sub] for sub in policies[:8]])
    plain_tail = TailSpec(None, 0, False, mean, std, 0, torch.float32)
    z = np.zeros(n, dtype=_lib.SAMPLE_DTYPE)
    zb = np.zeros((n, 2), dtype=_lib.BOX_DTYPE)
    ident = augment_batch(off, x, plain_tail, z, zb)
    # torch's CPU ToTensor/Normalize arithmetic (true fp32 division; CUDA torch multiplies by 1/255)
    tab = torch.from_numpy(exact_norm_table(mean, std))
    xc = torch.from_numpy(batch).permute(0, 3, 1, 2).long()
    ref = torch.stack([tab[c][xc[:, c]] for c in range(3)], 1)
    assert torch.equal(ident.cpu(), ref)
    # fp16 output = fp32 result rounded once
    tail16 = TailSpec(tail.out_size, tail.crop_pad, tail.hflip, mean, std, cutout, torch.float16)
    assert torch.equal(augment_batch(pol, x, tail16, samples, boxes), got.half())


def test_host_buffer_entry_matches_device_entry():
    """faa_augment_host (pinned H2D -> kernel -> D2H pipeline) == faa_augment"""
    import ctypes as C
    pol = CompiledPolicy(archive.fa_resnet50_rimagenet())
    tail = TailSpec.imagenet(out_dtype=torch.float16)
    B, H, W = 96, 224, 224
    batch = torch.from_numpy(synth_batch(B, (H, W), seed=1))
    rng = make_rng(99, 0, tail)
    want = augment_batch(pol, batch.cuda(), tail, rng=rng).cpu()
    t = tail.c_struct(H, W)
    for pinned in (True, False):
        h_in = batch.clone().pin_memory() if pinned else batch.clone()
        h_out = torch.empty((B, 3, H, W), dtype=torch.float16)
        if pinned:
            h_out = h_out.pin_memory()
        _lib.check(_lib.lib.faa_augment_host(pol.handle, h_in.data_ptr(), h_out.data_ptr(), None, B, H, W,
                                             C.byref(t), C.byref(rng),
                                             C.c_void_p(torch.cuda.current_stream().cuda_stream)))
        torch.cuda.synchronize()
        assert torch.equal(h_out, want), pinned


def test_reference_surface_single_image():
    """Augmentation(policy)(PIL) -> PIL and apply_augment(img, name, level): drop-in surface"""
    from fast_autoaugment_b200 import Augmentation
    from fast_autoaugment_b200.augmentations import apply_augment
    policies = archive.fa_reduced_cifar10()
    img = PIL.Image.fromarray(synth_batch(1, (32, 32), seed=4)[0])
    for s in range(12):
        seed_all(s)
        want = np.asarray(pil_path.PolicyTransform(policies)(img))
        seed_all(s)
        got = np.asarray(Augmentation(policies)(img))
        assert np.array_equal(got, want)
    seed_all(3)
    want = np.asarray(pil_path.apply_op(img, "Rotate", 0.8))
    seed_all(3)
    assert np.array_equal(np.asarray(apply_augment(img, "Rotate", 0.8)), want)
    with pytest.raises(KeyError):
        apply_augment(img, "NoSuchOp", 0.5)


def test_translate_accumulator_break():
    """Pillow's accumulated float offset snaps part-way through a 380-px row (level 0.75)"""
    policies = [[("TranslateX", 1.0, 0.75)], [("TranslateY", 1.0, 0.75)], [("TranslateX", 1.0, 0.25)]]
    pol = CompiledPolicy(policies)
    batch = synth_batch(24, (380, 380), seed=1)
    seed_all(3)
    want = oracle_policy(policies, batch)
    seed_all(3)
    samples, boxes = pol.sample_parity(len(batch), 380, 380)
    got = augment_batch(pol, dev(batch), TailSpec.raw_u8(), samples, boxes).cpu().numpy()
    assert np.array_equal(got, want)


@pytest.mark.parametrize("B,H,W,cutout,dtype", [(96, 224, 224, 0, torch.float16), (32, 380, 380, 16, torch.bfloat16)])
def test_resolve_ahead_and_split_paths_are_invisible(B, H, W, cutout, dtype):
    """fused Philox launches at a size that takes the split (light + cluster kernel) path, called
    back to back so that the resolve-ahead speculation hits, with a stride change and a seed change
    in the sequence: every result must equal the one computed from the device sampler's records
    (second case: CutoutDefault boxes - the post-pass of both pixel kernels - and bf16 output)"""
    import ctypes as C
    from fast_autoaugment_b200.engine import FusedAugmenter
    policies = archive.fa_resnet50_rimagenet()
    tail = TailSpec.imagenet(cutout, dtype)
    x = dev(synth_batch(B, (H, W), seed=21))
    pol = CompiledPolicy(policies)
    f = FusedAugmenter(pol, tail, H, W, seed=5)
    t = tail.c_struct(H, W)
    firsts = [0, B, 2 * B, 3 * B, 10 * B, 17 * B, 24 * B, 24 * B, 7]          # hits, stride change, repeat, odd
    outs = []
    for fi in firsts:
        outs.append(f(x, f.empty_out(B), fi).clone())
    f.rng.seed = 6
    outs.append(f(x, f.empty_out(B), 8 * B).clone())
    firsts.append(8 * B)
    torch.cuda.synchronize()
    ref_pol = CompiledPolicy(policies)                                           # fresh handle: no speculation state
    for k, fi in enumerate(firsts):
        rng = make_rng(6 if k == len(firsts) - 1 else 5, fi, tail)
        d_s = torch.zeros(B * 16, dtype=torch.uint8, device="cuda")
        d_b = torch.zeros(B * 2 * 8, dtype=torch.uint8, device="cuda")
        _lib.check(_lib.lib.faa_sample_philox(ref_pol.handle, B, H, W, C.byref(t), C.byref(rng), d_s.data_ptr(),
                                              d_b.data_ptr(), C.c_void_p(torch.cuda.current_stream().cuda_stream)))
        want = augment_batch(ref_pol, x, tail, d_s, d_b)
        assert torch.equal(outs[k], want), (k, fi)


@pytest.mark.parametrize("shape,n", [((160, 160), 48), ((8, 2048), 24), ((1, 4), 5), ((4, 4), 1)])
def test_odd_geometries(shape, n):
    """4-band clusters (160x160), rows too wide for the materialisation chunk (lazy fallback),
    degenerate images, batch of 1"""
    rng = random.Random(shape[0])
    names = ["Rotate", "Equalize", "Sharpness", "Contrast", "ShearY", "Color", "AutoContrast", "TranslateY", "Cutout"]
    policies = [[(rng.choice(names), 1.0, rng.random()), (rng.choice(names), 1.0, rng.random())] for _ in range(60)]
    pol = CompiledPolicy(policies)
    batch = synth_batch(n, shape, seed=shape[1])
    seed_all(4)
    want = oracle_policy(policies, batch)
    seed_all(4)
    samples, boxes = pol.sample_parity(n, shape[0], shape[1])
    got = augment_batch(pol, dev(batch), TailSpec.raw_u8(), samples, boxes).cpu().numpy()
    bad = [i for i in range(n) if not np.array_equal(got[i], want[i])]
    assert not bad, (shape, bad[:5], [policies[samples[i]["sub"]] for i in bad[:5]])
    tail = TailSpec(None, 0, True, IMAGENET_MEAN, IMAGENET_STD, 0, torch.float32)
    seed_all(4)
    want_f = pil_path.run_chain_on_batch(pil_path.fixed_shape_chain(policies, IMAGENET_MEAN, IMAGENET_STD, True, 0), batch)
    seed_all(4)
    samples, boxes = pol.sample_parity(n, shape[0], shape[1], tail)
    assert torch.equal(augment_batch(pol, dev(batch), tail, samples, boxes).cpu(), want_f)


def test_device_resident_loader_matches_oracle_chain():
    """get_dataloaders drop-in (reference data.py:37-225, row N1): reference signature + conf keys, device-resident
    uint8 dataset, batches come out augmented on the GPU; in parity mode they equal the reference chain applied
    to the same samples in the same order"""
    from sklearn.model_selection import StratifiedShuffleSplit
    from fast_autoaugment_b200.conf import Config as C
    from fast_autoaugment_b200.data import DeviceDataset, GpuAugmentedLoader, SubsetSampler, get_dataloaders
    n, b = 200, 32
    images = synth_batch(n, (32, 32), seed=50)
    labels = np.arange(n) % 10
    policies = archive.fa_reduced_cifar10()
    tail = TailSpec.cifar(16, torch.float32)
    loader = GpuAugmentedLoader(DeviceDataset(images[:96], labels[:96]), b, policies, tail, shuffle=False, parity=True)
    assert len(loader) == 3
    seed_all(13)
    got = [(d.cpu(), l.cpu()) for d, l in loader]
    seed_all(13)
    want = pil_path.run_chain_on_batch(pil_path.cifar_train_chain(policies, 16), images[:96])
    assert torch.equal(torch.cat([d for d, _ in got]), want)
    assert torch.equal(torch.cat([l for _, l in got]), torch.from_numpy(labels[:96]))
    # the reference signature: conf-driven policy / cutout, stratified split, samplers, four return values
    C.get().clear()
    C.get().update({"aug": "fa_reduced_cifar10", "cutout": 16, "faa_parity": True})
    root = {"train": (images, labels), "test": (images[:b], labels[:b])}
    sampler, train, valid, test = get_dataloaders("cifar10", b, root, split=0.15, split_idx=1)
    sss = StratifiedShuffleSplit(n_splits=5, test_size=0.15, random_state=0).split(list(range(n)), list(labels))
    for _ in range(2):
        tr_idx, va_idx = next(sss)
    assert isinstance(sampler, torch.utils.data.SubsetRandomSampler) and list(sampler.indices) == list(tr_idx)
    assert isinstance(valid.sampler, SubsetSampler) and list(valid.sampler.indices) == list(va_idx)
    assert len(train) == len(tr_idx) // b and len(valid) == -(-len(va_idx) // b)
    # the validation loader shares transform_train (data.py:217-219): policy + crop + flip + cutout, in order
    seed_all(3)
    got_v = torch.cat([d.cpu() for d, _ in valid])
    lab_v = torch.cat([l.cpu() for _, l in valid])
    seed_all(3)
    want_v = pil_path.run_chain_on_batch(pil_path.cifar_train_chain(policies, 16), images[va_idx])
    assert torch.equal(got_v, want_v) and torch.equal(lab_v, torch.from_numpy(labels[va_idx]))
    # test loader: ToTensor + Normalize only (transform_test, data.py:45-48)
    t0 = next(iter(test))[0]
    ref = torch.from_numpy(np.stack([pil_path.fixed_shape_chain(None, pil_path.CIFAR_MEAN, pil_path.CIFAR_STD, False, 0)(
        PIL.Image.fromarray(im)).numpy() for im in images[:b]]))
    assert t0.is_cuda and t0.dtype == torch.float32 and torch.equal(t0.cpu(), ref)
    # fused-Philox production mode, fp16: every epoch draws new decisions; split=0 -> empty validation loader
    C.get().update({"faa_parity": False, "faa_out_dtype": "float16"})
    sampler, train, valid, test = get_dataloaders("cifar10", b, root, split=0.0)
    assert sampler is None and len(valid) == 0 and len(train) == n // b
    a = [d.clone() for d, _ in train]
    assert a[0].is_cuda and a[0].dtype == torch.float16 and tuple(a[0].shape) == (b, 3, 32, 32)
    # target_lb filters both index lists (data.py:196-198)
    _, tr1, va1, _ = get_dataloaders("cifar10", b, root, split=0.15, target_lb=3)
    assert all(int(l) == 3 for _, ls in va1 for l in ls) and len(tr1.sampler) == sum(1 for i in StratifiedShuffleSplit(
        n_splits=5, test_size=0.15, random_state=0).split(list(range(n)), list(labels)).__next__()[0] if labels[i] == 3)
    with pytest.raises(ValueError):
        get_dataloaders("mnist", b, root)
    C.get().update({"aug": "no_such_policy"})
    with pytest.raises(ValueError):
        get_dataloaders("cifar10", b, root)
    C.get().clear()


def test_reference_train_loop_body_runs_unchanged():
    """reference train.py:47-58 (the body of run_epoch) against the drop-in loaders and mixup: `.cuda()` on the
    yielded tensors is a no-op, mixup returns the reference's 4-tuple, a WRN-style step consumes the batch"""
    from fast_autoaugment_b200.aug_mixup import mixup
    from fast_autoaugment_b200.conf import Config as C
    from fast_autoaugment_b200.data import get_dataloaders
    n, b = 256, 64
    images = synth_batch(n, (32, 32), seed=3)
    labels = np.arange(n) % 10
    C.get().clear()
    C.get().update({"aug": "fa_reduced_cifar10", "cutout": 16, "mixup": 0.2, "epoch": 1})
    _, loader, _, _ = get_dataloaders("cifar10", b, {"train": (images, labels)}, split=0.0)
    model = torch.nn.Sequential(torch.nn.Conv2d(3, 8, 3, padding=1), torch.nn.ReLU(), torch.nn.AdaptiveAvgPool2d(1),
                                torch.nn.Flatten(), torch.nn.Linear(8, 10)).cuda()
    optimizer = torch.optim.SGD(model.parameters(), lr=0.01)
    ce = torch.nn.CrossEntropyLoss()
    total_steps = len(loader)
    steps = 0
    for data, label in loader:                                    # train.py:47
        steps += 1
        ptr = data.data_ptr()
        data, label = data.cuda(), label.cuda()                   # train.py:49
        assert data.data_ptr() == ptr and data.dtype == torch.float32
        if C.get().conf.get('mixup', 0.0) <= 0.0 or optimizer is None:
            preds = model(data)
            loss = ce(preds, label)
        else:                                                     # train.py:54-58
            data, targets, shuffled_targets, lam = mixup(data, label, C.get()['mixup'])
            preds = model(data)
            loss = lam * ce(preds, targets) + (1 - lam) * ce(preds, shuffled_targets)
            assert 0.5 <= lam <= 1.0 and targets.shape == shuffled_targets.shape
            del shuffled_targets, lam
        optimizer.zero_grad()
        loss.backward()
        optimizer.step()
        assert torch.isfinite(loss)
    assert steps == total_steps == n // b
    C.get().clear()
