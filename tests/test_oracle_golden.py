"""Pin BOTH oracle layers against the committed outputs of the reference
(tests/golden/*, written by tests/golden/make_golden.py from the reference checkout)."""
import hashlib
import json
import os
import random

import numpy as np
import PIL.Image
import pytest
import torch

from helpers import ALL_OPS, GOLDEN, LIVE_POLICY_RUNS, golden_chain, live_input, seed_all, sha_policy

from fast_autoaugment_b200 import archive
from oracle import np_model, pil_path


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


@pytest.fixture(scope="module")
def hashes():
    with open(os.path.join(GOLDEN, "golden_hashes.json")) as f:
        return json.load(f)


def test_survey_table_hashes(hashes):
    """SURVEY.md 8c golden table: rng(1234) noise, seed 0, level 0.7 (Posterize 0.3), 32 and 224"""
    table = hashes["survey_table"]
    for s in (32, 224):
        img = np.random.default_rng(1234).integers(0, 256, (s, s, 3), dtype=np.uint8)
        assert sha(img) == table["input_%d" % s]
        for name in ALL_OPS:
            lvl = 0.3 if name == "Posterize" else 0.7
            random.seed(0)
            np.random.seed(0)
            out = np.asarray(pil_path.apply_op(PIL.Image.fromarray(img), name, lvl))
            assert sha(out) == table["%s_%d" % (name, s)], (name, s, "pil_path")
            random.seed(0)
            np.random.seed(0)
            out2 = np_model.policy_call(img, [[(name, 1.0, lvl)]])
            # policy_call draws choice+gate first; redo with the op-only draw order
            random.seed(0)
            np.random.seed(0)
            v = np_model.magnitude(name, lvl)
            mirror = (random.random() > 0.5) if name in np_model.MIRRORED else False
            ux = uy = 0.0
            if name in np_model.NEEDS_BOX:
                ux, uy = np.random.random_sample(), np.random.random_sample()
            out2 = np_model.run_op_resolved(img, name, v, mirror, ux, uy)
            assert sha(out2) == table["%s_%d" % (name, s)], (name, s, "np_model")


def test_chained_policy_digests(hashes):
    for key, want in hashes["chained_seeds_0_63"].items():
        pol_name, s = key.rsplit("_", 1)
        s = int(s)
        policies = getattr(archive, pol_name)()
        img = np.random.default_rng(1234).integers(0, 256, (s, s, 3), dtype=np.uint8)
        for layer in ("pil", "np"):
            h = hashlib.sha256()
            t = pil_path.PolicyTransform(policies)
            for seed in range(64):
                random.seed(seed)
                np.random.seed(seed)
                if layer == "pil":
                    h.update(np.asarray(t(PIL.Image.fromarray(img))).tobytes())
                else:
                    h.update(np_model.policy_call(img, policies).tobytes())
            assert h.hexdigest() == want, (key, layer)


@pytest.mark.parametrize("tag", ["32x32", "24x40"])
def test_per_op_arrays(tag):
    g = np.load(os.path.join(GOLDEN, "golden_ops.npz"))
    ins, outs, metas = g["in_" + tag], g["out_" + tag], g["meta_" + tag]
    for meta, want in zip(metas, outs):
        name, lvl, seed, kind = json.loads(str(meta))
        img = ins[kind]
        random.seed(seed)
        np.random.seed(seed)
        got = np.asarray(pil_path.apply_op(PIL.Image.fromarray(img), name, lvl))
        assert np.array_equal(got, want), (name, lvl, "pil_path")
        random.seed(seed)
        np.random.seed(seed)
        v = np_model.magnitude(name, lvl)
        mirror = (random.random() > 0.5) if name in np_model.MIRRORED else False
        ux = uy = 0.0
        if name in np_model.NEEDS_BOX and not (name == "Cutout" and v <= 0):
            ux, uy = np.random.random_sample(), np.random.random_sample()
        got2 = np_model.run_op_resolved(img, name, v, mirror, ux, uy)
        assert np.array_equal(got2, want), (name, lvl, "np_model")


def test_policy_outputs_and_chain():
    g = golden_chain()
    for pol_name in ("fa_reduced_cifar10", "autoaug_policy", "fa_reduced_svhn", "arsaug_policy",
                     "fa_resnet50_rimagenet"):
        batch, want = g["policy_%s_in" % pol_name], g["policy_%s_out" % pol_name]
        policies = getattr(archive, pol_name)()
        seed_all(5)
        t = pil_path.PolicyTransform(policies)
        got = np.stack([np.asarray(t(PIL.Image.fromarray(a))) for a in batch])
        assert np.array_equal(got, want), pol_name
        seed_all(5)
        got2 = np.stack([np_model.policy_call(a, policies) for a in batch])
        assert np.array_equal(got2, want), pol_name
    # full CIFAR transform_train, fp32
    seed_all(11)
    out = pil_path.run_chain_on_batch(pil_path.cifar_train_chain(archive.fa_reduced_cifar10(), 16),
                                      g["cifar_chain_in"])
    assert np.array_equal(out.numpy(), g["cifar_chain_out_f32"])
    # numpy model of the tail: pad-crop / flip / ToTensor+Normalize / zero box, same draw order
    seed_all(11)
    policies = archive.fa_reduced_cifar10()
    outs = []
    for a in g["cifar_chain_in"]:
        x = np_model.policy_call(a, policies)
        top = int(torch.randint(0, 9, size=(1,)).item())
        left = int(torch.randint(0, 9, size=(1,)).item())
        x = np_model.pad_crop(x, 4, top, left, 32, 32)
        if bool(torch.rand(1) < 0.5):
            x = np_model.hflip(x)
        t = np_model.to_tensor_normalize(x, pil_path.CIFAR_MEAN, pil_path.CIFAR_STD)
        cy = np.random.randint(32)
        cx = np.random.randint(32)
        outs.append(np_model.zero_box(t, 16, cy, cx))
    assert np.array_equal(np.stack(outs), g["cifar_chain_out_f32"])


def test_mixup_golden(hashes):
    g = golden_chain()
    x_in = g["cifar_chain_out_f32"][:16]                 # the reference mixed the first 16 chain outputs
    torch.manual_seed(3)
    np.random.seed(3)
    x = torch.from_numpy(x_in.copy())
    mixed, t1, t2, lam = pil_path.mixup_pairs(x, torch.arange(16), 0.2)
    assert lam == float(g["mixup_lam"][0])
    assert np.array_equal(t2.numpy(), g["mixup_t2"])
    assert mixed.dtype == torch.float32 and sha(mixed.numpy()) == hashes["mixup_out"]
    resolved = np_model.mixup_resolved(x_in, g["mixup_t2"], lam)
    assert resolved.dtype == np.float32 and sha(resolved) == hashes["mixup_out"]


def test_against_live_reference(hashes):
    """whole policies, image by image, against the reference's own Augmentation run on the same inputs and seeds
    (digests recorded by make_golden.py)"""
    live = hashes["live_reference"]
    rng = np.random.default_rng(5)
    for pol_name, s, n in LIVE_POLICY_RUNS:
        mine = getattr(archive, pol_name)()
        assert sha_policy(mine) == live["policies"][pol_name], pol_name
        want = live["outputs"]["%s_%d" % (pol_name, s)]
        assert len(want) == n
        for i in range(n):
            img = live_input(rng, s, i)
            random.seed(i)
            np.random.seed(i)
            got = pil_path.PolicyTransform(mine)(PIL.Image.fromarray(img))
            assert sha(np.asarray(got))[:16] == want[i], (pol_name, i, "pil_path")
            random.seed(i)
            np.random.seed(i)
            assert sha(np_model.policy_call(img, mine))[:16] == want[i], (pol_name, i, "np_model")
