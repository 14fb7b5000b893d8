"""Shared helpers of the test-suite (inputs, emulator driver, comparisons)."""
import ctypes as C
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
GOLDEN = os.path.join(ROOT, "tests", "golden")

ALL_OPS = ["ShearX", "ShearY", "TranslateX", "TranslateY", "Rotate", "AutoContrast", "Invert",
           "Equalize", "Solarize", "Posterize", "Contrast", "Color", "Brightness", "Sharpness",
           "Cutout", "CutoutAbs", "Posterize2", "TranslateXAbs", "TranslateYAbs"]


def synth(shape, kind, rng):
    """The three input families of SURVEY.md 8(d) (same generator as tests/golden/make_golden.py)."""
    h, w = shape
    if kind == 0:
        return rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
    if kind == 1:
        lo = int(rng.integers(0, 200))
        hi = int(rng.integers(lo + 1, 256))
        ramp = np.linspace(lo, hi, w)[None, :, None] + rng.normal(0, 8, (h, w, 3))
        return np.clip(ramp, 0, 255).astype(np.uint8)
    return np.broadcast_to(rng.integers(0, 256, 3, dtype=np.uint8), (h, w, 3)).copy()


def synth_batch(n, shape, seed):
    rng = np.random.default_rng(seed)
    return np.stack([synth(shape, i % 3, rng) for i in range(n)])


# (policy, image shape, batch) of the policy-level fixtures of tests/golden/golden_chain.npz, drawn in this order
GOLDEN_POLICY_BATCHES = (("fa_reduced_cifar10", (32, 32), 96), ("autoaug_policy", (32, 32), 96),
                         ("fa_reduced_svhn", (32, 32), 48), ("arsaug_policy", (24, 40), 48),
                         ("fa_resnet50_rimagenet", (56, 56), 48))


def make_chain_inputs():
    """The seeded inputs that tests/golden/make_golden.py feeds to the reference for golden_chain.npz."""
    rng = np.random.default_rng(77)
    ins = {}
    for pol, shape, n in GOLDEN_POLICY_BATCHES:
        ins["policy_%s_in" % pol] = np.stack([synth(shape, i % 3, rng) for i in range(n)])
    rng = np.random.default_rng(99)
    ins["cifar_chain_in"] = np.stack([synth((32, 32), i % 3, rng) for i in range(64)])
    return ins


# (policy, image size, images) of the whole-policy digests in golden_hashes.json["live_reference"], drawn in this order
LIVE_POLICY_RUNS = (("fa_reduced_cifar10", 32, 400), ("autoaug_policy", 32, 400), ("fa_resnet50_rimagenet", 64, 100))


def live_input(rng, s, i):
    """Image i of a whole-policy run: noise for odd i, a low-contrast ramp for even i."""
    if i % 2:
        return rng.integers(0, 256, (s, s, 3), dtype=np.uint8)
    return np.clip(np.linspace(60, 180, s)[None, :, None] + rng.normal(0, 6, (s, s, 3)), 0, 255).astype(np.uint8)


def sha_policy(policies):
    """Digest of a policy table, [[(name, prob, level), ...], ...]: equal digests <=> equal tables under `==`."""
    import hashlib
    import json
    rows = [[[str(name), float(p), float(lvl)] for name, p, lvl in sub] for sub in policies]
    return hashlib.sha256(json.dumps(rows).encode()).hexdigest()


def golden_chain():
    """golden_chain.npz (the reference's outputs) plus the inputs they were computed from; the regenerated inputs
    must match the digests make_golden.py recorded, so a change in NumPy's generators cannot pass unnoticed."""
    import hashlib
    import json
    with open(os.path.join(GOLDEN, "golden_hashes.json")) as f:
        want = json.load(f)["chain_inputs"]
    g = dict(np.load(os.path.join(GOLDEN, "golden_chain.npz")))
    for k, a in make_chain_inputs().items():
        assert hashlib.sha256(a.tobytes()).hexdigest() == want[k], k
        g[k] = a
    return g


def exact_norm_table(mean, std):
    """fp32 ToTensor+Normalize value of every byte, computed with torch itself."""
    import torch
    u = torch.arange(256, dtype=torch.uint8)
    x = u.to(torch.float32).div(255)
    m = torch.as_tensor(mean, dtype=torch.float32)[:, None]
    s = torch.as_tensor(std, dtype=torch.float32)[:, None]
    return ((x[None, :] - m) / s).numpy().astype(np.float32).copy()


# mean / std for which a fused multiply-add does NOT round like torch's (u / 255 - mean) / std in that dtype: the
# half-precision launches take the exact normalisation table (the TAB=true light / mid / cluster kernels)
TABLE_STATS = {"float16": ((0.7838, 0.3033, 0.4766), (0.2959, 0.455, 0.2573)),
               "bfloat16": ((0.2401, 0.9531, 0.3522), (0.1511, 0.186, 0.474))}


def fma_shortcut_rounds_like_the_table(mean, std, dt):
    """The host's rule (faa_cabi.cu normalisation()): for every channel and byte u, the dt-rounded
    fmaf(u, (float)(1 / (255 std)), (float)(-mean / std)) equals the dt-rounded exact value.  u * scale + bias is exact in
    float64 at these magnitudes (a 32-bit product plus a 24-bit addend within 2^4), so one rounding to float32 is fmaf."""
    import torch
    tab = torch.from_numpy(exact_norm_table(mean, std))
    u = np.arange(256, dtype=np.float64)
    for c in range(3):
        s, m = float(np.float32(std[c])), float(np.float32(mean[c]))
        scale, bias = float(np.float32(1.0 / (255.0 * s))), float(np.float32(-m / s))
        fma = torch.from_numpy((u * scale + bias).astype(np.float32))
        if not torch.equal(fma.to(dt), tab[c].to(dt)):
            return False
    return True


def emu_augment(emu, pol, batch_u8, samples, boxes, tail=None, norm=None, partner=None, lam=1.0,
                force_generic=False, pool=None, pool_samples=None, pool_boxes=None, first=0):
    """Drive tests/emu like engine.augment_batch drives the kernels.  norm=None -> uint8 HWC."""
    from fast_autoaugment_b200.engine import TailSpec
    tail = tail or TailSpec.raw_u8()
    B, H, W, _ = batch_u8.shape
    oh, ow = tail.out_size if tail.out_size is not None else (H, W)
    table = np.ascontiguousarray(pol.compiled_table(H, W))
    src = np.ascontiguousarray(batch_u8 if pool is None else pool)
    smp = np.ascontiguousarray(samples if pool_samples is None else pool_samples)
    bxs = np.ascontiguousarray(boxes if pool_boxes is None else pool_boxes)
    cur = src
    n_op = pol.n_op
    base = 0
    while base + 2 < n_op:                      # chained windows, like the engine
        nxt = np.zeros_like(cur)
        rc = emu.faa_emu_augment(cur.ctypes.data, cur.shape[0], 0, cur.shape[0], H, W, table.ctypes.data,
                                 pol.n_sub, n_op, smp.ctypes.data, bxs.ctypes.data, base, 0, H, W, 0, None,
                                 nxt.ctypes.data, None, C.c_float(1.0), C.c_float(0.0), int(force_generic))
        assert rc == 0
        cur, base = nxt, base + 2
    if norm is None:
        out = np.zeros((B, oh, ow, 3), np.uint8)
        tab = None
    else:
        out = np.zeros((B, 3, oh, ow), np.float32)
        norm = np.ascontiguousarray(norm, dtype=np.float32)
        tab = norm.ctypes.data
    part = None
    if partner is not None:
        partner = np.ascontiguousarray(partner, dtype=np.int32)
        part = partner.ctypes.data
    rc = emu.faa_emu_augment(cur.ctypes.data, cur.shape[0], first, B, H, W, table.ctypes.data, pol.n_sub, n_op,
                             smp.ctypes.data, bxs.ctypes.data, base, 1, oh, ow, int(tail.cutout > 0), tab,
                             out.ctypes.data, part, C.c_float(np.float32(lam)), C.c_float(np.float32(1 - lam)),
                             int(force_generic))
    assert rc == 0
    return out


def set_emu_sigs(emu):
    vp = C.c_void_p
    emu.faa_emu_augment.argtypes = [vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, vp, C.c_int, C.c_int, vp, vp,
                                    C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, vp, vp, vp, C.c_float, C.c_float,
                                    C.c_int]
    emu.faa_emu_augment.restype = C.c_int
    emu.faa_emu_philox.argtypes = [vp, vp, C.c_int, C.c_int, vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, vp, vp]
    emu.faa_emu_philox.restype = C.c_int
    emu.faa_emu_philox_block.argtypes = [vp, vp, vp]
    emu.faa_emu_philox_block.restype = None
    return emu


def seed_all(s):
    import random
    import torch
    random.seed(s)
    np.random.seed(s)
    torch.manual_seed(s)
