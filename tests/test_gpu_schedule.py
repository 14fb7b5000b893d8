"""The production schedule at benchmark size, image by image.

Every other GPU test drives the kernels with explicit decision records, which takes the unchained, event-ordered
route.  The launches users time - fused Philox sampling with `FusedAugmenter(..., overlap_calls=True)` and
`run_many` - take a different one: resolve(N+1), mid(N) and light(N) chained on one stream with programmatic
dependent launches and ticket words, persistent mid / light rows that loop over their schedule entries, two program
slots with completion counters and one scratch image per slot, resolve-ahead speculation, and for tiny images
self-resolving CTAs that release the next step at once.  Here those launches are compared with two independent
references on the same decisions:

* the records route: `philox_records` + `augment_batch(..., d_s, d_b)` on a fresh policy handle (no chain, no
  persistent rows, no speculation), `torch.equal` for every image of every step;
* the host emulation (tests/emu) on the same records copied to the host, for every image of two steps per case:
  fp32 bit-exact, fp16 / bf16 equal to the emulator's fp32 value rounded once, uint8 equal to its bytes.

Runs in about 80 s on one B200 (1000 W power limit), half of it in the fallback-schedule subprocesses.
"""
import hashlib
import json
import os
import random
import subprocess
import sys

import numpy as np
import pytest
import torch

from helpers import ROOT, TABLE_STATS, emu_augment, exact_norm_table, fma_shortcut_rounds_like_the_table, synth_batch

from fast_autoaugment_b200 import _lib, archive
from fast_autoaugment_b200.distributed import philox_records
from fast_autoaugment_b200.engine import CompiledPolicy, FusedAugmenter, TailSpec, augment_batch

pytestmark = pytest.mark.gpu

SEED = 41
DTYPES = (torch.float16, torch.bfloat16, torch.float32, torch.uint8)
WORKLOADS = {"imagenet224": (224, 512, "fa_resnet50_rimagenet"),
             "effnet380": (380, 256, "fa_resnet50_rimagenet"),
             "cifar32": (32, 512, "fa_reduced_cifar10")}


def _tail(workload, dt):
    if workload == "cifar32":
        return TailSpec.cifar(16, dt)
    return TailSpec.imagenet(16 if workload == "effnet380" else 0, dt)


def _pool(n, size, seed):
    return torch.from_numpy(synth_batch(n, (size, size), seed=seed)).cuda()


def _host_records(d_s, d_b, n, n_op):
    samples = d_s.cpu().numpy().reshape(-1).view(_lib.SAMPLE_DTYPE)
    boxes = d_b.cpu().numpy().reshape(-1).view(_lib.BOX_DTYPE).reshape(n, n_op)
    return samples, boxes


def _bad(got, want):
    return [i for i in range(got.shape[0]) if not torch.equal(got[i], want[i])]


def _check_records_route(pol, tail, steps, seed=SEED, what=""):
    """steps: [(input, output, first_index)] -> each output equals the records route on a fresh handle; returns the
    records of every step"""
    ref = CompiledPolicy(pol.policies)
    H, W = steps[0][0].shape[1:3]
    recs = []
    for k, (x, got, fi) in enumerate(steps):
        B = x.shape[0]
        d_s, d_b = philox_records(ref, B, H, W, tail, seed, fi, "cuda")
        want = augment_batch(ref, x, tail, d_s, d_b)
        bad = _bad(got, want)
        assert not bad, (what, tail.out_dtype, "step", k, "first_index", fi, "B", B, len(bad), bad[:8])
        recs.append((d_s, d_b))
    return recs


def _emu_reference(emu, pol, x, recs, tail):
    """(uint8 HWC, fp32 NCHW) of the host emulation on the same decisions"""
    B = x.shape[0]
    samples, boxes = _host_records(*recs, B, pol.n_op)
    xn = x.cpu().numpy()
    f32 = emu_augment(emu, pol, xn, samples, boxes, tail, exact_norm_table(tail.mean, tail.std))
    u8 = emu_augment(emu, pol, xn, samples, boxes, tail, None)
    return torch.from_numpy(u8), torch.from_numpy(f32)


def _check_emu(got, dt, u8, f32, what):
    want = u8 if dt == torch.uint8 else f32.to(dt)
    bad = _bad(got.cpu(), want)
    assert not bad, (what, dt, "vs emulator", len(bad), bad[:8])


def _bench_like(pol, tail, xs, B, K, warmup, world=1, rank=0, seed=SEED):
    """bench.py's sequence on one rank: `warmup` overlapped single calls, then K steps in one run_many, the inputs rotated;
    every step writes its own output.  -> [(input, output, first_index)]"""
    H, W = xs[0].shape[1:3]
    f = FusedAugmenter(pol, tail, H, W, seed, overlap_calls=True)
    outs = [f.empty_out(B) for _ in range(warmup + K)]
    steps = []
    for i in range(warmup):
        fi = (i * world + rank) * B
        f(xs[i % len(xs)], outs[i], fi)
        steps.append((xs[i % len(xs)], outs[i], fi))
    ins = [xs[(warmup + i) % len(xs)] for i in range(K)]
    plan = f.plan_many(ins, outs[warmup:])
    f0 = (warmup * world + rank) * B
    f.run_many(plan, f0, stride=world * B)
    steps += [(ins[i], outs[warmup + i], f0 + i * world * B) for i in range(K)]
    torch.cuda.synchronize()
    return steps


# ---------------------------------------------------------------------------------------------------------------
# (a) the benchmark workloads, every output dtype, both references

@pytest.mark.parametrize("workload,world,rank", [("imagenet224", 1, 0), ("imagenet224", 8, 3), ("effnet380", 1, 0),
                                                 ("cifar32", 1, 0)])
def test_benchmark_workload_equals_records_route_and_emulator(workload, world, rank, emu):
    """bench.py's launches: 2 overlapped calls + run_many of 8 steps, 4 input buffers rotated; world=8 rank=3 is the
    stride / offset of rank 3 of an 8-GPU run.  224 / 380: chained resolve + persistent mid + light rows; CIFAR:
    self-resolving launches (chain = 3)."""
    S, B, pol_name = WORKLOADS[workload]
    pol = CompiledPolicy(getattr(archive, pol_name)())
    xs = [_pool(B, S, seed=100 + k) for k in range(4)]
    emu_ref = {}
    for dt in DTYPES:
        tail = _tail(workload, dt)
        steps = _bench_like(pol, tail, xs, B, K=8, warmup=2, world=world, rank=rank)
        recs = _check_records_route(pol, tail, steps, what=workload)
        for k in (1, 6):                   # one overlapped single call, one run_many step
            if k not in emu_ref:
                emu_ref[k] = _emu_reference(emu, pol, steps[k][0], recs[k], tail)
            _check_emu(steps[k][1], dt, *emu_ref[k], (workload, "step", k))


@pytest.mark.parametrize("dt", [torch.float16, torch.bfloat16])
def test_exact_table_half_outputs_in_the_chained_schedule(dt, emu):
    """custom Normalize stats that refuse the fma shortcut: the fp16 / bf16 TAB=true light and mid kernels, persistent,
    chained, at 224x224 b512"""
    mean, std = TABLE_STATS[str(dt)[len("torch."):]]
    assert not fma_shortcut_rounds_like_the_table(mean, std, dt)
    pol = CompiledPolicy(archive.fa_resnet50_rimagenet())
    tail = TailSpec(None, 0, True, mean, std, 0, dt)
    xs = [_pool(512, 224, seed=120 + k) for k in range(4)]
    steps = _bench_like(pol, tail, xs, 512, K=4, warmup=1)
    recs = _check_records_route(pol, tail, steps, what="table")
    for k in (0, 3):
        _check_emu(steps[k][1], dt, *_emu_reference(emu, pol, steps[k][0], recs[k], tail), ("table", k))


# ---------------------------------------------------------------------------------------------------------------
# (b) persistent rows that run many rounds of different programs

GEO = ["ShearX", "ShearY", "TranslateX", "TranslateY", "Rotate", "TranslateXAbs", "TranslateYAbs"]
LUTS = ["Invert", "Solarize", "Posterize", "Brightness", "Posterize2"]
STATS = ["Equalize", "AutoContrast", "Contrast"]


def _light_policy(rng):
    """LUT, Color, Cutout and gather programs at varying levels: every program of the streaming kernel"""
    subs = []
    for _ in range(64):
        r = rng.random
        t = rng.randrange(8)
        if t == 0:
            subs.append([(rng.choice(LUTS), 1.0, r()), (rng.choice(LUTS), 1.0, r())])
        elif t == 1:
            subs.append([("Color", 1.0, r()), (rng.choice(LUTS), 1.0, r())])
        elif t == 2:
            subs.append([("Color", 1.0, r())])
        elif t == 3:
            subs.append([("Cutout", 1.0, 0.05 + 0.95 * r())])
        elif t == 4:
            subs.append([(rng.choice(GEO), 1.0, r()), (rng.choice(LUTS), 1.0, r())])
        elif t == 5:
            subs.append([(rng.choice(LUTS), 1.0, r()), (rng.choice(GEO), 1.0, r())])
        elif t == 6:
            subs.append([(rng.choice(GEO), 1.0, r()), (rng.choice(GEO), 1.0, r())])
        else:
            subs.append([(rng.choice(LUTS), 1.0, r())])
    return subs


def _mid_policy(rng):
    """statistics LUTs, Sharpness and the two-stage pairs of the mid kernel (Sharpness -> gather and Sharpness -> Color /
    Cutout go through the scratch image of the slot)"""
    subs = []
    for _ in range(64):
        r = rng.random
        t = rng.randrange(9)
        if t == 0:
            subs.append([(rng.choice(STATS), 1.0, r())])
        elif t == 1:
            subs.append([(rng.choice(STATS), 1.0, r()), (rng.choice(LUTS), 1.0, r())])
        elif t == 2:
            subs.append([("Sharpness", 1.0, r())])
        elif t == 3:
            subs.append([("Sharpness", 1.0, r()), (rng.choice(LUTS), 1.0, r())])
        elif t == 4:
            subs.append([("Sharpness", 1.0, r()), (rng.choice(GEO), 1.0, r())])
        elif t == 5:
            subs.append([("Sharpness", 1.0, r()), (rng.choice(["Color", "Cutout"]), 1.0, 0.05 + 0.95 * r())])
        elif t == 6:
            subs.append([(rng.choice(STATS), 1.0, r()), (rng.choice(["Color", "Cutout", "Sharpness"]), 1.0, 0.05 + 0.95 * r())])
        elif t == 7:
            subs.append([(rng.choice(STATS), 1.0, r()), (rng.choice(GEO), 1.0, r())])
        else:
            subs.append([(rng.choice(LUTS + GEO), 1.0, r()), (rng.choice(STATS + ["Sharpness"]), 1.0, r())])
    return subs


def _segment_policy(kind):
    rng = random.Random({"light": 1, "mid": 2, "mix": 3}[kind])
    if kind == "light":
        return _light_policy(rng)
    if kind == "mid":
        return _mid_policy(rng)
    return _light_policy(rng)[:32] + _mid_policy(rng)[:32]


@pytest.fixture(scope="module")
def pool224():
    return _pool(2048 + 2, 224, seed=7)


@pytest.mark.parametrize("B", [1, 73, 74, 75, 84, 85, 589, 2048])
@pytest.mark.parametrize("kind", ["light", "mid", "mix"])
def test_persistent_rows_over_many_rounds(kind, B, pool224, monkeypatch):
    """entry counts below, at and above the persistent rows (84 light rows, 74 mid rows on a B200): a row's second and
    later rounds must not see state (LUTs, float tables, program, mbarrier phase, statistics records, scratch image) of
    the entry before"""
    monkeypatch.setenv("FAA_SPLIT_MIN", "0")
    pol = CompiledPolicy(_segment_policy(kind))
    tail = TailSpec.imagenet(0, torch.float16)
    f = FusedAugmenter(pol, tail, 224, 224, SEED)
    xs = [pool224[k:k + B] for k in range(3)]
    outs = [f.empty_out(B) for _ in range(3)]
    f.run_many(f.plan_many(xs, outs), 5 * B, stride=B)
    torch.cuda.synchronize()
    _check_records_route(pol, tail, [(xs[k], outs[k], 5 * B + k * B) for k in range(3)], what=(kind, B))


# ---------------------------------------------------------------------------------------------------------------
# (c) overlapped single calls: the overlap guard, speculation misses, batch-size changes

SHARP_POLICY = [[("Sharpness", 1.0, 0.9), ("ShearX", 1.0, 0.3)], [("Sharpness", 1.0, 0.1), ("Rotate", 1.0, 0.8)],
                [("Sharpness", 1.0, 0.7), ("TranslateY", 1.0, 0.6)], [("Sharpness", 1.0, 0.3), ("Color", 1.0, 0.8)],
                [("Sharpness", 1.0, 0.6), ("Equalize", 1.0, 0.5)], [("Equalize", 1.0, 0.4), ("Sharpness", 1.0, 0.2)],
                [("Sharpness", 1.0, 0.8), ("Cutout", 1.0, 0.5)], [("Invert", 1.0, 0.5), ("Solarize", 1.0, 0.3)]]


def test_overlapped_calls_with_hits_misses_and_seed_change(pool224):
    """speculation hits, stride changes, a repeated index, an odd index and a seed change, every call overlapped"""
    pol = CompiledPolicy(archive.fa_resnet50_rimagenet())
    tail = TailSpec.imagenet(0, torch.float16)
    B = 512
    f = FusedAugmenter(pol, tail, 224, 224, SEED, overlap_calls=True)
    firsts = [0, B, 2 * B, 3 * B, 10 * B, 17 * B, 24 * B, 24 * B, 7, 7 + B]
    calls = []
    for k, fi in enumerate(firsts):
        x = pool224[(k % 4) * 8:(k % 4) * 8 + B]
        calls.append((x, f(x, f.empty_out(B), fi), fi))
    f.rng.seed = SEED + 1
    seeded = [(pool224[:B], f(pool224[:B], f.empty_out(B), 8 * B), 8 * B), (pool224[8:8 + B], f(pool224[8:8 + B], f.empty_out(B), 9 * B), 9 * B)]
    torch.cuda.synchronize()
    _check_records_route(pol, tail, calls, what="sequence")
    _check_records_route(pol, tail, seeded, seed=SEED + 1, what="seed change")


@pytest.mark.parametrize("policy", ["fa_resnet50_rimagenet", "sharpness"])
def test_batch_size_changes_inside_a_live_chain(policy, pool224):
    """GpuAugmentedLoader(drop_last=False) changes the batch size on every epoch's last batch: the program and scratch
    slots move with the batch, the speculation misses; 83 / 84 images at 224x224 fall on both sides of the split
    threshold (one kernel vs resolve + mid + light)"""
    pol = CompiledPolicy(archive.fa_resnet50_rimagenet() if policy != "sharpness" else SHARP_POLICY)
    tail = TailSpec.imagenet(0, torch.float16)
    f = FusedAugmenter(pol, tail, 224, 224, SEED, overlap_calls=True)
    calls, fi = [], 0
    for k, B in enumerate([512, 512, 300, 512, 83, 84, 83, 512]):
        x = pool224[k * 3:k * 3 + B]
        calls.append((x, f(x, f.empty_out(B), fi), fi))
        fi += B
    torch.cuda.synchronize()
    _check_records_route(pol, tail, calls, what=("batch sizes", policy))


@pytest.mark.parametrize("workload", ["imagenet224", "cifar32"])
def test_output_fed_back_as_input(workload, emu):
    """uint8 HWC outputs fed to the next call: the overlap guard must order the launch behind the step that wrote its
    input (and behind the step that read the buffer it writes)"""
    S = 224 if workload == "imagenet224" else 32
    B = 96
    pol = CompiledPolicy(getattr(archive, WORKLOADS[workload][2])())
    tail = TailSpec.imagenet(0, torch.uint8) if S == 224 else TailSpec.cifar(16, torch.uint8)
    x0 = _pool(B, S, seed=33)
    f = FusedAugmenter(pol, tail, S, S, SEED, overlap_calls=True)
    a, b, c = f.empty_out(B), f.empty_out(B), f.empty_out(B)
    f(x0, a, 0)                     # a = aug(x0)
    f(a, b, B)                      # reads what the previous call wrote
    f(b, a, 2 * B)                  # reads the previous output, writes the previous input
    f(x0, c, 3 * B)                 # independent again
    torch.cuda.synchronize()
    ref = CompiledPolicy(pol.policies)

    def records_route(x, fi):
        d_s, d_b = philox_records(ref, B, S, S, tail, SEED, fi, "cuda")
        return augment_batch(ref, x, tail, d_s, d_b), (d_s, d_b)

    w1, _ = records_route(x0, 0)
    w2, r2 = records_route(w1, B)
    w3, _ = records_route(w2, 2 * B)
    w4, _ = records_route(x0, 3 * B)
    for k, (got, want) in enumerate([(b, w2), (a, w3), (c, w4)]):
        bad = _bad(got, want)
        assert not bad, (workload, "call", k + 2, len(bad), bad[:8])
    u8, _ = _emu_reference(emu, pol, w1, r2, tail)
    _check_emu(b, torch.uint8, u8, None, (workload, "fed back"))


def test_calls_alternating_between_two_streams(pool224):
    """one handle, consecutive calls handed from stream to stream (each stream waits for the other): a call is
    only overlapped with its predecessor on the same stream"""
    pol = CompiledPolicy(archive.fa_resnet50_rimagenet())
    tail = TailSpec.imagenet(0, torch.float16)
    B = 512
    f = FusedAugmenter(pol, tail, 224, 224, SEED, overlap_calls=True)
    streams = [torch.cuda.Stream(), torch.cuda.Stream()]
    outs = [f.empty_out(B) for _ in range(6)]
    torch.cuda.synchronize()
    calls = []
    for k in range(6):
        s = streams[k % 2]
        s.wait_stream(streams[(k + 1) % 2])
        x = pool224[k * 5:k * 5 + B]
        with torch.cuda.stream(s):
            f(x, outs[k], k * B)
        calls.append((x, outs[k], k * B))
    torch.cuda.synchronize()
    _check_records_route(pol, tail, calls, what="two streams")


# ---------------------------------------------------------------------------------------------------------------
# (d) the documented fallback schedules (read once per process: each runs in a subprocess)

KNOBS = ["FAA_CHAIN=0", "FAA_PERSIST=0", "FAA_SELF=0", "FAA_MID=0", "FAA_HEAVY=1", "FAA_OCTETS=0", "FAA_STAGE=0"]
SCHEDULE_KNOBS = ("FAA_CHAIN", "FAA_PERSIST", "FAA_SELF", "FAA_MID", "FAA_HEAVY", "FAA_OCTETS", "FAA_STAGE", "FAA_SPLIT",
                  "FAA_SPLIT_MIN", "FAA_AHEAD", "FAA_LPT", "FAA_MAT", "FAA_PDL", "FAA_CHAIN_SMALL", "FAA_BANDS",
                  "FAA_LIGHT_BANDS", "FAA_MID_BANDS", "FAA_MID_THREADS", "FAA_ROWS_MID", "FAA_ROWS_LIGHT", "FAA_PRIO",
                  "FAA_ORDER", "FAA_MID_STREAM", "FAA_SMALL_THREADS")


def schedule_digests(path):
    """Per-image SHA-256 of a short bench-like run (224x224 b512 and CIFAR b128, fp16) -> JSON at `path`."""
    res = {}
    for name, S, B in (("imagenet224", 224, 512), ("cifar32", 32, 128)):
        pol = CompiledPolicy(getattr(archive, WORKLOADS[name][2])())
        xs = [_pool(B, S, seed=200 + k) for k in range(4)]
        steps = _bench_like(pol, _tail(name, torch.float16), xs, B, K=3, warmup=1)
        res[name] = [[hashlib.sha256(o[i].cpu().numpy().tobytes()).hexdigest() for i in range(B)] for _, o, _ in steps]
    with open(path, "w") as f:
        json.dump(res, f)


def _digests_in_subprocess(tmp_path, knob):
    env = {k: v for k, v in os.environ.items() if k not in SCHEDULE_KNOBS}
    if knob:
        k, v = knob.split("=")
        env[k] = v
    out = os.path.join(str(tmp_path), "digests.json")
    code = ("import sys; sys.path[:0] = [%r, %r]; import test_gpu_schedule as m; m.schedule_digests(%r)"
            % (os.path.join(ROOT, "tests"), ROOT, out))
    cmd = [sys.executable] + (["-s"] if sys.flags.no_user_site else []) + ["-B", "-c", code]
    # the chained and persistent kernels spin on tickets and counters: a deadlock must fail, not hang the session
    r = subprocess.run(cmd, env=env, cwd=str(tmp_path), capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, (knob, r.stdout[-2000:], r.stderr[-4000:])
    with open(out) as f:
        return json.load(f)


@pytest.fixture(scope="module")
def default_digests(tmp_path_factory):
    return _digests_in_subprocess(tmp_path_factory.mktemp("default"), None)


@pytest.mark.parametrize("knob", KNOBS)
def test_fallback_schedules_compute_the_default_result(knob, default_digests, tmp_path):
    got = _digests_in_subprocess(tmp_path, knob)
    for name, want in default_digests.items():
        for k, (g, w) in enumerate(zip(got[name], want)):
            bad = [i for i in range(len(w)) if g[i] != w[i]]
            assert not bad, (knob, name, "step", k, len(bad), bad[:8])
