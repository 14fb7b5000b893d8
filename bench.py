#!/usr/bin/env python
"""bench.py - augmented images/sec of the Fast AutoAugment hot path on B200.

    python bench.py --gpus N --steps K --warmup W            (ours; N>1 via torchrun)
    python bench.py --impl reference --gpus N --steps K --warmup W   (CPU PIL path, rank 0 only)
    python bench.py ... --dump-outputs DIR      (also save what the last timed step computed, see dump_outputs)

A "step" is one pass of the hot path over one batch of synthetic uint8 HWC images:
policy ops -> HFlip -> ToTensor -> Normalize -> NCHW fp16, with the per-sample decisions
drawn by the fused Philox sampler.  Workload = BASELINE.json configs[2] (the configuration the
metric is quoted on): 224x224, batch 512 per GPU, fa_reduced_imagenet policy.  Weak scaling:
every rank processes its own 512-image shard, no data-path collective (images are
independent; SURVEY.md 8e).

The JSON line carries the device-timed `value`, the host-buffer `e2e`, the HBM `roofline`
of the fused kernel (algorithmic bytes 9*H*W per image / measured launch time / measured
copy peak) and the CPU `cpu_baseline` (the reference's PIL/torchvision call sequence as
restated in oracle/pil_path.py, run through a torch DataLoader like reference data.py:214).
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # the benchmark leaves the source tree as it found it (it may be read-only)

WORKLOADS = {
    # name: (H, W, per-GPU batch, policy fn name, tail kind, cutout)
    "imagenet224_b512": (224, 224, 512, "fa_resnet50_rimagenet", "imagenet", 0),
    "cifar32_b512": (32, 32, 512, "fa_reduced_cifar10", "cifar", 16),
    "effnetb4_380_b256": (380, 380, 256, "fa_resnet50_rimagenet", "imagenet", 16),
}
METRIC = "augmented images/sec at 224x224 b512 (1/2/4/8 GPU) + % HBM roofline vs CPU PIL"


def synth_batch(n, h, w, seed):
    """SURVEY.md 8(d) input families, interleaved: uniform noise / low-contrast ramp+noise /
    constant colour (histogram worst case)."""
    import numpy as np
    rng = np.random.default_rng(seed)
    out = np.empty((n, h, w, 3), np.uint8)
    for i in range(n):
        k = i % 3
        if k == 0:
            out[i] = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
        elif k == 1:
            lo = int(rng.integers(0, 200))
            hi = int(rng.integers(lo + 1, 256))
            ramp = np.linspace(lo, hi, w)[None, :, None] + rng.normal(0, 8, (h, w, 3))
            out[i] = np.clip(ramp, 0, 255).astype(np.uint8)
        else:
            out[i] = rng.integers(0, 256, 3, dtype=np.uint8)
    return out


# --------------------------------------------------------------------------------------
# CPU arm: the reference's per-sample PIL chain inside a torch DataLoader
class _ArrayDataset:
    def __init__(self, arrays, n_total, chain):
        self.arrays, self.n_total, self.chain = arrays, n_total, chain

    def __len__(self):
        return self.n_total

    def __getitem__(self, i):
        import PIL.Image
        return self.chain(PIL.Image.fromarray(self.arrays[i % len(self.arrays)])), 0


def _policy_lists(pol_name):
    """The policy table straight from ``fast_autoaugment_b200/policies/*.json`` - WITHOUT importing the
    package (its __init__ dlopens libfaa_b200.so, which must not appear in the reference arm's process)."""
    with open(os.path.join(ROOT, "fast_autoaugment_b200", "policies", pol_name + ".json")) as f:
        d = json.load(f)
    k, rows = d["n_op"], d["table"]
    return [[[d["ops"][int(rows[s * k + j][0])], rows[s * k + j][1], rows[s * k + j][2]] for j in range(k)]
            for s in range(d["n_sub"])]


def _cpu_chain(workload):
    """(chain, kind): the reference's own classes from ``oracle/_ref`` (the verbatim reference package,
    placed there by oracle/build_ref.py) composed like reference data.py:39-44,60-73,92,112 -> kind
    "reference"; the oracle's restatement of the same call sequence when ``oracle/_ref`` is absent -> "port"."""
    h, w, b, pol_name, tail_kind, cutout = WORKLOADS[workload]
    try:
        from oracle import build_ref
        mods = build_ref.import_ref()
    except Exception:
        mods = None
    if mods is not None:
        from torchvision import transforms
        _, ref_archive, _, ref_data = mods
        policies = getattr(ref_archive, pol_name)()
        if tail_kind == "cifar":      # data.py:39-44
            chain = transforms.Compose([transforms.RandomCrop(32, padding=4), transforms.RandomHorizontalFlip(),
                                        transforms.ToTensor(), transforms.Normalize(ref_data._CIFAR_MEAN, ref_data._CIFAR_STD)])
        else:                         # data.py:64,70,72 on an already-sized image (SURVEY.md 3-D)
            chain = transforms.Compose([transforms.RandomHorizontalFlip(), transforms.ToTensor(),
                                        transforms.Normalize(mean=[0.485, 0.456, 0.406], std=[0.229, 0.224, 0.225])])
        chain.transforms.insert(0, ref_data.Augmentation(policies))       # data.py:92-95
        if cutout > 0:
            chain.transforms.append(ref_data.CutoutDefault(cutout))       # data.py:111-112
        return chain, "reference"
    from oracle import pil_path
    policies = _policy_lists(pol_name)
    if tail_kind == "cifar":
        return pil_path.cifar_train_chain(policies, cutout), "port"
    return pil_path.fixed_shape_chain(policies, pil_path.IMAGENET_MEAN, pil_path.IMAGENET_STD, True, cutout), "port"


def cpu_throughput(workload, n_batches, warm_batches, workers):
    """images/s of the reference CPU path over `n_batches` batches after `warm_batches`
    (worker start-up excluded, reference-style DataLoader: data.py:214-216)."""
    import torch
    from torch.utils.data import DataLoader
    h, w, b, *_ = WORKLOADS[workload]
    arrays = synth_batch(min(b, 256), h, w, 1234)
    # Worker task = b/workers images instead of the reference's whole batch per worker: the
    # steady-state rate is the same (workers x per-core rate) but a step (= b images) is then
    # one even round over all workers, so a short timed region is not distorted by whole
    # batches that were prefetched before the clock started.
    task = max(1, b // max(1, min(workers, 16)))  # >= b/16 images per task keeps the main process (IPC) off the critical path
    tasks_per_step = (b + task - 1) // task
    # warm-up must cover the prefetch depth (2 tasks per worker) or the timed steps would drain work
    # that was done before the clock started
    warm_batches = max(warm_batches, 3, (2 * workers + tasks_per_step - 1) // tasks_per_step + 1)
    chain, kind = _cpu_chain(workload)
    ds = _ArrayDataset(arrays, task * tasks_per_step * (n_batches + warm_batches), chain)
    torch.set_num_threads(1)
    dl = DataLoader(ds, batch_size=task, shuffle=False, num_workers=workers, drop_last=True,
                    persistent_workers=False, prefetch_factor=(2 if workers > 0 else None))
    it = iter(dl)
    for _ in range(warm_batches * tasks_per_step):
        next(it)
    t0 = time.perf_counter()
    n = 0
    for _ in range(n_batches * tasks_per_step):
        x, _ = next(it)
        n += x.shape[0]
    dt = time.perf_counter() - t0
    del it
    return n / dt, dt, kind


def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


# --------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu, self.proc, self.lines = gpu_index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.perf_counter(), line.strip()))

    def stop(self, t0, t1):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        for ts, line in self.lines:
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                clk, mxc = float(f[1]), float(f[2])
            except ValueError:
                continue
            mx = mxc
            if t0 - 0.05 <= ts <= t1 + 0.15:
                sm.append(clk)
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        if not sm:       # region shorter than the sampling period: take every sample we have
            for ts, line in self.lines:
                f = [x.strip() for x in line.split(",")]
                try:
                    sm.append(float(f[1]))
                except (ValueError, IndexError):
                    pass
        sm.sort()
        return {"sm_mhz": (sm[len(sm) // 2] if sm else None), "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, STREAM-style copy)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def ncu_traffic(workload):
    """per-launch DRAM bytes of the fused kernel from the committed ncu capture, if any"""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            return json.load(f).get(workload)
    except Exception:
        return None


# --------------------------------------------------------------------------------------
def workload_string(name):
    """One description per workload, IDENTICAL in both arms (what differs - output dtype, sampler, DataLoader -
    goes into separate config keys)."""
    H, W, B, pol_name, tail_kind, cutout = WORKLOADS[name]
    tail = "RandomCrop(32,pad 4)+HFlip+ToTensor+Normalize(CIFAR)" if tail_kind == "cifar" else "HFlip+ToTensor+Normalize(ImageNet)"
    return "%s: synthetic uint8 HWC %dx%d, batch %d per GPU, %s policy, %s%s -> NCHW" % (
        name, H, W, B, pol_name, tail, "+CutoutDefault(%d)" % cutout if cutout else "")


class _Workload:
    """Device-resident buffers + the pre-bound launch of one workload on this rank."""
    NSETS = 4      # input/output sets rotate so that no step finds its data in the 126 MB L2
    DUMP_BYTES = 60 * 10**6     # --dump-outputs: float32 images kept from the last step's output (stays under 64 MB)

    def __init__(self, name, seed, rank, world):
        import torch
        from fast_autoaugment_b200 import archive
        from fast_autoaugment_b200.engine import CompiledPolicy, FusedAugmenter, TailSpec
        self.name, self.rank, self.world = name, rank, world
        self.H, self.W, self.B, pol_name, tail_kind, cutout = WORKLOADS[name]
        self.pol = CompiledPolicy(getattr(archive, pol_name)())
        self.tail = TailSpec.cifar(cutout, torch.float16) if tail_kind == "cifar" else TailSpec.imagenet(cutout, torch.float16)
        self.t_c = self.tail.c_struct(self.H, self.W)
        self.out_shape = (self.B, 3, self.t_c.out_h, self.t_c.out_w)
        self.host_in = torch.from_numpy(synth_batch(self.B, self.H, self.W, 1234 + rank)).pin_memory()
        self.ins = [self.host_in.cuda().clone() for _ in range(self.NSETS)]
        self.outs = [torch.empty(self.out_shape, dtype=torch.float16, device="cuda") for _ in range(self.NSETS)]
        self.in_bytes = self.B * self.H * self.W * 3
        self.out_bytes = self.B * 3 * self.t_c.out_h * self.t_c.out_w * 2
        self.fused = FusedAugmenter(self.pol, self.tail, self.H, self.W, seed, overlap_calls=True)   # (device-resident inputs, never rewritten)
        self.stream = torch.cuda.current_stream()
        self.raw_stream = self.stream.cuda_stream

    def step(self, i):
        self.fused(self.ins[i % self.NSETS], self.outs[i % self.NSETS], (i * self.world + self.rank) * self.B, self.raw_stream)

    def timed(self, steps, warmup, barrier):
        """K steps bracketed by barrier+synchronize, CUDA events on the launching stream -> ms (this rank)."""
        import torch
        for i in range(warmup):
            self.step(i)
        barrier()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        # the K timed steps are issued by ONE call (FusedAugmenter.run_many -> C ABI faa_augment_many): same launches as K
        # calls of self.step, without the interpreter between them (small-image steps are host-bound otherwise)
        plan = self.fused.plan_many([self.ins[(warmup + i) % self.NSETS] for i in range(steps)],
                                    [self.outs[(warmup + i) % self.NSETS] for i in range(steps)])
        t0 = time.perf_counter()
        ev0.record(self.stream)
        self.fused.run_many(plan, (warmup * self.world + self.rank) * self.B, stride=self.world * self.B, stream=self.raw_stream)
        ev1.record(self.stream)
        barrier()
        return ev0.elapsed_time(ev1), t0, time.perf_counter()

    def last_output(self, steps, warmup):
        """(images, rows): float32 copy of what the last of `steps` timed steps after `warmup` wrote, and which rows of
        the batch they are.  An output larger than DUMP_BYTES is represented by a fixed, seeded sample of its images."""
        import numpy as np
        import torch
        out = self.outs[(warmup + steps - 1) % self.NSETS]
        n = min(self.B, self.DUMP_BYTES // (out[0].numel() * 4 + 8))
        rows = np.arange(self.B) if n == self.B else np.sort(np.random.default_rng(0).choice(self.B, n, replace=False))
        return out[torch.from_numpy(rows).to(out.device)].float().cpu().numpy(), rows

    def roofline(self, ms_per_step):
        peak, peak_src = measured_peak()
        alg = self.in_bytes + self.out_bytes          # 3HW read + 6 out_h out_w written (= 9HW when no crop)
        ach = alg / (ms_per_step / 1e3) / 1e9
        return {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                "traffic": ncu_traffic(self.name), "peak_source": peak_src, "algorithmic_bytes_per_launch": alg,
                "kernel": "faa_augment_mid_kernel + faa_augment_light_kernel (+ faa_augment_kernel for crops / odd widths); one step = one pass over the batch"}


def measure_mixup(args, rank, world, barrier, max_over_ranks):
    """Config 4.  One step = augment the local shard once to uint8, partner-only all-to-all of the augmented images,
    one streaming pass that normalises both sources and mixes them in fp32 (aug_mixup.py:21) -> fp16 NCHW.
    Device-timed like the main metric."""
    import torch
    from fast_autoaugment_b200 import archive
    import torch.distributed as dist
    from fast_autoaugment_b200.distributed import PeerPool, mixup_global, mixup_global_peer
    from fast_autoaugment_b200.engine import CompiledPolicy, TailSpec
    H = W = 224
    G = 2048
    b = G // world
    pol = CompiledPolicy(archive.fa_resnet50_rimagenet())
    tail = TailSpec.imagenet(0, torch.float16)
    xs = [torch.from_numpy(synth_batch(b, H, W, 4321 + rank + 17 * i)).cuda() for i in range(2)]
    y = torch.arange(rank * b, (rank + 1) * b, device="cuda")
    steps = args.steps
    tim = {}
    # world > 1: the exchange is fused into the mix kernel (partners read over NVLink peer memory); FAA_MIXUP_A2A=1 or a
    # failing peer mapping selects the NCCL all-to-all route
    peer_pool, route = None, "local"
    if world > 1:
        route = "nccl_all_to_all"
        if os.environ.get("FAA_MIXUP_A2A", "0") != "1":
            try:
                peer_pool = PeerPool(b, H, W, torch.device("cuda", torch.cuda.current_device()))
                route = "nvlink_peer_loads"
            except Exception as e:                      # noqa: BLE001 - report and fall back
                sys.stderr.write("[bench] peer pool unavailable (%s): NCCL all-to-all route\n" % e)
        flag = torch.tensor([1.0 if peer_pool is not None else 0.0], device="cuda")
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)     # all ranks or none
        if float(flag.item()) == 0.0:
            peer_pool, route = None, "nccl_all_to_all"

    def mixup_global(pol_, x_, y_, tail_, alpha_, seed_, step_, timing=None, _a2a=mixup_global):
        if peer_pool is not None:
            return mixup_global_peer(pol_, x_, y_, tail_, alpha_, seed_, step_, peer_pool, timing=timing)
        return _a2a(pol_, x_, y_, tail_, alpha_, seed_, step_, timing=timing)
    for i in range(3):
        mixup_global(pol, xs[i % 2], y, tail, 0.2, args.seed, i)
    barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ex_ms, recv = 0.0, 0
    barrier()
    ev0.record()
    pairs = []
    for i in range(steps):
        t = {}
        mixup_global(pol, xs[i % 2], y, tail, 0.2, args.seed, 3 + i, timing=t)
        pairs.append(t)
    ev1.record()
    barrier()
    ms = ev0.elapsed_time(ev1)
    ex_ms = sum(t["ex0"].elapsed_time(t["ex1"]) for t in pairs) / steps
    recv = pairs[-1]["recv_bytes"]
    aug_ms = sum(t["a0"].elapsed_time(t["ex0"]) for t in pairs) / steps
    mix_ms = sum(t["m0"].elapsed_time(t["m1"]) for t in pairs) / steps
    ms, ex_ms, aug_ms, mix_ms = max_over_ranks([ms, ex_ms, aug_ms, mix_ms])
    alg = G * 9 * H * W
    peak, _ = measured_peak()
    return {"workload": "imagenet224_b2048_mixup: synthetic uint8 HWC 224x224, GLOBAL batch 2048 (%d per GPU), fa_resnet50_rimagenet policy, "
                        "HFlip+ToTensor+Normalize(ImageNet), Mixup alpha 0.2 with global pairing -> NCHW fp16" % b,
            "value": G * steps / (ms / 1e3), "unit": "images/s", "steps": steps, "ms_per_step": ms / steps, "scaling": "strong",
            "phases_ms": {"augment_to_u8": aug_ms, "exchange": ex_ms, "mix": mix_ms,
                          "note": "device time between events around each phase; the rest of ms_per_step is host / gaps"},
            "exchange": {"kind": ("partner images read over NVLink peer memory inside the mix kernel (CUDA IPC mapped buffers, one tiny "
                                  "all-reduce as the step barrier) + all-gather of the labels" if route == "nvlink_peer_loads" else
                                  "partner-only all-to-all of the augmented uint8 images (NCCL all_to_all_single) + all-gather of the labels")
                                 if world > 1 else "none (single GPU: every partner is local)",
                         "route": route,
                         "ms_per_step": ex_ms, "nvlink_bytes_received_per_gpu_per_step": recv,
                         "whole_pool_allgather_bytes_per_gpu_per_step": (world - 1) * b * H * W * 3},
            "roofline": {"bound": "hbm", "achieved": alg / world / (ms / steps / 1e3) / 1e9, "peak": peak, "unit": "GB/s",
                         "frac": alg / world / (ms / steps / 1e3) / 1e9 / peak,
                         "algorithmic_bytes_per_launch": alg // world,
                         "note": "same 9HW per output image as the main metric; the partner's raw read (3HW) is implementation traffic"}}


def measure_train_step(args):
    """North star's last clause: is a CIFAR-10 WRN-40-2 training step still augmentation-bound?  Fused augmentation of
    one 128-image batch (full train chain, fp32 out - what the reference's loader yields) vs one fp32 SGD step of a
    WideResNet-40-2 (reference confs/wresnet40x2_cifar.yaml: depth 40, widen 2, batch 128) on the same GPU."""
    import torch
    import torch.nn as nn
    import torch.nn.functional as F
    from fast_autoaugment_b200 import archive
    from fast_autoaugment_b200.engine import CompiledPolicy, FusedAugmenter, TailSpec

    class Block(nn.Module):
        def __init__(self, i, o, stride):
            super().__init__()
            self.bn1, self.conv1 = nn.BatchNorm2d(i), nn.Conv2d(i, o, 3, stride, 1, bias=False)
            self.bn2, self.conv2 = nn.BatchNorm2d(o), nn.Conv2d(o, o, 3, 1, 1, bias=False)
            self.short = None if (i == o and stride == 1) else nn.Conv2d(i, o, 1, stride, 0, bias=False)

        def forward(self, x):
            y = F.relu(self.bn1(x))
            s = x if self.short is None else self.short(y)
            return self.conv2(F.relu(self.bn2(self.conv1(y)))) + s

    class WRN(nn.Module):                      # plain restatement of the standard architecture, timing only
        def __init__(self, depth=40, widen=2, classes=10):
            super().__init__()
            n, w = (depth - 4) // 6, [16, 16 * widen, 32 * widen, 64 * widen]
            layers = [nn.Conv2d(3, w[0], 3, 1, 1, bias=False)]
            for g in range(3):
                for k in range(n):
                    layers.append(Block(w[g] if k == 0 else w[g + 1], w[g + 1], (1 if g == 0 else 2) if k == 0 else 1))
            self.body, self.bn, self.fc = nn.Sequential(*layers), nn.BatchNorm2d(w[3]), nn.Linear(w[3], classes)

        def forward(self, x):
            return self.fc(F.adaptive_avg_pool2d(F.relu(self.bn(self.body(x))), 1).flatten(1))

    B = 128
    x_u8 = torch.from_numpy(synth_batch(B, 32, 32, 7)).cuda()
    y = torch.randint(0, 10, (B,), device="cuda")
    aug = FusedAugmenter(CompiledPolicy(archive.fa_reduced_cifar10()), TailSpec.cifar(16, torch.float32), 32, 32, 1)
    out = aug.empty_out(B)
    model = WRN().cuda()
    opt = torch.optim.SGD(model.parameters(), lr=0.1, momentum=0.9, nesterov=True, weight_decay=2e-4)
    step = [0]

    def do_aug():
        aug(x_u8, out, step[0] * B)
        step[0] += 1

    def do_train():
        opt.zero_grad(set_to_none=True)
        F.cross_entropy(model(out), y).backward()
        opt.step()

    def both():
        do_aug()
        do_train()

    def timed(fn, n):
        for _ in range(5):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / n

    t_aug, t_train, t_both = timed(do_aug, 300), timed(do_train, 20), timed(both, 20)
    return {"what": "CIFAR-10 b128: fused augmentation (full train chain, fp32 out) vs one fp32 SGD step of WideResNet-40-2",
            "augment_us_per_batch": t_aug * 1e3, "train_step_ms": t_train, "augment_plus_train_step_ms": t_both,
            "augmentation_fraction_of_step": t_aug / t_both,
            "reference_loader_note": "the reference's 8 DataLoader workers deliver ~14-18 k img/s on this chain (BASELINE.md), "
                                     "i.e. ~8 ms per 128-image batch: its step IS augmentation-bound"}


def run_ours(args):
    import torch
    import torch.distributed as dist
    from fast_autoaugment_b200 import _lib
    from fast_autoaugment_b200.engine import make_rng

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (the product has no CPU fallback)"
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(vals):
        t = torch.tensor(vals, device="cuda", dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return [float(v) for v in t.tolist()]

    def all_ranks(val):
        t = torch.zeros(world, device="cuda", dtype=torch.float64)
        t[rank] = val
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return [float(v) for v in t.tolist()]

    wl = _Workload(args.workload, args.seed, rank, world)
    H, W, B, t_c, stream = wl.H, wl.W, wl.B, wl.t_c, wl.stream
    for i in range(args.warmup):
        wl.step(i)
    barrier()
    clocks = ClockSampler(local)
    clocks.start()
    # keep the GPU busy while the clock sampler starts (an idle GPU drops its clocks; the timed region of a
    # 20-step run is ~1.5 ms): untimed extra warm-up steps for ~0.3 s, then straight into the timed region
    tb = time.perf_counter()
    j = args.warmup
    while time.perf_counter() - tb < 0.3:
        for _ in range(8):
            wl.step(j)
            j += 1
        torch.cuda.synchronize()
    # ---- device-timed region: exactly K steps
    launches0 = _lib.lib.faa_launch_count()
    ms_local, t0, t1 = wl.timed(args.steps, args.warmup, barrier)
    launches = int(_lib.lib.faa_launch_count() - launches0)
    if args.dump_outputs and rank == 0:          # (before any later launch reuses the output buffers)
        dump_outputs(args.dump_outputs, *wl.last_output(args.steps, args.warmup))
    # keep the GPU busy a little longer if the region was too short for a clock sample
    if t1 - t0 < 0.4:
        tb = time.perf_counter()
        j = 0
        while time.perf_counter() - tb < 0.5:
            wl.step(j)
            j += 1
        torch.cuda.synchronize()
        t1 = time.perf_counter()
    clk = clocks.stop(t0, t1)

    # ---- end to end through the C ABI with HOST buffers (pinned): H2D + kernel + D2H per step
    host_out = torch.empty(wl.out_shape, dtype=torch.float16).pin_memory()
    keep = torch.empty(wl.out_shape, dtype=torch.float16, device="cuda")

    def e2e_step(i, back):
        rng = make_rng(args.seed, (i * world + rank) * B, wl.tail)
        _lib.check(_lib.lib.faa_augment_host(wl.pol.handle, wl.host_in.data_ptr(), host_out.data_ptr() if back else None,
                                             keep.data_ptr(), B, H, W, C.byref(t_c), C.byref(rng),
                                             C.c_void_p(stream.cuda_stream)))
        if not back:                           # the consumer reads one scalar of the result
            return keep[0, 0, 0, 0].item()

    e2e = {}
    for name, back in (("roundtrip", True), ("device_out", False)):
        for i in range(max(3, args.warmup)):   # same call as the timed one, including the scalar read-back
            e2e_step(i, back)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for i in range(args.steps):
            e2e_step(i, back)
        e1.record(stream)
        barrier()
        e2e[name] = e0.elapsed_time(e1)

    # ---- the other single-GPU configurations of BASELINE.json (configs[1] CIFAR b512, configs[4] 380x380 b256
    #      + CutoutDefault), device-timed the same way, as extra keys of the one line
    also = {}
    for name in ([] if args.no_also else [n for n in ("cifar32_b512", "effnetb4_380_b256") if n != args.workload]):
        w2 = _Workload(name, args.seed, rank, world)
        k2 = args.steps
        ms2, _, _ = w2.timed(k2, max(args.warmup, 5), barrier)
        ms2 = max_over_ranks([ms2])[0]
        also[name] = {"value": world * w2.B * k2 / (ms2 / 1e3), "unit": "images/s", "steps": k2, "ms_per_step": ms2 / k2,
                      "workload": workload_string(name), "roofline": w2.roofline(ms2 / k2)}
        del w2
        torch.cuda.empty_cache()

    # ---- BASELINE configs[3]: 224x224, GLOBAL batch 2048 + Mixup(alpha 0.2) with global pairing, sharded over the ranks
    #      (strong scaling: 2048 / N images per GPU); partners travel by a partner-only all-to-all of raw uint8 images
    mix = None
    if not args.no_also and 2048 % world == 0:
        mix = measure_mixup(args, rank, world, barrier, max_over_ranks)
    train = None
    if not args.no_also and world == 1:
        train = measure_train_step(args)

    # ---- max over ranks
    per_rank = all_ranks(ms_local / args.steps)
    ms, ms_rt, ms_dev = max_over_ranks([ms_local, e2e["roundtrip"], e2e["device_out"]])

    if rank == 0:
        total = world * B * args.steps
        value = total / (ms / 1e3)
        line = {
            "metric": METRIC, "value": value, "unit": "images/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms / args.steps, "per_rank_ms": per_rank, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": {"workload": workload_string(args.workload), "out_dtype": "fp16", "sampler": "fused Philox4x32-10 (device)",
                       "global_batch": world * B, "parallelism": "dp%d (independent shards, no collective)" % world,
                       "l2": "inputs/outputs rotate over %d buffer sets (%.0f MB) > 126 MB L2" % (
                           wl.NSETS, wl.NSETS * (wl.in_bytes + wl.out_bytes) / 1e6)},
            "clocks": clk,
            "e2e": {"value": total / (ms_rt / 1e3), "unit": "images/s", "h2d_bytes_per_step": wl.in_bytes,
                    "d2h_bytes_per_step": wl.out_bytes,
                    "what": "faa_augment_host: pinned host uint8 in -> pinned host fp16 out (chunked H2D/kernel/D2H pipeline)"},
            "e2e_device_out": {"value": total / (ms_dev / 1e3), "unit": "images/s", "h2d_bytes_per_step": wl.in_bytes,
                               "d2h_bytes_per_step": 2,
                               "what": "same call, result left on the device for the model (train.py:49 becomes a no-op); one scalar read back"},
            "gpu_launches": launches,
            "roofline": wl.roofline(ms / args.steps),
        }
        if also:
            line["also"] = also
        if mix:
            line["mixup_b2048"] = mix
        if train:
            line["train_step"] = train
        if world == 1 and not args.no_cpu:
            cores = host_cores()
            workers = min(8, cores)
            nb = 24 if H >= 224 else 80
            v, dt, kind = cpu_throughput(args.workload, nb, 2, workers)
            v1, dt1, _ = cpu_throughput(args.workload, 1 if H >= 224 else 4, 1, 0)
            line["cpu_baseline"] = {"value": v, "unit": "images/s", "cores": workers, "kind": kind,
                                    "host_cores": cores, "one_core": {"value": v1, "unit": "images/s", "seconds": dt1},
                                    "sample": "%d batches of %d through the reference's Augmentation + torchvision chain in a torch "
                                              "DataLoader with %d workers (reference data.py:215), first batches excluded; %.1f s; "
                                              "one_core = the same chain in the main process (num_workers=0)" % (nb, B, workers, dt),
                                    "note": "the reference's DataLoader architecture is main-process-bound beyond ~8 workers "
                                            "(per-worker rate drops from ~700 to ~60 img/s at 128 workers): see --impl reference"}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def dump_outputs(out_dir, images, rows):
    """What the timed path returned to its caller in its last step: ``out.npy`` (float32 [n, 3, out_h, out_w], the
    fp16 NCHW output widened exactly) and ``out_rows.npy`` (float64 [n], the batch rows those images are).  Inputs,
    seed and step indices depend only on the arguments, so two builds run with the same arguments can be compared
    array for array."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "out.npy"), images.astype(np.float32))
    np.save(os.path.join(out_dir, "out_rows.npy"), rows.astype(np.float64))


def run_reference(args):
    """Reference arm: the reference's own CPU implementation of the path - its Augmentation /
    CutoutDefault classes from ``oracle/_ref`` (verbatim reference package; falls back to the oracle port
    when absent) inside a torch DataLoader with every host core as a worker.  Rank 0 only.  This process
    never imports fast_autoaugment_b200 (no CUDA library is loaded)."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    H, W, B, *_ = WORKLOADS[args.workload]
    cores = host_cores()
    workers = max(1, cores)
    steps = args.steps
    warm = max(1, args.warmup)
    v, dt, kind = cpu_throughput(args.workload, steps, warm, workers)
    line = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": "images/s",
        "n_gpus": int(os.environ.get("WORLD_SIZE", str(args.gpus))), "steps": steps, "warmup": warm,
        "ms_per_step": dt / steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u8", "data": "synthetic",
        "config": {"workload": workload_string(args.workload), "out_dtype": "fp32", "sampler": "Python random / numpy / torch CPU generators",
                   "global_batch": B, "parallelism": "torch DataLoader, %d worker processes" % workers},
        "cpu_baseline": {"value": v, "unit": "images/s", "cores": workers, "kind": kind,
                         "sample": "%d steps of one %d-image batch each, %d DataLoader workers, %d warm-up batches excluded" % (steps, B, workers, warm),
                         "note": "main-process-bound: the DataLoader's collate/IPC in the parent limits the rate beyond ~8 workers"},
        "e2e": {"value": v, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2000)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="imagenet224_b512", choices=sorted(WORKLOADS))
    ap.add_argument("--seed", type=int, default=2024)
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-also", action="store_true", help="skip the extra single-GPU configurations (CIFAR b512, 380x380 b256)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed to DIR/*.npy (float32, at most 64 MB; rank 0)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs saves the outputs of --impl ours")
    args.warmup = max(3, args.warmup) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        return run_reference(args)
    if args.gpus > 1 and "WORLD_SIZE" not in os.environ:      # convenience: self-launch under torchrun
        import socket
        s = socket.socket()
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
        s.close()
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(args.gpus),
               "--master-addr", "127.0.0.1", "--master-port", str(port), os.path.abspath(__file__)] + sys.argv[1:]
        sys.exit(subprocess.call(cmd))
    run_ours(args)


if __name__ == "__main__":
    main()
