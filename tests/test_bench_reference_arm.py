"""bench.py's reference arm runs on a CPU-only box and prints the contract's JSON line."""
import json
import os
import subprocess
import sys

from helpers import ROOT


def test_reference_arm_json_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload",
                          "cifar32_b512", "--steps", "2", "--warmup", "1"], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better",
              "scaling", "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in line, k
    assert line["impl"] == "reference" and line["value"] > 0 and line["unit"] == "images/s"
    ref_there = os.path.isdir(os.path.join(ROOT, "oracle", "_ref", "FastAutoAugment"))
    assert line["cpu_baseline"]["kind"] == ("reference" if ref_there else "port") and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["d2h_bytes_per_step"] == 0
    # other ranks of a torchrun launch stay silent
    env = dict(os.environ, RANK="1", WORLD_SIZE="2")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2"],
                         capture_output=True, text=True, timeout=120, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_reference_arm_never_loads_the_cuda_library():
    """VERDICT r01 weak #2a: the reference arm's process must not map libfaa_b200.so (nor import the package)."""
    code = ("import sys, bench\n"
            "chain, kind = bench._cpu_chain('imagenet224_b512')\n"
            "import PIL.Image, numpy as np\n"
            "chain(PIL.Image.fromarray(np.zeros((224, 224, 3), np.uint8)))\n"
            "assert not any(m.startswith('fast_autoaugment_b200') for m in sys.modules), 'package imported'\n"
            "assert 'libfaa_b200' not in open('/proc/self/maps').read(), 'library mapped'\n"
            "print(kind)\n")
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    assert out.stdout.strip().splitlines()[-1] in ("reference", "port")


def test_workload_string_is_shared_by_both_arms():
    sys.path.insert(0, ROOT)
    import bench
    s = bench.workload_string("imagenet224_b512")
    assert "fp16" not in s and "fp32" not in s and "Philox" not in s      # arm-specific facts live in other keys
