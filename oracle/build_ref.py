#!/usr/bin/env python
"""Recipe for ``oracle/_ref``: the UNMODIFIED reference package, importable on the GPU box.

TEST / BASELINE INFRASTRUCTURE ONLY (see ``oracle/__init__.py``).

The reference (kakaobrain/fast-autoaugment @ 2424224) is pure Python - there is nothing to
compile - so "building" it means placing its package where ``bench.py --impl reference`` and
the tests can import it when ``/root/reference`` does not exist (the GPU box):

    oracle/_ref/FastAutoAugment/   verbatim copy of /root/reference/FastAutoAugment (git-ignored:
                                   the reference's sources never enter this repository's history)
    oracle/_ref/theconf.py         import shim: ``theconf`` is not installed (reference data.py:16)
    oracle/_ref/torch_six_shim.py  import shim: ``torch._six`` no longer exists
                                   (reference networks/efficientnet_pytorch/condconv.py:4)
    oracle/_ref/MANIFEST.json      sha256 of every copied file + the commit they came from

Run here (build container): ``python oracle/build_ref.py``; ``__graft_entry__.build()`` calls it
whenever ``/root/reference`` is present.  ``oracle/_ref/`` is listed in ``.gitignore`` but not in
``.gpurunignore``, so it travels to the GPU box with the snapshot.
"""
from __future__ import annotations

import hashlib
import json
import os
import shutil
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
REF_ROOT = os.environ.get("FAA_REFERENCE_ROOT", "/root/reference")
DST = os.path.join(HERE, "_ref")

THECONF = '''"""Import shim for the `theconf` package (not installed): the two names reference data.py /
train.py import.  `Config.get()` returns one process-wide dict, like theconf's singleton."""


class Config:
    _d = {}

    @classmethod
    def get(cls):
        return cls._d


class ConfigArgumentParser:  # only imported by train.py / search.py, never constructed here
    def __init__(self, *a, **k):
        raise RuntimeError("theconf shim: ConfigArgumentParser is not available")
'''

SIX = '''"""Import shim: `torch._six` was removed from torch; the reference only needs `container_abcs`."""
import collections.abc
import sys
import types


def install():
    if "torch._six" not in sys.modules:
        m = types.ModuleType("torch._six")
        m.container_abcs = collections.abc
        sys.modules["torch._six"] = m
'''


def build(force: bool = False) -> str | None:
    src = os.path.join(REF_ROOT, "FastAutoAugment")
    if not os.path.isdir(src):
        return DST if os.path.isdir(os.path.join(DST, "FastAutoAugment")) else None
    man_path = os.path.join(DST, "MANIFEST.json")
    files = {}
    for root, _, names in os.walk(src):
        for n in sorted(names):
            if n.endswith(".py"):
                p = os.path.join(root, n)
                with open(p, "rb") as f:
                    files[os.path.relpath(p, REF_ROOT)] = hashlib.sha256(f.read()).hexdigest()
    if not force and os.path.exists(man_path):
        try:
            with open(man_path) as f:
                if json.load(f).get("files") == files:
                    return DST
        except Exception:
            pass
    shutil.rmtree(DST, ignore_errors=True)
    os.makedirs(DST)
    shutil.copytree(src, os.path.join(DST, "FastAutoAugment"),
                    ignore=shutil.ignore_patterns("__pycache__", "*.pyc"))
    with open(os.path.join(DST, "theconf.py"), "w") as f:
        f.write(THECONF)
    with open(os.path.join(DST, "torch_six_shim.py"), "w") as f:
        f.write(SIX)
    commit = None
    try:
        with open(os.path.join(REF_ROOT, ".SUBMODULES.json")) as f:
            commit = json.load(f).get("commit")
    except Exception:
        pass
    with open(man_path, "w") as f:
        json.dump({"source": "kakaobrain/fast-autoaugment", "commit": commit, "files": files}, f, indent=1)
    return DST


def import_ref():
    """Import the vendored reference (``oracle/_ref``, placed by ``build()``).  Never reads or copies
    the reference checkout itself, so callers (bench.py, tests) write nothing into the tree.
    Returns (augmentations, archive, aug_mixup, data) modules of the reference, or None."""
    if not os.path.isdir(os.path.join(DST, "FastAutoAugment")):
        return None
    if DST not in sys.path:
        sys.path.insert(0, DST)
    import torch_six_shim
    torch_six_shim.install()
    from FastAutoAugment import augmentations, archive, aug_mixup, data
    return augmentations, archive, aug_mixup, data


if __name__ == "__main__":
    out = build(force="--force" in sys.argv)
    print("oracle/_ref:", out)
