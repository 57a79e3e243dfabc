#!/usr/bin/env python
"""Stage the UNMODIFIED reference (LikeLy-Journey/SegmenTron) under ``baseline/_ref/`` so that it travels to the GPU box.

``/root/reference`` exists only in the build container; ``baseline/_ref/`` is git-ignored (no reference source ever enters the
history) but not gpurun-ignored, so the snapshot that goes to the B200 box carries it exactly like the built ``.so``.  What is
staged: the ``segmentron`` package, ``tools/`` and ``configs/`` byte for byte, plus -- OUTSIDE that tree, under
``baseline/_ref/_stubs`` -- the one stub the reference needs on a current stack (``thop``, SURVEY.md App. B3).  The other
compatibility shims (``np.int``, ``--local-rank``) are applied by the process that imports it (``tools/ref_harness.py``,
``segmentron_b200/launch.py``), never by editing the copy.

    python tools/make_baseline_ref.py [--src /root/reference] [--force]

Run by hand: ``__graft_entry__.build()`` does not stage the reference, and without a staged copy ``bench.py`` times the oracle port
for ``cpu_baseline`` / ``cudnn_ref``.  A ``MANIFEST.json`` with the sha256 of every staged file lets ``verify()`` check that the copy
is unmodified.
"""
import argparse
import hashlib
import json
import os
import shutil
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DST = os.path.join(ROOT, "baseline", "_ref")
KEEP = ("segmentron", "tools", "configs")
SKIP_EXT = (".png", ".jpg", ".pyc", ".so", ".o")


def sha(path):
    h = hashlib.sha256()
    with open(path, "rb") as f:
        h.update(f.read())
    return h.hexdigest()


def stage(src="/root/reference", force=False):
    """Copy the reference tree; returns the number of files staged (0 when the copy is already current)."""
    if not os.path.isdir(os.path.join(src, "segmentron")):
        raise FileNotFoundError(f"no reference at {src}")
    man_path = os.path.join(DST, "MANIFEST.json")
    files = []
    for top in KEEP:
        for d, _, fs in os.walk(os.path.join(src, top)):
            if "__pycache__" in d:
                continue
            for f in sorted(fs):
                if f.endswith(SKIP_EXT):
                    continue
                files.append(os.path.relpath(os.path.join(d, f), src))
    files.sort()
    want = {f: sha(os.path.join(src, f)) for f in files}
    if not force and os.path.exists(man_path):
        try:
            have = json.load(open(man_path))["files"]
            if have == want and all(os.path.exists(os.path.join(DST, f)) for f in want):
                return 0
        except Exception:
            pass
    for top in KEEP:
        shutil.rmtree(os.path.join(DST, top), ignore_errors=True)
    for f in files:
        out = os.path.join(DST, f)
        os.makedirs(os.path.dirname(out), exist_ok=True)
        shutil.copyfile(os.path.join(src, f), out)
    stub = os.path.join(DST, "_stubs", "thop")
    os.makedirs(stub, exist_ok=True)
    with open(os.path.join(stub, "__init__.py"), "w") as f:
        f.write('"""Stub for the optional `thop` profiler the reference imports unconditionally (utils/visualize.py:8).\n'
                'Not reference code: it only lets `tools/train.py` import; the call site is wrapped in try/except."""\n\n\n'
                'def profile(*a, **k):\n    raise RuntimeError("thop is not installed (stub)")\n')
    with open(man_path, "w") as f:
        json.dump({"source": "LikeLy-Journey/SegmenTron (read-only mount /root/reference)", "files": want}, f, indent=0, sort_keys=True)
    return len(files)


def verify():
    """True when every staged file still matches the manifest (the copy is unmodified)."""
    man = json.load(open(os.path.join(DST, "MANIFEST.json")))["files"]
    return all(os.path.exists(os.path.join(DST, f)) and sha(os.path.join(DST, f)) == h for f, h in man.items())


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--src", default="/root/reference")
    ap.add_argument("--force", action="store_true")
    a = ap.parse_args()
    n = stage(a.src, a.force)
    print(f"[baseline/_ref] staged {n} files" if n else "[baseline/_ref] up to date", file=sys.stderr)
