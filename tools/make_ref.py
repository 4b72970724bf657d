"""Recipe for ``oracle/_ref/``: an UNMODIFIED copy of the reference files the CPU baseline runs.

    python tools/make_ref.py            (called by __graft_entry__.build() whenever /root/reference is present)

Why a copy: the reference is pure Python (nothing to compile) and has no setup.py / pyproject.toml (``pip install
--target baseline/_ref /root/reference`` fails: "neither 'setup.py' nor 'pyproject.toml' found"), yet
``/root/reference`` does not exist on the GPU box.  ``oracle/_ref/`` is git-ignored (it never enters the history)
but not gpurun-ignored, so it travels with the snapshot exactly like the built ``.so``.  Files are copied byte for
byte; ``MANIFEST.json`` records their SHA-256.

TEST / BENCH INFRASTRUCTURE ONLY: the product never imports anything from here.  Consumers:
``bench.py --impl reference`` and ``cpu_baseline`` (the reference's own FAISSRetriever / UnifiedIndex / filter.py
code timed on the host cores).
"""
from __future__ import annotations

import hashlib
import json
import os
import shutil
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.environ.get("IVR_REFERENCE_SRC", "/root/reference")
DST = os.path.join(ROOT, "oracle", "_ref")
# the modules on the hot path (SURVEY.md section 8a) and what they import from the reference itself
FILES = ("core.py", "utils.py", "unified_index.py", "unified_builder.py", "filter.py", "filter_research_update.py",
         "video_frame_filter.py")


def sha256(path: str) -> str:
    h = hashlib.sha256()
    with open(path, "rb") as f:
        for blk in iter(lambda: f.read(1 << 20), b""):
            h.update(blk)
    return h.hexdigest()


def main() -> int:
    if not os.path.isdir(SRC):
        print(f"make_ref: {SRC} not present (GPU box?) -- keeping whatever oracle/_ref already holds")
        return 0
    os.makedirs(DST, exist_ok=True)
    manifest = {}
    for name in FILES:
        src, dst = os.path.join(SRC, name), os.path.join(DST, name)
        if not os.path.isfile(src):
            print(f"make_ref: {src} missing", file=sys.stderr)
            return 1
        if not (os.path.isfile(dst) and sha256(dst) == sha256(src)):
            shutil.copyfile(src, dst)
            os.chmod(dst, 0o644)
        manifest[name] = sha256(dst)
    with open(os.path.join(DST, "MANIFEST.json"), "w") as f:
        json.dump({"source": SRC, "sha256": manifest}, f, indent=1, sort_keys=True)
    print(f"make_ref: {len(FILES)} reference files in {DST}")
    return 0


if __name__ == "__main__":
    sys.exit(main())
