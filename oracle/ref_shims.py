"""Import shims that run the REFERENCE'S OWN files in the authoring container.

TEST / BENCH INFRASTRUCTURE ONLY.  Used by tests/golden/make_golden*.py to produce golden
vectors from the unmodified reference at /root/reference, and -- through the byte-for-byte,
git-ignored copy ``oracle/_ref`` that tools/make_ref.py makes at build time and that travels
to the GPU box with the snapshot -- by ``bench.py``'s CPU arm (the reference's own wrappers
and filter.py timed on the host cores).  No reference source enters the git history.

What is shimmed and why (SURVEY.md section 0, fact 4):
  * ``transformers``  -- filter.py:46-48 calls ``from_pretrained`` at import
                         (network); a stub class is injected instead.
  * ``faiss``         -- unified_index.py:31 / core.py:32 import it
                         unconditionally; not installed.  A caller-supplied
                         faiss-shaped module (the oracle's, or the product's
                         ``faiss_compat``) is injected.
  * ``h5py``, ``lz4``, ``lz4.frame`` -- unified_index.py:29-30; empty stubs
                         (only the .rvdb I/O uses them, which is out of scope).
  * ``imagehash``, ``colorama`` -- filter_research_update.py:15,17; absent; stubs
                         (perceptual hashing of image files and coloured logging only).
  * CWD               -- ``utils.Config()`` creates exports/ index/ logs/
                         metadata/ relative to the CWD (utils.py:267-268), so the
                         import happens inside a temp dir.
"""
from __future__ import annotations

import contextlib
import importlib
import os
import sys
import tempfile
import types

_HERE = os.path.dirname(os.path.abspath(__file__))


def _find_reference() -> str:
    """IVR_REFERENCE_DIR, else /root/reference (authoring container), else oracle/_ref -- the byte-for-byte copy
    tools/make_ref.py makes at build time, which is what exists on the GPU box."""
    for cand in (os.environ.get("IVR_REFERENCE_DIR"), "/root/reference", os.path.join(_HERE, "_ref")):
        if cand and os.path.isfile(os.path.join(cand, "filter.py")) and os.path.isfile(os.path.join(cand, "core.py")):
            return cand
    return os.path.join(_HERE, "_ref")


REFERENCE_DIR = _find_reference()


def reference_available() -> bool:
    return os.path.isfile(os.path.join(REFERENCE_DIR, "filter.py"))


def _stub_transformers():
    tr = types.ModuleType("transformers")

    class _Stub:
        @classmethod
        def from_pretrained(cls, *a, **k):
            return cls()

        def to(self, *a, **k):
            return self

        def eval(self):
            return self

    for name in ("AutoImageProcessor", "AutoModel", "CLIPModel", "CLIPProcessor",
                 "CLIPTokenizer", "AutoTokenizer", "AutoProcessor"):
        setattr(tr, name, _Stub)
    return tr


def _stub_colorama():
    """colorama is only used for coloured log lines (filter_research_update.py:17-35)."""
    co = types.ModuleType("colorama")

    class _Codes:
        def __getattr__(self, _):
            return ""

    co.Fore, co.Back, co.Style = _Codes(), _Codes(), _Codes()
    co.init = lambda *a, **k: None
    return co


def oracle_faiss_module():
    """A ``faiss``-shaped module backed by oracle.flat_ip (for pinning the wrappers)."""
    from . import flat_ip
    m = types.ModuleType("faiss")
    m.IndexFlatIP = flat_ip.IndexFlatIP
    m.Index = flat_ip.IndexFlatIP
    m.normalize_L2 = flat_ip.normalize_L2
    return m


@contextlib.contextmanager
def reference_modules(faiss_module=None, names=("filter",), stub_transformers=False):
    """Yield a dict {name: module} of reference modules imported under shims.

    Modules are removed from ``sys.modules`` again on exit so the product's own
    same-named modules are never shadowed.  ``stub_transformers`` also stubs HuggingFace
    for ``core`` (only its CLIP extractor uses it): saves ~20 s of import when just the
    retriever classes are wanted.
    """
    if not reference_available():
        raise RuntimeError(f"reference not present at {REFERENCE_DIR}")
    saved = {k: sys.modules.get(k) for k in
             ("transformers", "faiss", "h5py", "lz4", "lz4.frame", "imagehash", "colorama",
              "filter", "filter_research_update", "core", "utils", "unified_index", "unified_builder")}
    old_path = list(sys.path)
    old_cwd = os.getcwd()
    tmp = tempfile.mkdtemp(prefix="ivr_ref_")
    try:
        if "filter" in names or "filter_research_update" in names or stub_transformers:
            sys.modules["transformers"] = _stub_transformers()
        if "filter_research_update" in names:       # filter_research_update.py:15,17 -- absent, presentation only
            sys.modules["imagehash"] = types.ModuleType("imagehash")
            sys.modules["colorama"] = _stub_colorama()
        sys.modules["faiss"] = faiss_module or oracle_faiss_module()
        for stub in ("h5py", "lz4", "lz4.frame"):
            mod = types.ModuleType(stub)
            if stub == "h5py":
                mod.File = object
            sys.modules[stub] = mod
        sys.modules["lz4"].frame = sys.modules["lz4.frame"]
        for k in ("filter", "filter_research_update", "core", "utils", "unified_index", "unified_builder"):
            sys.modules.pop(k, None)
        sys.path.insert(0, REFERENCE_DIR)
        os.chdir(tmp)
        out = {n: importlib.import_module(n) for n in names}
        yield out
    finally:
        os.chdir(old_cwd)
        sys.path[:] = old_path
        for k, v in saved.items():
            if v is None:
                sys.modules.pop(k, None)
            else:
                sys.modules[k] = v
