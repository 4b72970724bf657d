"""Builds and times the REFERENCE'S OWN retrieval / dedup classes (TEST / BENCH INFRASTRUCTURE ONLY).

The classes come from the unmodified reference files (``/root/reference`` here, the byte-for-byte copy
``oracle/_ref`` on the GPU box -- tools/make_ref.py) imported under ``oracle/ref_shims``; the ``faiss`` module
under them is whatever the caller injects:

* ``oracle.flat_ip_mt.faiss_module()``  -> the reference's CPU path (bench.py ``--impl reference`` / ``cpu_baseline``):
  FAISS itself is an un-vendored, absent dependency, so the flat search UNDER the reference's wrappers is the
  oracle's multi-threaded restatement of its contract; everything above it is reference code.

Reference constructors read ``utils.Config`` / create log directories; the objects are therefore assembled the
way tests/golden/make_golden.py does it (``__new__`` + the attributes ``__init__`` would set: core.py:700-734).
"""
from __future__ import annotations

import contextlib
import io
import threading
import time

import numpy as np

from . import ref_shims


class _Log:
    def __getattr__(self, _):
        return lambda *a, **k: None


class _Cfg:
    def get(self, key, default=None):
        return {"retrieval.faiss_index_type": "IndexFlatIP", "retrieval.enable_gpu": False}.get(key, default)


class _Timer:
    def __enter__(self):
        return self

    def __exit__(self, *a):
        return False


class _Perf:
    def timer(self, *a, **k):
        return _Timer()


def make_faiss_retriever(core):
    """core.FAISSRetriever with the state its __init__ sets (core.py:700-734), minus utils.Config side effects."""
    fr = core.FAISSRetriever.__new__(core.FAISSRetriever)
    fr.config, fr.logger, fr.cache = _Cfg(), _Log(), None
    fr.perf_monitor = _Perf()
    fr.index, fr.index_type, fr.use_gpu = None, "IndexFlatIP", False
    fr.dimension, fr.is_trained = None, False
    fr.id_to_metadata, fr.metadata_to_id, fr.next_id = {}, {}, 0
    fr.validator = core.DataConsistencyValidator(_Log())
    fr._lock = threading.RLock()
    return fr


def keyframe_metadata(core, feats: np.ndarray, frames_per_folder: int = 1000):
    """One core.KeyframeMetadata per row; ``clip_features`` are views of ``feats`` (the reference re-scores against
    them: core.py:913-916)."""
    return [core.KeyframeMetadata(folder_name=f"L{i // frames_per_folder:05d}_V001",
                                  image_name=f"{i % frames_per_folder:06d}", frame_id=i % frames_per_folder,
                                  file_path=f"keyframes/L{i // frames_per_folder:05d}_V001/{i % frames_per_folder:06d}.jpg",
                                  clip_features=feats[i]) for i in range(len(feats))]


def metadata_dicts(n: int, frames_per_folder: int = 1000):
    """The metadata dicts of a unified index (unified_index.py:870-877)."""
    return [{"file_path": f"keyframes/L{i // frames_per_folder:05d}_V001/{i % frames_per_folder:06d}.jpg",
             "folder_name": f"L{i // frames_per_folder:05d}_V001", "image_name": f"{i % frames_per_folder:06d}.jpg",
             "frame_id": i % frames_per_folder, "file_hash": f"{i:016x}", "file_size": 1000 + i} for i in range(n)]


def make_unified_index(unified_index_mod, faiss_mod, xb: np.ndarray, meta):
    """unified_index.UnifiedIndex in the state ``_setup_memory_maps`` leaves it (unified_index.py:1175-1234), the
    index built like ``_build_faiss_index_from_file`` (1755-1793): IndexFlatIP(dim); 10 000-row chunks,
    normalize_L2 each, add."""
    index = faiss_mod.IndexFlatIP(xb.shape[1])
    for s in range(0, len(xb), 10000):
        chunk = xb[s:s + 10000].astype("float32").copy()
        faiss_mod.normalize_L2(chunk)
        index.add(chunk)
    u = unified_index_mod.UnifiedIndex()
    u.faiss_index, u.metadata_list, u.is_loaded, u.vectors = index, meta, True, xb
    u.memory_maps = {"thumbnails": {}, "temporal": {}}
    return u


def time_faiss_retriever(xb: np.ndarray, xq: np.ndarray, k: int, steps: int = 1, warmup: int = 0, faiss_module=None):
    """The reference's batched entry point, ``FAISSRetriever.build_index`` + ``.search(xq, k)`` (core.py:758-930), on
    the host.  Returns {"step_s": median seconds per search call, "search_s": of which inside index.search,
    "build_s", "hits"}."""
    from . import flat_ip_mt
    fm = faiss_module or flat_ip_mt.faiss_module()
    with ref_shims.reference_modules(faiss_module=fm, names=("core",), stub_transformers=True) as mods:
        core = mods["core"]
        t0 = time.perf_counter()
        kms = keyframe_metadata(core, xb)
        fr = make_faiss_retriever(core)
        fr.build_index(xb, kms, validate_consistency=False)     # the validator stats real files (core.py:300-330)
        build_s = time.perf_counter() - t0
        for _ in range(warmup):
            fr.search(xq[:8], k)
        ts, inner, hits = [], [], 0
        for _ in range(max(steps, 1)):
            s0 = getattr(fr.index, "search_seconds", 0.0)
            t0 = time.perf_counter()
            out = fr.search(xq, k)
            ts.append(time.perf_counter() - t0)
            inner.append(getattr(fr.index, "search_seconds", 0.0) - s0)
            hits = len(out)
    i = int(np.argsort(ts)[len(ts) // 2])
    return {"step_s": ts[i], "search_s": inner[i], "build_s": build_s, "hits": hits}


def time_search_vectors(xb: np.ndarray, xq: np.ndarray, k: int, faiss_module=None):
    """The reference's production path: ``UnifiedIndex.search_vectors`` called once per query
    (unified_index.py:480-538; system.py:733-826 loops over queries).  Returns seconds for the whole loop."""
    from . import flat_ip_mt
    fm = faiss_module or flat_ip_mt.faiss_module()
    with ref_shims.reference_modules(faiss_module=fm, names=("unified_index",), stub_transformers=True) as mods:
        u = make_unified_index(mods["unified_index"], fm, xb, metadata_dicts(len(xb)))
        u.search_vectors(xq[0], k)
        t0 = time.perf_counter()
        n_hits = sum(len(u.search_vectors(q, k)) for q in xq)
        return {"loop_s": time.perf_counter() - t0, "hits": n_hits}


def time_filter_pipeline(x: np.ndarray, window: int = 8, threshold: float = 0.95, transition: float = 0.75,
                         min_scene: int = 2):
    """The reference's own similarity stage (filter.py:142-315) on float32 frames: calculate_similarities ->
    detect_scene_transitions -> group_into_scenes -> apply_similarity_filtering_to_scenes (advanced window rule).
    One Python thread by construction.  Returns {"seconds", "kept": global indices}."""
    cfg = {"enable_similarity_filtering": True, "similarity_threshold": threshold, "similarity_window_size": window,
           "use_advanced_similarity_filtering": True, "min_frame_distance": 1}
    with ref_shims.reference_modules(names=("filter",)) as mods:
        rf = mods["filter"]
        emb = list(x)
        t0 = time.perf_counter()
        with contextlib.redirect_stdout(io.StringIO()):
            sims = rf.calculate_similarities(emb)
            scenes = rf.group_into_scenes(rf.detect_scene_transitions(sims, transition), len(emb), min_scene)
            kept = rf.apply_similarity_filtering_to_scenes(emb, list(range(len(emb))), scenes, cfg)[1]
        return {"seconds": time.perf_counter() - t0, "kept": kept, "scenes": len(scenes)}
